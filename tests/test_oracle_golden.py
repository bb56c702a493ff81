"""The CPU oracle restatements against the committed golden vectors (produced by the reference's own code through
oracle/make_golden.py).  Runs anywhere (no GPU, no /root/reference)."""
import os

import numpy as np
import pytest
import torch

from oracle import bicubic_oracle as BO
from oracle import eval_oracle as EO
from oracle import fsrnet_oracle as FO


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name), allow_pickle=False)


def test_fsrnet_param_inventory():
    shapes = FO.fsrnet_param_shapes()
    assert len(shapes) == 202
    total = sum(int(np.prod(s)) for _, s in shapes)
    dead = sum(int(np.prod(s)) for k, s in shapes if FO.fsrnet_dead_param(k))
    assert total == 6970311 and dead == 888789          # SURVEY.md Appendix A / E


def test_seeded_init_matches_reference_checksums(golden_dir):
    g = _load(golden_dir, "fsrnet_init_checksums.npz")
    sd = FO.build_fsrnet_state_dict(1234)
    assert list(sd.keys()) == [str(n) for n in g["names"]]
    sums = np.array([v.double().sum().item() for v in sd.values()])
    abss = np.array([v.double().abs().sum().item() for v in sd.values()])
    np.testing.assert_allclose(sums, g["sums"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(abss, g["abssums"], rtol=1e-12)


def test_fsrnet_forward_backward_small(golden_dir):
    g = _load(golden_dir, "fsrnet_small.npz")
    sd = FO.build_fsrnet_state_dict(1234)
    x, hr, lbl, hm = FO.synthetic_batch(2, 64)
    outs, total, parts, gd = FO.fsrnet_loss_and_grads(sd, x, hr, hm, lbl)
    for name, o in zip(("coarse", "out", "landmark", "parsing"), outs):
        np.testing.assert_allclose(o.numpy(), g[name], rtol=1e-3, atol=2e-4)
    np.testing.assert_allclose(total.item(), g["total"], rtol=1e-5)
    np.testing.assert_allclose([p.item() for p in parts], g["parts"], rtol=1e-5)
    norms = dict(zip([str(n) for n in g["grad_names"]], g["grad_norms"]))
    for k, v in gd.items():
        if v is None:
            assert FO.fsrnet_dead_param(k)
            continue
        if k in FO.FSRNET_NULL_GRAD:
            assert v.norm().item() < 1e-3 * g["global_grad_norm"]
            continue
        assert abs(v.norm().item() - norms[k]) <= 2e-2 * norms[k] + 1e-6, k
    for k in g.files:
        if k.startswith("grad:") and k[5:] not in FO.FSRNET_NULL_GRAD:
            ref = torch.from_numpy(g[k])
            got = gd[k[5:]]
            if "gidx:" + k[5:] in g.files:          # large gradients are stored as a fixed sample of their elements
                got = got.reshape(-1)[torch.from_numpy(g["gidx:" + k[5:]]).long()]
            assert ((got - ref).norm() / (ref.norm() + 1e-30)).item() < 2e-2, k


@pytest.mark.timeout(300)
def test_fsrnet_known_answer_128(golden_dir):
    """SURVEY.md Appendix E: config 1 (B=4, 128x128, fp32 CPU)."""
    g = _load(golden_dir, "fsrnet_kat128.npz")
    sd = FO.build_fsrnet_state_dict(1234)
    x, hr, lbl, hm = FO.synthetic_batch(4, 128)
    with torch.no_grad():
        outs = FO.fsrnet_forward(sd, x)
        total, parts = FO.fsrnet_loss(outs, hr, hm, lbl)
    np.testing.assert_allclose([p.item() for p in parts], g["parts"], rtol=2e-5)
    np.testing.assert_allclose(total.item(), 52551.878906, rtol=2e-5)
    np.testing.assert_allclose(total.item(), g["total"], rtol=2e-5)
    assert abs(outs[1].mean().item() - g["out_mean"]) < 1e-4 and abs(outs[1].std().item() - g["out_std"]) < 1e-4


def test_losses_golden(golden_dir):
    g = _load(golden_dir, "losses.npz")
    t = {k: torch.from_numpy(g[k]) for k in ("a", "t", "lm", "hm", "lg", "lb")}
    got = [FO.mse97(t["a"], t["t"]).item(), FO.landmark_loss(t["lm"], t["hm"]).item(), FO.ce2d(t["lg"], t["lb"]).item()]
    np.testing.assert_allclose(got, g["values"], rtol=1e-6)


def test_bicubic_golden(golden_dir):
    g = _load(golden_dir, "bicubic.npz")
    for key in g.files:
        if not key.startswith("src_"):
            continue
        _, s, o = key.split("_")
        src, dst = g[key], g["dst_%s_%s" % (s, o)]
        got = BO.bicubic_u8(src, int(o), int(o))
        assert np.array_equal(got, dst), key


def test_bicubic_edge_cases():
    # identity size, 1-pixel images and non-square targets follow the same window arithmetic
    rng = np.random.default_rng(3)
    a = rng.integers(0, 256, (5, 7, 3), dtype=np.uint8)
    assert np.array_equal(BO.bicubic_u8(a, 5, 7), a)
    one = np.full((1, 1, 3), 77, np.uint8)
    assert np.array_equal(BO.bicubic_u8(one, 8, 8), np.full((8, 8, 3), 77, np.uint8))
    try:
        from PIL import Image
    except ImportError:
        return
    ref = np.asarray(Image.fromarray(a).resize((21, 40), Image.BICUBIC))
    assert np.array_equal(BO.bicubic_u8(a, 40, 21), ref)


def test_eval_golden(golden_dir):
    g = _load(golden_dir, "eval.npz")
    assert abs(EO.accuracy(g["scores"], g["target"], (1,))[0] - g["top1"]) < 1e-5
    np.testing.assert_allclose(EO.accuracy(g["scores"], g["target"], (1, 5)), g["top15"])
    assert np.array_equal(EO.topk_indices(g["scores"], 5), g["top5_idx"])
    dist = EO.pair_sqdist(g["e1"], g["e2"])
    got = np.array([EO.calculate_accuracy(t, dist, g["same"]) for t in g["thr"]])
    np.testing.assert_allclose(got, g["calc_acc"])


def test_eval_edge_cases():
    # ties resolve to the lowest index; all-same / all-different label sets do not divide by zero
    s = np.array([[1.0, 3.0, 3.0, 3.0, 0.0]], np.float32)
    assert EO.topk_indices(s, 3).tolist() == [[1, 2, 3]]
    d = np.array([0.1, 0.2, 5.0]);
    assert EO.calculate_accuracy(1.0, d, np.array([True, True, True])) == (2 / 3, 0, 2 / 3)
    assert EO.calculate_accuracy(1.0, d, np.array([False, False, False])) == (0, 2 / 3, 1 / 3)
    tpr, fpr, acc, best = EO.calculate_roc(np.arange(0, 4, 0.5), np.zeros((20, 4)), np.ones((20, 4)) * np.arange(20)[:, None] / 10,
                                           np.arange(20) < 10, nrof_folds=5, seed=1)
    assert 0.0 <= acc <= 1.0 and len(best) == 5


def test_matcher_oracle_planted_identities():
    g, p, ids = EO.synthetic_gallery(2000, 64, dim=128, seed=5)
    val, idx = EO.cosine_topk(p, g, 5)
    assert np.array_equal(idx[:, 0], ids)
    assert np.all(np.diff(val, axis=1) <= 0)


def test_resnet34_kd_oracle_against_reference_fixture(golden_dir):
    """oracle/resnet_oracle.py (ResNet_34 + KD losses) against tests/golden/resnet34.npz, which make_golden.py produced by
    running the reference's own model/resnet.py with torch.nn.MSELoss (distill_main.py:63,68-70)."""
    from oracle import resnet_oracle as RO
    g = _load(golden_dir, "resnet34.npz")
    sds = [RO.randomize_norm_params(RO.build_resnet34_state_dict(seed), 100 + i) for i, seed in enumerate((77, 78, 79))]
    names = RO.resnet34_param_names(sds[1])
    assert names == [str(n) for n in g["names"]] and len(names) == 114
    assert sum(1 for k in sds[1] if k.endswith("running_mean")) == 38
    x = RO.synthetic_faces(8)
    l_s, l_a, g_s, g_a, g_as, (t_outs, s_outs, a_outs) = RO.kd_step(sds[0], sds[1], sds[2], x)
    np.testing.assert_allclose(l_s.item(), float(g["l_s"]), rtol=1e-4)
    np.testing.assert_allclose(l_a.item(), float(g["l_a"]), rtol=1e-4)
    rel = lambda a, b: float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30))
    assert rel(t_outs[0].numpy(), g["emb_t"]) < 1e-3 and rel(s_outs[0].detach().numpy(), g["emb_s"]) < 1e-3
    assert rel(a_outs[0].detach().numpy(), g["emb_a"]) < 1e-3
    np.testing.assert_allclose([o.norm().item() for o in s_outs[1:]], g["feat_norms_s"], rtol=1e-4)
    for gs, key in ((g_s, "gnorm_s"), (g_a, "gnorm_a"), (g_as, "gnorm_as")):
        ours = np.array([gs[k].norm().item() for k in names])
        keep = np.array([k not in RO.RESNET_NULL_GRAD for k in names])
        np.testing.assert_allclose(ours[keep], g[key][keep], rtol=2e-2)
    for k in ("bn1.weight", "layer2.0.downsample.1.weight", "bn_o2.weight"):
        assert rel(g_s[k].numpy(), g["gs:" + k]) < 2e-2 and rel(g_a[k].numpy(), g["ga:" + k]) < 2e-2
        assert rel(g_as[k].numpy(), g["gas:" + k]) < 2e-2
    nb = {}
    RO.resnet34_forward(sds[1], x, training=True, new_buffers=nb)
    np.testing.assert_allclose(nb["bn1.running_mean"].numpy(), g["bn1_running_mean"], rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(nb["bn1.running_var"].numpy(), g["bn1_running_var"], rtol=1e-4)
    np.testing.assert_allclose(nb["bn_o2.running_var"].numpy(), g["bn_o2_running_var"], rtol=1e-3)


def test_ir50_oracle_against_reference_fixture(golden_dir):
    """oracle ir50_forward (eval mode) against the embedding the reference's own IR_50 produced (make_golden.py)."""
    from oracle import resnet_oracle as RO
    g = _load(golden_dir, "ir50.npz")
    sd0 = RO.build_ir50_state_dict(91)
    assert list(sd0) == [str(n) for n in g["names"]]
    np.testing.assert_allclose([v.double().sum().item() for v in sd0.values()], g["checksums"], rtol=0, atol=1e-9)
    assert len(RO.ir50_block_specs()) == 24
    sd = RO.randomize_bn_everywhere(sd0, 191)
    with torch.no_grad():
        emb = RO.ir50_forward(sd, RO.synthetic_faces(4, seed=4322))
    assert float(np.linalg.norm(emb.numpy() - g["emb"]) / np.linalg.norm(g["emb"])) < 1e-4


def test_landmark_heatmap_oracle_against_reference_fixture(golden_dir):
    g = _load(golden_dir, "heatmap.npz")
    for l, ref in zip(g["landmarks"], g["hm"]):
        assert np.array_equal(BO.landmark_heatmap(l, 32, 32, 1.3), ref)


def test_augment_oracle_against_pillow_fixture(golden_dir):
    """Image.rotate + ImageEnhance.Contrast (helen_loader.py:75-104): the restatement against vectors Pillow produced."""
    from oracle import augment_oracle as AO
    g = np.load(os.path.join(golden_dir, "augment.npz"))
    for i in range(int(g["count"])):
        src, ang, fac = g["src%d" % i], float(g["angle%d" % i]), g["fac%d" % i]
        h, w = src.shape[:2]
        assert np.array_equal(AO.rotate_coeffs(h, w, ang), g["coef%d" % i])
        assert np.array_equal(AO.rotate_u8(src, ang), g["rot%d" % i])
        assert np.array_equal(AO.augment_u8(src, ang, fac), g["out%d" % i])
    img = np.arange(5 * 7 * 3, dtype=np.uint8).reshape(5, 7, 3)
    assert np.array_equal(AO.rotate_u8(img, 0.0), img) and np.array_equal(AO.rotate_u8(img, 720.0), img)
    assert np.array_equal(AO.contrast_u8(img, 1.0), img)
    assert np.array_equal(AO.contrast_u8(img, 0.0), np.full_like(img, AO.luma_mean(img)))
    lm = np.array([[56.0, 56.0], [66.0, 56.0]])
    out = AO.rotate_landmarks(lm, 90.0, 56.0)         # rotate_matrix(-90): (x, y) - c -> (y', -x') ... about the centre
    assert np.allclose(out[0], [56.0, 56.0]) and np.allclose(out[1], [56.0, 46.0])
