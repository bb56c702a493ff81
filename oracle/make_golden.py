"""Pins the oracle restatements against the live reference and writes tests/golden/*.npz.

Run in the build container only (needs /root/reference and Pillow):  python -m oracle.make_golden
Every fixture is produced by the REFERENCE's own code (modules loaded by file path, SURVEY.md 8c); the oracle
restatement is asserted against it before anything is written.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import bicubic_oracle as BO      # noqa: E402
from oracle import eval_oracle as EO         # noqa: E402
from oracle import fsrnet_oracle as FO       # noqa: E402
from oracle import ref_loader as R           # noqa: E402
from oracle import resnet_oracle as RO       # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")
GRAD_SAMPLE = 8192          # elements stored of each large full-gradient tensor in fsrnet_small.npz


def ref_fsrnet(seed):
    F = R.load("model/FSRnet.py")
    torch.manual_seed(seed)
    net = F.OverallNetwork()
    net.apply(R.reference_weights_init)
    net.train()
    return net


def ref_loss(outs, hr, hm, lbl, batch):
    L = R.load("loss/loss.py")
    parts = (L.MSELossFunc()(outs[1], hr), L.MSELossFunc()(outs[0], hr), L.MSELoss_Landmark()(outs[2], hm),
             L.CrossEntropyLoss2d()(outs[3], lbl))
    return (5. * parts[0] + 5. * parts[1] + parts[2] + parts[3]) / (2.0 * batch), parts


def golden_fsrnet():
    net = ref_fsrnet(1234)
    ref_sd = net.state_dict()
    sd = FO.build_fsrnet_state_dict(1234)
    assert list(sd) == list(ref_sd) and all(torch.equal(sd[k], ref_sd[k]) for k in sd), "seeded init differs"
    np.savez_compressed(os.path.join(OUT, "fsrnet_init_checksums.npz"),
                        names=np.array(list(sd)), sums=np.array([v.double().sum().item() for v in sd.values()]),
                        abssums=np.array([v.double().abs().sum().item() for v in sd.values()]))
    for tag, b, size in (("small", 2, 64), ("kat128", 4, 128)):
        x, hr, lbl, hm = FO.synthetic_batch(b, size)
        net.zero_grad()
        outs = R.reference_fsrnet_forward(net, x)
        total, parts = ref_loss(outs, hr, hm, lbl, b)
        total.backward()
        o_outs, o_total, o_parts, gd = FO.fsrnet_loss_and_grads(ref_sd, x, hr, hm, lbl)
        for a, c in zip(outs, o_outs):
            assert torch.allclose(a, c, rtol=1e-4, atol=1e-4), (a - c).abs().max()
        assert abs(total.item() - o_total.item()) <= 1e-5 * abs(total.item())
        names, gnorm, small = [], [], {}
        for k, p in net.named_parameters():
            if p.grad is None:
                assert FO.fsrnet_dead_param(k), k
                continue
            g = p.grad
            if k not in FO.FSRNET_NULL_GRAD:
                rel = ((g - gd[k]).norm() / (g.norm() + 1e-30)).item()
                assert rel < 2e-2, (k, rel)
            names.append(k); gnorm.append(g.norm().item())
            if g.numel() <= 192:
                small["grad:" + k] = g.numpy()
        d = dict(total=total.item(), parts=np.array([p.item() for p in parts]),
                 grad_names=np.array(names), grad_norms=np.array(gnorm),
                 global_grad_norm=float(np.sqrt(np.sum(np.square(gnorm)))))
        if tag == "small":
            d.update(coarse=outs[0].detach().numpy(), out=outs[1].detach().numpy(),
                     landmark=outs[2].detach().numpy(), parsing=outs[3].detach().numpy())
            d.update(small)
            for k in ("_coarse_sr_network.residual.0.conv1.weight", "_fine_sr_decoder.deconv.weight",
                      "_prior_estimation_network.hg.hg.0.0.0.conv1.weight", "_fine_sr_encoder.conv_input.weight",
                      "_fine_sr_decoder.conv_out.weight", "_prior_estimation_network.fc_landmark.weight"):
                a = dict(net.named_parameters())[k].grad.numpy()
                if a.size > 2 * GRAD_SAMPLE:      # keeps the fixture under 1 MB: a seeded sample plus its flat indices
                    idx = np.sort(np.random.default_rng(0).choice(a.size, GRAD_SAMPLE, replace=False))
                    a = a.reshape(-1)[idx]
                    d["gidx:" + k] = idx.astype(np.int32)
                d["grad:" + k] = a
        else:
            d.update(out_mean=outs[1].mean().item(), out_std=outs[1].std().item(), coarse_mean=outs[0].mean().item())
        np.savez_compressed(os.path.join(OUT, "fsrnet_%s.npz" % tag), **d)
        print("fsrnet", tag, "total", total.item(), [p.item() for p in parts])


def golden_losses():
    L = R.load("loss/loss.py")
    g = torch.Generator().manual_seed(7)
    a = torch.randn(3, 3, 16, 16, generator=g); t = torch.randn(3, 3, 16, 16, generator=g)
    lm = torch.randn(3, 97, 8, 8, generator=g); hm = torch.rand(3, 8, 8, generator=g)
    lg = torch.randn(3, 11, 8, 8, generator=g); lb = torch.randint(0, 11, (3, 1, 8, 8), generator=g)
    v = [L.MSELossFunc()(a, t), L.MSELoss_Landmark()(lm, hm), L.CrossEntropyLoss2d()(lg, lb)]
    o = [FO.mse97(a, t), FO.landmark_loss(lm, hm), FO.ce2d(lg, lb)]
    for x, y in zip(v, o):
        assert torch.allclose(x, y, rtol=1e-6), (x, y)
    np.savez_compressed(os.path.join(OUT, "losses.npz"), a=a.numpy(), t=t.numpy(), lm=lm.numpy(), hm=hm.numpy(),
                        lg=lg.numpy(), lb=lb.numpy(), values=np.array([x.item() for x in v]))
    print("losses", [x.item() for x in v])


def golden_bicubic():
    from PIL import Image
    import PIL
    rng = np.random.default_rng(20261018)
    d = {"pillow_version": np.array(PIL.__version__)}
    for s, o, n in ((16, 128, 4), (28, 224, 2), (16, 64, 1), (20, 50, 1), (128, 16, 2), (112, 28, 1), (50, 20, 1)):
        src = rng.integers(0, 256, (n, s, s, 3), dtype=np.uint8)
        src[0, :, : s // 2] = 255 * (np.arange(s)[:, None, None] % 2)       # hard edges: exercises the clip
        dst = np.stack([np.asarray(Image.fromarray(a).resize((o, o), Image.BICUBIC)) for a in src])
        assert np.array_equal(dst, BO.bicubic_u8(src, o, o)), (s, o)
        d["src_%d_%d" % (s, o)] = src; d["dst_%d_%d" % (s, o)] = dst
    np.savez_compressed(os.path.join(OUT, "bicubic.npz"), **d)
    print("bicubic ok")


def golden_eval():
    E = R.load("utils/eval.py")
    U = R.load("utils/utils.py")
    rng = np.random.RandomState(11)
    scores = rng.standard_normal((64, 200)).astype(np.float32)
    target = rng.randint(0, 200, 64)
    top1 = E.accuracy(torch.from_numpy(scores), torch.from_numpy(target), topk=(1,))[0].item()
    res = U.accuracy(torch.from_numpy(scores).contiguous(), torch.from_numpy(target), topk=(1,))
    assert abs(EO.accuracy(scores, target, (1,))[0] - top1) < 1e-5 and abs(res[0].item() - top1) < 1e-5
    # make some probes hits so the percentage is non-trivial
    for i in range(0, 64, 3):
        scores[i, target[i]] = 10.0
    top1 = E.accuracy(torch.from_numpy(scores), torch.from_numpy(target), topk=(1,))[0].item()
    o15 = EO.accuracy(scores, target, (1, 5))
    assert abs(o15[0] - top1) < 1e-5
    ref_top5_idx = torch.from_numpy(scores).topk(5, 1, True, True)[1].numpy()
    assert np.array_equal(ref_top5_idx, EO.topk_indices(scores, 5))
    e1 = rng.standard_normal((300, 32)).astype(np.float32); e2 = e1 + 0.8 * rng.standard_normal((300, 32)).astype(np.float32)
    e2[150:] = rng.standard_normal((150, 32)).astype(np.float32)
    same = np.arange(300) < 150
    dist = np.sum(np.square(e1 - e2), 1)
    thr = np.arange(0, 120, 3).astype(np.float64)
    ca = np.array([U.calculate_accuracy(t, dist, same) for t in thr])
    assert np.allclose(ca, np.array([EO.calculate_accuracy(t, dist, same) for t in thr]))
    np.savez_compressed(os.path.join(OUT, "eval.npz"), scores=scores, target=target, top1=top1, top5_idx=ref_top5_idx,
                        top15=np.array(o15), e1=e1, e2=e2, same=same, thr=thr, calc_acc=ca)
    print("eval ok", top1, o15)


def golden_resnet():
    """ResNet_34 (model/resnet.py) + the KD losses of distill_main.py:63,68-70 on the reference's own modules."""
    RM = R.load("model/resnet.py")
    nets, sds = [], []
    for i, seed in enumerate((77, 78, 79)):          # teacher, student, assistant
        torch.manual_seed(seed)
        net = RM.ResNet_34()
        sd = RO.build_resnet34_state_dict(seed)
        ref_sd = net.state_dict()
        assert list(sd) == list(ref_sd) and all(torch.equal(sd[k], ref_sd[k]) for k in sd), "seeded init differs"
        sd = RO.randomize_norm_params(sd, 100 + i)
        net.load_state_dict(sd)
        nets.append(net); sds.append(sd)
    teacher, student, assistant = nets
    teacher.eval(); student.train(); assistant.train()
    x = RO.synthetic_faces(8)
    t_outs = teacher(x)
    s_outs = student(x)
    a_outs = assistant(x)
    mse = torch.nn.MSELoss()
    l_s = mse(s_outs[0], t_outs[0].detach())
    l_a = (mse(t_outs[1] - s_outs[1], a_outs[1]) + mse(t_outs[2] - s_outs[2], a_outs[2])
           + mse(t_outs[3] - s_outs[3], a_outs[3]) + mse(t_outs[4] - s_outs[4], a_outs[4])
           + mse(t_outs[0] - s_outs[0], a_outs[0]))
    names = [k for k, _ in student.named_parameters()]
    g_s = torch.autograd.grad(l_s, list(student.parameters()), retain_graph=True, allow_unused=True)
    g_a = torch.autograd.grad(l_a, list(assistant.parameters()), retain_graph=True, allow_unused=True)
    g_as = torch.autograd.grad(l_a, list(student.parameters()), allow_unused=True)
    o_ls, o_la, og_s, og_a, og_as, (ot, os_, oa) = RO.kd_step(sds[0], sds[1], sds[2], x)
    assert names == RO.resnet34_param_names(sds[1])
    relo = lambda a, b: ((a - b).norm() / (b.norm() + 1e-30)).item()
    for ref_o, ora_o in ((t_outs, ot), (s_outs, os_), (a_outs, oa)):
        errs = [relo(b, a) for a, b in zip(ref_o, ora_o)]
        print("output rel errors (emb, x1..x4):", ["%.2e" % e for e in errs])
        # BatchNorm1d over a batch of 4 amplifies fp32 summation-order noise of the 25088-long dot products
        assert errs[0] < 1e-3 and max(errs[1:]) < 1e-4, errs
    assert abs(l_s.item() - o_ls.item()) <= 1e-5 * abs(l_s.item()) and abs(l_a.item() - o_la.item()) <= 1e-5 * abs(l_a.item())
    rel = lambda a, b: ((a - b).norm() / (b.norm() + 1e-30)).item()
    for gs, og in ((g_s, og_s), (g_a, og_a), (g_as, og_as)):
        # fc.bias feeds a train-mode BatchNorm1d: its gradient is mathematically zero (rounding noise only)
        worst = max((rel(og[k], g), k) for k, g in zip(names, gs) if k not in RO.RESNET_NULL_GRAD)
        print("worst gradient rel error", worst)
        assert worst[0] < 2e-2, worst   # fp32 summation-order noise through 36 train-mode BatchNorms (as for FSRNet)
    nb = {}
    RO.resnet34_forward(sds[1], x, training=True, new_buffers=nb)
    new_sd = student.state_dict()
    for k, v in nb.items():
        assert torch.allclose(v.float(), new_sd[k].float(), rtol=1e-5, atol=1e-6), k
    d = dict(l_s=l_s.item(), l_a=l_a.item(), names=np.array(names),
             emb_t=t_outs[0].detach().numpy(), emb_s=s_outs[0].detach().numpy(), emb_a=a_outs[0].detach().numpy(),
             feat_norms_s=np.array([o.norm().item() for o in s_outs[1:]]),
             feat_means_s=np.array([o.mean().item() for o in s_outs[1:]]),
             gnorm_s=np.array([g.norm().item() for g in g_s]), gnorm_a=np.array([g.norm().item() for g in g_a]),
             gnorm_as=np.array([g.norm().item() for g in g_as]),
             bn1_running_mean=new_sd["bn1.running_mean"].numpy(), bn1_running_var=new_sd["bn1.running_var"].numpy(),
             bn_o2_running_var=new_sd["bn_o2.running_var"].numpy())
    for k in ("bn1.weight", "layer2.0.downsample.1.weight", "layer4.2.bn2.bias", "bn_o2.weight", "fc.bias"):
        i = names.index(k)
        d["gs:" + k] = g_s[i].numpy(); d["ga:" + k] = g_a[i].numpy(); d["gas:" + k] = g_as[i].numpy()
    np.savez_compressed(os.path.join(OUT, "resnet34.npz"), **d)
    print("resnet34 kd", l_s.item(), l_a.item())


def golden_augment():
    """Image.rotate + ImageEnhance.Contrast (helen_loader.py:75-104) against Pillow itself, bit for bit."""
    import random
    from PIL import Image, ImageEnhance
    from oracle import augment_oracle as AO
    rng, nrng = random.Random(5), np.random.default_rng(6)
    d = {}
    for i, (h, w, c) in enumerate([(28, 28, 3), (33, 40, 1), (56, 56, 3), (112, 112, 1), (128, 128, 3), (224, 224, 3)]):
        for rep in range(40 if h <= 56 else 6):        # many random draws are checked, the first of each size is stored
            src = nrng.integers(0, 256, (h, w, c), dtype=np.uint8)
            ang = rng.uniform(-10, 10) if rep % 4 else rng.uniform(-180, 180)
            fac = [rng.uniform(0.9, 1.1), rng.uniform(0.8, 1.2), rng.uniform(0.9, 1.1)]
            im = Image.fromarray(src if c == 3 else src[..., 0])
            rot = im.rotate(ang)
            stages = [np.asarray(rot).reshape(h, w, c)]
            cur = rot
            for f in fac:
                cur = ImageEnhance.Contrast(cur).enhance(f)
                stages.append(np.asarray(cur).reshape(h, w, c))
            assert np.array_equal(AO.rotate_u8(src, ang), stages[0]), (h, w, c, ang)
            o = stages[0]
            for k, f in enumerate(fac):
                o = AO.contrast_u8(o, f)
                assert np.array_equal(o, stages[k + 1]), (h, w, c, k, f)
            assert np.array_equal(AO.augment_u8(src, ang, fac), stages[-1])
            if rep == 0 and h <= 112:                  # the larger sizes are checked here but not stored (random bytes)
                d["src%d" % i], d["angle%d" % i], d["fac%d" % i] = src, np.float64(ang), np.array(fac, np.float64)
                d["rot%d" % i], d["out%d" % i] = stages[0], stages[-1]
                d["coef%d" % i] = AO.rotate_coeffs(h, w, ang)
    # interpolation-only and degenerate factors
    src = nrng.integers(0, 256, (28, 28, 3), dtype=np.uint8)
    im = Image.fromarray(src)
    for f in (0.0, 1.0, 0.5, 1.5, -0.25):
        assert np.array_equal(AO.contrast_u8(src, f), np.asarray(ImageEnhance.Contrast(im).enhance(f))), f
    d["count"] = np.int64(4)
    np.savez_compressed(os.path.join(OUT, "augment.npz"), **d)
    print("augment ok")


def golden_heatmap():
    """Landmark heat-map target: HelenLoader.generate_hm (helen_loader.py:118-143) called on the reference's own class
    (matplotlib / scipy.misc, which the module imports but this method does not use, are stubbed)."""
    import types
    for name in ("matplotlib", "matplotlib.pyplot", "scipy.misc"):
        if name not in sys.modules:
            try:
                __import__(name)
            except Exception:
                sys.modules[name] = types.ModuleType(name)
    HL = R.load("helen_loader.py")
    rng = np.random.RandomState(5)
    lm = (rng.rand(3, 97, 2) * 36.0 - 2.0).astype(np.float32)      # some landmarks fall outside the 32x32 map
    loader = HL.HelenLoader.__new__(HL.HelenLoader)
    ref = np.stack([HL.HelenLoader.generate_hm(loader, height=32, width=32, landmark=[p for p in l.astype(np.float64)], s=1.3)
                    for l in lm])
    ora = np.stack([BO.landmark_heatmap(l, 32, 32, 1.3) for l in lm])
    assert ref.dtype == np.float32 and np.array_equal(ref, ora), np.abs(ref - ora).max()
    np.savez_compressed(os.path.join(OUT, "heatmap.npz"), landmarks=lm, hm=ref)
    print("heatmap ok", float(ref.max()))


def golden_ir50():
    """IR_50 teacher (DISTILLATION/model/model_irse.py) in eval mode on the reference's own module."""
    IR = R.load("DISTILLATION/model/model_irse.py")
    torch.manual_seed(91)
    net = IR.IR_50([112, 112])
    sd = RO.build_ir50_state_dict(91)
    ref_sd = net.state_dict()
    assert list(sd) == list(ref_sd) and all(torch.equal(sd[k], ref_sd[k]) for k in sd), "seeded init differs"
    assert len(list(net.named_parameters())) == 187 and sum(1 for k in sd if k.endswith("running_mean")) == 54
    sd = RO.randomize_bn_everywhere(sd, 191)
    net.load_state_dict(sd)
    net.eval()
    x = RO.synthetic_faces(4, seed=4322)
    with torch.no_grad():
        emb = net(x)
        o = RO.ir50_forward(sd, x)
    rel = ((o - emb).norm() / emb.norm()).item()
    assert rel < 1e-4, rel
    np.savez_compressed(os.path.join(OUT, "ir50.npz"), emb=emb.numpy(), names=np.array(list(sd)),
                        checksums=np.array([v.double().sum().item() for v in RO.build_ir50_state_dict(91).values()]))
    print("ir50 eval forward ok, rel", rel, "emb norm", emb.norm().item())


def golden_gan():
    """OverallNetwork_GAN + Discriminator (model/FSRnet.py:461-486, 512-545) at the only size the reference's Discriminator
    accepts (224 x 224 -> 56 x 56 maps, fc 64*56*56): the oracle restatement is pinned against the reference modules, and
    the fixture keeps the two discriminator embeddings plus how far the oracle's own bf16-storage evaluation moves them."""
    F = R.load("model/FSRnet.py")
    torch.manual_seed(4242)
    net = F.OverallNetwork_GAN()
    net.apply(R.reference_weights_init)
    net.train()
    sd = {k: v.detach().clone() for k, v in net.state_dict().items() if "running_" not in k and "num_batches" not in k}
    g = torch.Generator().manual_seed(99)
    lr, hr = torch.randn(4, 3, 224, 224, generator=g), torch.randn(4, 3, 224, 224, generator=g)
    with torch.no_grad():
        ref = net(lr, hr)
        ours = FO.gan_forward(sd, lr, hr)
        emu = FO.gan_forward(sd, lr, hr, FO.Precision("bf16"))
    for a, b, name in zip(ref, ours, ("sr", "coarse", "landmark", "parsing", "embedding1", "embedding2")):
        assert torch.allclose(a, b, rtol=1e-3, atol=2e-4), (name, (a - b).abs().max())
    rel = lambda a, b: ((a - b).double().norm() / b.double().norm()).item()
    np.savez_compressed(os.path.join(OUT, "gan224.npz"), embedding1=ref[4].numpy(), embedding2=ref[5].numpy(),
                        sr_mean=ref[0].mean().item(), sr_std=ref[0].std().item(),
                        emu_rel=np.array([rel(e, r) for e, r in zip(emu, ref)]),
                        keys=np.array(list(sd.keys())))
    print("gan224: oracle == reference; bf16-storage deviation per output", [round(rel(e, r), 4) for e, r in zip(emu, ref)])


def golden_sr():
    """SUPER_RESOLUTION/model/FSRnet.py:251-416: the four sub-networks of the newer FSRNet variant.  The restatement in
    oracle/sr_oracle.py is pinned against the reference's modules; the fixture keeps the small outputs, statistics of the
    large ones and the deviation of the oracle's own bf16-storage evaluation."""
    from oracle import sr_oracle as SO
    F = R.load("SUPER_RESOLUTION/model/FSRnet.py")
    g = torch.Generator().manual_seed(31)
    x = torch.randn(2, 3, 64, 64, generator=g)
    xd = torch.randn(2, 128, 64, 64, generator=g)
    rel = lambda a, b: ((a - b).double().norm() / b.double().norm()).item()
    out = {}
    for seed, (name, cls, fn, inp) in enumerate((("coarse", F.Coarse_SR_Network, SO.coarse_forward, x),
                                                 ("encoder", F.Fine_SR_Encoder, SO.encoder_forward, x),
                                                 ("prior", F.Prior_Estimation_Network, SO.prior_forward, x),
                                                 ("decoder", F.Fine_SR_Decoder, SO.decoder_forward, xd)), start=700):
        torch.manual_seed(seed)
        net = cls()
        with torch.no_grad():                    # non-trivial affine / PReLU parameters
            for k, p in net.named_parameters():
                if p.dim() == 1:
                    p.add_(0.2 * torch.randn_like(p))
        net.train()
        sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
        with torch.no_grad():
            ref = net(inp)
            ours = fn(sd, inp)
            emu = fn(sd, inp, pr=FO.Precision("bf16"))
        ref = ref if isinstance(ref, tuple) else (ref,)
        ours = ours if isinstance(ours, tuple) else (ours,)
        emu = emu if isinstance(emu, tuple) else (emu,)
        for a, b in zip(ref, ours):
            assert torch.allclose(a, b, rtol=1e-3, atol=2e-4), (name, (a - b).abs().max())
        out[name + "_seed"] = seed
        for i, (a, e) in enumerate(zip(ref, emu)):
            out["%s_%d_emu_rel" % (name, i)] = rel(e, a)
            out["%s_%d_mean_std_norm" % (name, i)] = np.array([a.mean().item(), a.std().item(), a.norm().item()])
            out["%s_%d_sample" % (name, i)] = a[:, :, ::8, ::8].numpy()
        print("sr", name, "oracle == reference; bf16-storage deviation", [round(rel(e, a), 4) for a, e in zip(ref, emu)])
    np.savez_compressed(os.path.join(OUT, "sr_variant.npz"), **out)


if __name__ == "__main__":
    assert R.available(), "reference tree not present"
    os.makedirs(OUT, exist_ok=True)
    which = sys.argv[1:] or ["losses", "bicubic", "eval", "fsrnet", "resnet", "ir50", "heatmap", "augment", "gan", "sr"]
    for w in which:
        globals()["golden_" + w]()
