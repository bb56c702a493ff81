"""Per-kernel parity on the GPU: every C-ABI family against a plain fp32 PyTorch (CPU) statement of the same op on
identical bf16-representable inputs.  Tolerances: outputs stored as bf16 carry one rounding (2^-9 relative per
element) -> norm-wise 5e-3; fp32 results (weight gradients, losses) -> 1e-4 (north_star tolerance)."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.util import bf16_round, max_abs, nhwc_from, rel_err, to_nchw

pytestmark = pytest.mark.gpu

BF16_TOL = 5e-3
F32_TOL = 1e-4


def _ops():
    from crfr_b200 import ops
    return ops


def _L():
    from crfr_b200 import _lib
    return _lib


# (cin, cout, k, stride, pad, h) - the edge layers of FSRNet that stay on the CUDA-core engine, plus a 64->64 case
DIRECT_SHAPES = [
    (3, 64, 3, 1, 1, 32),      # coarse conv_input  (FSRnet.py:312)
    (64, 3, 3, 1, 1, 32),      # conv_mid / conv_out (:318, :439)
    (3, 64, 7, 4, 3, 64),      # encoder stem       (:345)
    (3, 128, 7, 4, 3, 32),     # prior stem         (:384)
    (128, 11, 1, 1, 0, 16),    # fc                 (:391)
    (128, 97, 1, 1, 0, 16),    # fc_landmark        (:392)
    (64, 64, 3, 1, 1, 16),     # residual conv on the direct engine (cross-check path)
    (192, 64, 3, 1, 1, 8),     # decoder conv_input (:432)
    (3, 64, 7, 2, 3, 112),     # ResNet stem        (model/resnet.py:158)
    (64, 128, 3, 2, 1, 56),    # layer2.0.conv1     (model/resnet.py:193-200: stage transition)
    (64, 128, 1, 2, 0, 56),    # layer2.0.downsample.0
    (256, 512, 3, 2, 1, 14),   # layer4.0.conv1
    (256, 512, 1, 2, 0, 14),   # layer4.0.downsample.0
    (3, 64, 7, 4, 3, 48),      # stems at sizes whose pixel count is no multiple of the gather kernel's 64-pixel blocks
    (3, 64, 7, 2, 3, 50),
    (3, 64, 3, 1, 1, 112),     # IR stem            (model/model_irse.py:131)
]


@pytest.mark.parametrize("engine", ["direct", "auto"])
@pytest.mark.parametrize("cin,cout,k,stride,pad,h", DIRECT_SHAPES)
def test_edge_conv_fwd_dgrad_wgrad(cuda, cin, cout, k, stride, pad, h, engine):
    """engine 'direct' = CUDA-core kernels; 'auto' = the lowered im2col + tcgen05 GEMM recipes where they apply."""
    ops, L = _ops(), _L()
    ENG = L.ENGINE_DIRECT if engine == "direct" else L.ENGINE_AUTO
    g = torch.Generator().manual_seed(cin * 1000 + cout)
    n = 2
    x = bf16_round(torch.randn(n, cin, h, h, generator=g))
    w = bf16_round(torch.randn(cout, cin, k, k, generator=g) * 0.1)
    b = torch.randn(cout, generator=g)
    xr = x.clone().requires_grad_(True)
    wr = w.clone().requires_grad_(True)
    br = b.clone().requires_grad_(True)
    y_ref = F.conv2d(xr, wr, br, stride, pad)
    dy = bf16_round(torch.randn(y_ref.shape, generator=g))
    y_ref.backward(dy)

    in_ld = 4 if cin < 8 else cin
    out_ld = 4 if cout < 8 else (cout + 7) // 8 * 8
    xg = nhwc_from(x, in_ld)
    wp = ops.pack_conv_weight(w.cuda())
    y, _, _ = ops.conv_fwd(xg, wp, cin, cout, k, stride, pad, bias=b.cuda(), engine=ENG)
    assert rel_err(to_nchw(y, cout), y_ref) < BF16_TOL
    _, yn, _ = ops.conv_fwd(xg, wp, cin, cout, k, stride, pad, bias=b.cuda(), engine=ENG, nchw_out=True)
    assert rel_err(yn, y_ref) < F32_TOL

    dyg = nhwc_from(dy, out_ld)
    wt = ops.pack_conv_weight(w.cuda(), for_dgrad=True)
    dx = ops.conv_dgrad(dyg, wt, (n, h, h, in_ld), cin, cout, k, stride, pad, engine=ENG)
    assert rel_err(to_nchw(dx, cin), xr.grad) < BF16_TOL
    if in_ld > cin:
        assert float(dx[..., cin:].float().abs().max()) == 0.0     # channel padding stays zero
    dw, db = ops.conv_wgrad(xg, dyg, cin, cout, k, stride, pad, engine=ENG, want_bias=True)
    assert rel_err(dw, wr.grad) < F32_TOL
    assert rel_err(db, br.grad) < F32_TOL


@pytest.mark.parametrize("engine", ["direct", "auto"])
def test_deconv(cuda, engine):
    """ConvTranspose2d 7x7 s4 p2 op1 64->64 (FSRnet.py:436)."""
    ops, L = _ops(), _L()
    ENG = L.ENGINE_DIRECT if engine == "direct" else L.ENGINE_AUTO
    g = torch.Generator().manual_seed(7)
    n, c, h = 2, 64, 8
    x = bf16_round(torch.randn(n, c, h, h, generator=g))
    w = bf16_round(torch.randn(c, c, 7, 7, generator=g) * 0.05)
    b = torch.randn(c, generator=g)
    xr, wr, br = (t.clone().requires_grad_(True) for t in (x, w, b))
    y_ref = F.conv_transpose2d(xr, wr, br, 4, 2, 1)
    dy = bf16_round(torch.randn(y_ref.shape, generator=g))
    y_ref.backward(dy)
    xg = nhwc_from(x)
    wp = ops.pack_conv_weight(w.cuda(), transposed=True)
    y, _, st = ops.conv_fwd(xg, wp, c, c, 7, 4, 2, bias=b.cuda(), engine=ENG, transposed=True,
                            out_hw=(4 * h, 4 * h), want_stats=True)
    assert rel_err(to_nchw(y), y_ref) < BF16_TOL
    yb = to_nchw(y)
    assert max_abs(st[..., 0], yb.mean((2, 3))) < 1e-4
    assert rel_err(st[..., 1], 1.0 / torch.sqrt(yb.var((2, 3), unbiased=False) + 1e-5)) < 1e-4
    dyg = nhwc_from(dy)
    wt = ops.pack_conv_weight(w.cuda(), for_dgrad=True, transposed=True)
    dx = ops.conv_dgrad(dyg, wt, (n, h, h, c), c, c, 7, 4, 2, engine=ENG, transposed=True)
    assert rel_err(to_nchw(dx), xr.grad) < BF16_TOL
    dw, db = ops.conv_wgrad(xg, dyg, c, c, 7, 4, 2, engine=ENG, transposed=True, want_bias=True)
    assert rel_err(dw, wr.grad) < F32_TOL
    assert rel_err(db, br.grad) < F32_TOL


@pytest.mark.parametrize("n,c,h,w,ld,zero_to", [(2, 3, 16, 16, 4, 4), (3, 97, 9, 7, 128, 97), (2, 64, 56, 56, 64, 64),
                                                 (3, 40, 5, 33, 48, 48), (2, 512, 7, 7, 512, 512)])
def test_layout_conversions(cuda, n, c, h, w, ld, zero_to):
    """fp32 NCHW <-> bf16 NHWC at the nn.Module boundary (per-pixel kernels for images, tiled transposes for feature
    maps): exact on bf16-representable data, zero fill of [c, zero_to), channels beyond zero_to left untouched."""
    ops = _ops()
    g = torch.Generator().manual_seed(c * h + w)
    x = bf16_round(torch.randn(n, c, h, w, generator=g))
    sentinel = 7.0
    out = torch.full((n, h, w, ld), sentinel, dtype=torch.bfloat16, device="cuda")
    from crfr_b200 import _lib as L
    L.call("crfr_nchw_f32_to_nhwc_bf16", ops.ptr(x.cuda()), ops.ptr(out), n, c, h, w, ld, zero_to, ops.stream())
    torch.cuda.synchronize()
    ref = x.permute(0, 2, 3, 1)
    assert torch.equal(out[..., :c].float().cpu(), ref)
    assert float(out[..., c:zero_to].float().abs().max()) == 0.0 if zero_to > c else True
    if ld > zero_to:
        assert torch.equal(out[..., zero_to:].float().cpu(), torch.full((n, h, w, ld - zero_to), sentinel))
    back = ops.nhwc_to_nchw(out, c)
    assert torch.equal(back.cpu(), x)


@pytest.mark.parametrize("n,h,w,c", [(16, 128, 128, 3), (5, 112, 112, 1), (3, 33, 40, 3), (2, 224, 224, 3)])
def test_augment_u8_bit_exact(cuda, golden_dir, n, h, w, c):
    """Rotation + contrast enhancements of helen_loader.py:75-104 on the device: bit-exact with the oracle (pinned to
    Pillow) on random batches, with the stored Pillow vectors, and for the degenerate factors."""
    import random
    from oracle import augment_oracle as AO
    ops = _ops()
    rng, nrng = random.Random(n * h + c), np.random.default_rng(h + w)
    src = nrng.integers(0, 256, (n, h, w, c), dtype=np.uint8)
    angles = [rng.uniform(-10, 10) for _ in range(n)]
    angles[0] = 0.0
    fac = np.array([[rng.uniform(0.9, 1.1), rng.uniform(0.8, 1.2), rng.uniform(0.9, 1.1)] for _ in range(n)])
    fac[-1] = [0.0, 1.0, 1.5]
    out = ops.augment_u8(torch.from_numpy(src).cuda(), angles, fac).cpu().numpy()
    rot = ops.augment_u8(torch.from_numpy(src).cuda(), angles).cpu().numpy()
    for i in range(n):
        assert np.array_equal(rot[i], AO.rotate_u8(src[i], angles[i])), i
        assert np.array_equal(out[i], AO.augment_u8(src[i], angles[i], fac[i])), i
    g = np.load(os.path.join(golden_dir, "augment.npz"))
    for i in range(int(g["count"])):
        s_, ang, f_ = g["src%d" % i], float(g["angle%d" % i]), g["fac%d" % i]
        o = ops.augment_u8(torch.from_numpy(s_[None]).cuda(), [ang], f_[None]).cpu().numpy()[0]
        assert np.array_equal(o, g["out%d" % i]), i


def test_fhn_pipeline_rotate_crop_resample_enhance(cuda):
    """SUPER_RESOLUTION/FHN_loader.py:55-86 on the device, stage by stage against the Pillow-pinned oracles (bit-exact):
    rotate, random 112-crop, LR synthesis (down by 2/4/8, bicubic back up), three contrast enhancements on both images."""
    import random
    from oracle import augment_oracle as AO
    from oracle import bicubic_oracle as BO
    ops = _ops()
    rng, nrng = random.Random(12), np.random.default_rng(13)
    n = 6
    src = nrng.integers(0, 256, (n, 128, 128, 3), dtype=np.uint8)
    angles = [rng.uniform(-20, 20) for _ in range(n)]
    offs = [(rng.randint(0, 16), rng.randint(0, 16)) for _ in range(n)]
    fac = np.array([[rng.uniform(0.93, 1.07), rng.uniform(0.92, 1.08), rng.uniform(0.93, 1.07)] for _ in range(n)])
    scales = [2, 4, 8, 8, 4, 2]
    rot = ops.augment_u8(torch.from_numpy(src).cuda(), angles)
    sr = ops.crop_u8(rot, offs, 112, 112)
    sr_np = sr.cpu().numpy()
    zeros = [0.0] * n
    hr = ops.augment_u8(sr, zeros, fac).cpu().numpy()
    for i in range(n):
        ref_sr = AO.rotate_u8(src[i], angles[i])[offs[i][0]:offs[i][0] + 112, offs[i][1]:offs[i][1] + 112]
        assert np.array_equal(sr_np[i], ref_sr), i
        assert np.array_equal(hr[i], AO.augment_u8(ref_sr, 0.0, fac[i])), i
        s_ = 128 // scales[i]
        small, _ = ops.bicubic_u8(sr[i:i + 1], s_, s_)
        lr, _ = ops.bicubic_u8(small, 112, 112)
        ref_lr = BO.bicubic_u8(BO.bicubic_u8(ref_sr, s_, s_), 112, 112)
        assert np.array_equal(lr[0].cpu().numpy(), ref_lr), i
        lr_e = ops.augment_u8(lr, [0.0], fac[i:i + 1]).cpu().numpy()[0]
        assert np.array_equal(lr_e, AO.augment_u8(ref_lr, 0.0, fac[i])), i
    with pytest.raises(ValueError):
        ops.crop_u8(rot, [(20, 0)] * n, 112, 112)


def _prelu(x, a):
    return torch.clamp(x, min=0) + a.view(1, -1, 1, 1) * torch.clamp(x, max=0)


@pytest.mark.parametrize("c,h,affine,act,res", [(64, 32, True, True, True), (128, 8, False, True, True),
                                                 (64, 16, True, False, False), (128, 16, True, True, False)])
def test_instance_norm_prelu_add(cuda, c, h, affine, act, res):
    """IN + PReLU + residual forward/backward (FSRnet.py:75-98, 105-135)."""
    ops = _ops()
    g = torch.Generator().manual_seed(c + h)
    n = 3
    y = bf16_round(torch.randn(n, c, h, h, generator=g) * 2 + 0.5)
    r = bf16_round(torch.randn(n, c, h, h, generator=g)) if res else None
    gamma = (torch.rand(c, generator=g) + 0.5) if affine else None
    beta = torch.randn(c, generator=g) if affine else None
    alpha = (torch.rand(c, generator=g) * 0.5) if act else None
    leaves = [t.clone().requires_grad_(True) if t is not None else None for t in (y, r, gamma, beta, alpha)]
    yr, rr, gr, br, ar = leaves
    z = F.instance_norm(yr, weight=gr, bias=br, eps=1e-5)
    if res:
        z = z + rr
    out_ref = _prelu(z, ar) if act else z
    dout = bf16_round(torch.randn(out_ref.shape, generator=g))
    dout2 = bf16_round(torch.randn(out_ref.shape, generator=g))
    out_ref.backward(dout + dout2)

    cu = lambda t: None if t is None else t.cuda()
    yg = nhwc_from(y)
    stats = ops.norm_stats(yg)
    assert max_abs(stats[..., 0], y.mean((2, 3))) < 1e-4
    out = ops.norm_act_fwd(yg, stats, cu(gamma), cu(beta), cu(alpha), res=None if r is None else nhwc_from(r))
    assert rel_err(to_nchw(out), out_ref) < BF16_TOL
    dz, dy, dg, db, da = ops.norm_act_bwd(nhwc_from(dout), yg, stats, cu(gamma), cu(beta), cu(alpha),
                                          res=None if r is None else nhwc_from(r), dout_b=nhwc_from(dout2))
    # two bf16 roundings (dz, dy): measured 1.7e-3 .. 2.5e-3 on B200 (tools/norm_bwd_error_probe.py); north_star bound 1e-2
    assert rel_err(to_nchw(dy), yr.grad) < 6e-3
    if res:
        assert rel_err(to_nchw(dz), rr.grad) < BF16_TOL
    if affine:
        assert rel_err(dg, gr.grad) < 1e-2 and rel_err(db, br.grad) < 1e-2
    if act:
        assert rel_err(da, ar.grad) < 1e-2


@pytest.mark.parametrize("n,c,h,res,two", [(40, 64, 32, True, True), (40, 64, 32, False, False), (24, 128, 16, True, False),
                                           (300, 64, 8, False, True), (5, 64, 40, True, True)])
def test_instance_norm_bwd_implementations(cuda, n, c, h, res, two):
    """The two implementations of crfr_norm_act_bwd - register-staged passes (0) and the persistent TMA-fed passes (1),
    whose CTAs own contiguous pixel ranges that straddle image boundaries - against autograd and against each other, on
    enough images that every CTA of the persistent grid has work."""
    ops = _ops()
    g = torch.Generator().manual_seed(n + c + h)
    y = bf16_round(torch.randn(n, c, h, h, generator=g) * 1.7 + 0.8)
    r = bf16_round(torch.randn(n, c, h, h, generator=g)) if res else None
    gamma, beta = torch.rand(c, generator=g) + 0.5, torch.randn(c, generator=g)
    alpha = torch.rand(c, generator=g) * 0.5
    yr, gr, br, ar = (t.clone().requires_grad_(True) for t in (y, gamma, beta, alpha))
    rr = r.clone().requires_grad_(True) if res else None
    z = F.instance_norm(yr, weight=gr, bias=br, eps=1e-5)
    if res:
        z = z + rr
    out_ref = _prelu(z, ar)
    dout = bf16_round(torch.randn(out_ref.shape, generator=g))
    dout2 = bf16_round(torch.randn(out_ref.shape, generator=g)) if two else None
    out_ref.backward(dout + dout2 if two else dout)
    yg = nhwc_from(y)
    stats = ops.norm_stats(yg)
    args = (nhwc_from(dout), yg, stats, gamma.cuda(), beta.cuda(), alpha.cuda())
    kw = dict(res=None if r is None else nhwc_from(r), dout_b=None if dout2 is None else nhwc_from(dout2))
    results = {}
    try:
        for mode in (0, 1):
            ops.set_option("norm_bwd_impl", mode)
            results[mode] = ops.norm_act_bwd(*args, **kw)
            torch.cuda.synchronize()
        ops.set_option("norm_bwd_impl", 1)
        again = ops.norm_act_bwd(*args, **kw)
    finally:
        ops.set_option("norm_bwd_impl", -1)
    for mode in (0, 1):
        dz, dy, dg, db, da = results[mode]
        assert rel_err(to_nchw(dy), yr.grad) < 6e-3          # measured <= 2.5e-3 (tools/norm_bwd_error_probe.py)
        if res:
            assert rel_err(to_nchw(dz), rr.grad) < BF16_TOL
        assert rel_err(dg, gr.grad) < 5e-3 and rel_err(db, br.grad) < 5e-3 and rel_err(da, ar.grad) < 1e-4
    # same per-element arithmetic up to the association of the fp32 sums: dz identical, dy within one bf16 ulp
    if results[0][0] is not None:
        assert torch.equal(results[0][0], results[1][0])
    assert rel_err(results[1][1].float(), results[0][1].float()) < 3e-3
    for k in (2, 3, 4):
        assert rel_err(results[1][k], results[0][k]) < 1e-5
    # deterministic: a second run reproduces every bit
    for a, b in zip(again, results[1]):
        assert (a is None and b is None) or torch.equal(a, b)


def test_instance_norm_bwd_full_size_properties(cuda):
    """BASELINE.json config 2 size (128 images x 64 ch x 128 x 128, the shape of 36 of the 98 layers), checked through
    properties that do not need a CPU reference: dy of an InstanceNorm is orthogonal to 1 and to x_hat over every
    (image, channel) plane; dz is the masked / scaled dout exactly; images are independent (a permuted batch gives the
    permuted result); the two implementations agree."""
    ops = _ops()
    n, c, h = 128, 64, 128
    g = torch.Generator(device="cuda").manual_seed(77)
    mk = lambda s=1.0, m=0.0: (torch.randn(n, h, h, c, generator=g, device="cuda") * s + m).to(torch.bfloat16)
    y, res, dout = mk(1.5, 0.4), mk(), mk()
    gamma = torch.rand(c, generator=g, device="cuda") + 0.5
    beta = torch.randn(c, generator=g, device="cuda")
    alpha = torch.rand(c, generator=g, device="cuda") * 0.5
    stats = ops.norm_stats(y)
    dz, dy, dg, db, da = ops.norm_act_bwd(dout, y, stats, gamma, beta, alpha, res=res)
    torch.cuda.synchronize()
    # dz = dout * (z > 0 ? 1 : alpha), z = gamma * x_hat + beta + res (fp32), rounded once to bf16
    xh = (y.float() - stats[:, None, None, :, 0]) * stats[:, None, None, :, 1]
    z = xh * gamma + beta + res.float()
    mask = torch.where(z > 0, torch.ones_like(z), alpha.expand_as(z))
    dz_ref = (dout.float() * mask).to(torch.bfloat16)
    mism = (dz != dz_ref).float().mean().item()       # z within an ulp of 0 may take the other branch
    assert mism < 1e-5, mism
    del z, mask, dz_ref
    # orthogonality: sum_p dy = 0 and sum_p dy * x_hat = 0 per (image, channel), up to the bf16 rounding of dy
    dyf = dy.float()
    scale = dyf.abs().sum((1, 2))
    assert (dyf.sum((1, 2)).abs() / scale).max().item() < 2e-3
    assert ((dyf * xh).sum((1, 2)).abs() / scale).max().item() < 2e-3
    # parameter gradients against their definitions
    dzf = dz.float()
    assert rel_err(db, dzf.sum((0, 1, 2))) < 1e-4 and rel_err(dg, (dzf * xh).sum((0, 1, 2))) < 1e-4
    del dyf, dzf, xh
    # independence of the images: reversed batch -> reversed result (sums are regrouped: fp32 rounding only)
    flip = lambda t: t.flip(0).contiguous()
    dz2, dy2, dg2, db2, da2 = ops.norm_act_bwd(flip(dout), flip(y), flip(stats), gamma, beta, alpha, res=flip(res))
    assert torch.equal(flip(dz2), dz)
    assert rel_err(flip(dy2).float(), dy.float()) < 1e-3
    assert rel_err(dg2, dg) < 1e-5 and rel_err(da2, da) < 1e-5
    # the register-staged implementation
    try:
        ops.set_option("norm_bwd_impl", 0)
        dz0, dy0, dg0, db0, da0 = ops.norm_act_bwd(dout, y, stats, gamma, beta, alpha, res=res)
    finally:
        ops.set_option("norm_bwd_impl", -1)
    assert torch.equal(dz0, dz) and rel_err(dy0.float(), dy.float()) < 1e-3
    assert rel_err(dg0, dg) < 1e-5 and rel_err(db0, db) < 1e-5 and rel_err(da0, da) < 1e-5


@pytest.mark.parametrize("n,c,h,res,bn", [(5, 64, 40, True, False), (40, 64, 32, False, False), (7, 128, 16, True, False),
                                          (8, 256, 14, True, True), (3, 512, 5, False, True)])
def test_norm_fwd_stream_matches_register_kernel(cuda, n, c, h, res, bn):
    """The TMA-fed forward pass (crfr_set_option norm_fwd_stream) performs the same operations per element as the
    register-staged kernel: identical bits, for InstanceNorm + PReLU (+ residual) and for BatchNorm + ReLU."""
    ops = _ops()
    g = torch.Generator().manual_seed(n * c + h)
    y = nhwc_from(bf16_round(torch.randn(n, c, h, h, generator=g) * 1.3 + 0.2))
    r = nhwc_from(bf16_round(torch.randn(n, c, h, h, generator=g))) if res else None
    gamma, beta = (torch.rand(c, generator=g) + 0.5).cuda(), torch.randn(c, generator=g).cuda()
    alpha = None if bn else (torch.rand(c, generator=g) * 0.5).cuda()
    stats = ops.norm_stats(y, groups_as_batch=bn)
    outs = []
    try:
        for mode in (0, 1):
            ops.set_option("norm_fwd_stream", mode)
            outs.append(ops.norm_act_fwd(y, stats, gamma, beta, alpha, relu=bn, res=r, batch_norm=bn))
            torch.cuda.synchronize()
    finally:
        ops.set_option("norm_fwd_stream", 1)
    assert torch.equal(outs[0], outs[1])


def test_batch_norm_relu_mode(cuda):
    """The same kernels with one statistic group over the whole batch = train-mode BatchNorm2d + ReLU (resnet.py:24-28)."""
    ops = _ops()
    g = torch.Generator().manual_seed(5)
    n, c, h = 4, 64, 14
    y = bf16_round(torch.randn(n, c, h, h, generator=g) * 1.5 - 0.3)
    gamma, beta = torch.rand(c, generator=g) + 0.5, torch.randn(c, generator=g)
    yr, gr, br = (t.clone().requires_grad_(True) for t in (y, gamma, beta))
    out_ref = F.relu(F.batch_norm(yr, None, None, gr, br, True, 0.1, 1e-5))
    dout = bf16_round(torch.randn(out_ref.shape, generator=g))
    out_ref.backward(dout)
    yg = nhwc_from(y)
    stats = ops.norm_stats(yg, groups_as_batch=True)
    out = ops.norm_act_fwd(yg, stats, gamma.cuda(), beta.cuda(), relu=True, batch_norm=True)
    assert rel_err(to_nchw(out), out_ref) < BF16_TOL
    dz, dy, dg, db, _ = ops.norm_act_bwd(nhwc_from(dout), yg, stats, gamma.cuda(), beta.cuda(), relu=True, batch_norm=True)
    assert rel_err(to_nchw(dy), yr.grad) < 1e-2
    assert rel_err(dg, gr.grad) < 1e-2 and rel_err(db, br.grad) < 1e-2


@pytest.mark.parametrize("n,c,h", [(8, 128, 28), (8, 256, 14), (8, 512, 7), (3, 512, 5)])
def test_batch_norm_bwd_wide_channels(cuda, n, c, h):
    """BatchNorm backward at the channel widths of ResNet_34's later stages (model/resnet.py:193-200), where one TMA box
    of the streaming kernels is narrower than a swizzle atom: both implementations against autograd."""
    ops = _ops()
    g = torch.Generator().manual_seed(c + h)
    y = bf16_round(torch.randn(n, c, h, h, generator=g) * 1.5 - 0.3)
    r = bf16_round(torch.randn(n, c, h, h, generator=g))
    gamma, beta = torch.rand(c, generator=g) + 0.5, torch.randn(c, generator=g)
    yr, rr, gr, br = (t.clone().requires_grad_(True) for t in (y, r, gamma, beta))
    out_ref = F.relu(F.batch_norm(yr, None, None, gr, br, True, 0.1, 1e-5) + rr)
    dout = bf16_round(torch.randn(out_ref.shape, generator=g))
    out_ref.backward(dout)
    yg = nhwc_from(y)
    stats = ops.norm_stats(yg, groups_as_batch=True)
    try:
        for mode in (0, 1):
            ops.set_option("norm_bwd_impl", mode)
            dz, dy, dg, db, _ = ops.norm_act_bwd(nhwc_from(dout), yg, stats, gamma.cuda(), beta.cuda(), relu=True,
                                                 res=nhwc_from(r), batch_norm=True)
            assert rel_err(to_nchw(dy), yr.grad) < 1e-2, mode
            assert rel_err(to_nchw(dz), rr.grad) < BF16_TOL, mode
            assert rel_err(dg, gr.grad) < 1e-2 and rel_err(db, br.grad) < 1e-2, mode
    finally:
        ops.set_option("norm_bwd_impl", -1)


def test_pool_upsample_add(cuda):
    ops = _ops()
    g = torch.Generator().manual_seed(9)
    n, c, h = 2, 128, 16
    x = bf16_round(torch.randn(n, c, h, h, generator=g))
    xr = x.clone().requires_grad_(True)
    p_ref = F.max_pool2d(xr, 2, 2)
    dp = bf16_round(torch.randn(p_ref.shape, generator=g))
    p_ref.backward(dp)
    xg = nhwc_from(x)
    assert max_abs(to_nchw(ops.maxpool2_fwd(xg)), p_ref) == 0.0
    assert max_abs(to_nchw(ops.maxpool2_bwd(xg, nhwc_from(dp))), xr.grad) == 0.0
    low = bf16_round(torch.randn(n, c, h // 2, h // 2, generator=g))
    lr_ = low.clone().requires_grad_(True)
    u_ref = x + F.interpolate(lr_, scale_factor=2)
    du = bf16_round(torch.randn(u_ref.shape, generator=g))
    u_ref.backward(du)
    assert rel_err(to_nchw(ops.upnearest2_add_fwd(xg, nhwc_from(low))), u_ref) < BF16_TOL
    assert rel_err(to_nchw(ops.upnearest2_bwd(nhwc_from(du))), lr_.grad) < BF16_TOL
    a3 = ops.add_n(xg, nhwc_from(du), nhwc_from(x))
    assert rel_err(to_nchw(a3), x + du + x) < BF16_TOL


def test_losses_against_golden_and_torch(cuda, golden_dir):
    import os
    ops = _ops()
    gd = np.load(os.path.join(golden_dir, "losses.npz"))
    a, t, lm, hm, lg, lb = (torch.from_numpy(gd[k]) for k in ("a", "t", "lm", "hm", "lg", "lb"))
    ar, lmr, lgr = (v.clone().requires_grad_(True) for v in (a, lm, lg))
    l1 = ((ar - t) ** 2).mean() * 97.0
    l2 = ((lmr.sum(1) - hm) ** 2).mean() * 97.0
    l3 = F.nll_loss(F.log_softmax(lgr, 1), lb.squeeze())
    (0.7 * l1 + 0.3 * l2 + 1.3 * l3).backward()
    loss, dx = ops.loss_mse97(a.cuda(), t.cuda(), 0.7)
    assert abs(loss.item() - gd["values"][0]) < F32_TOL * abs(gd["values"][0])
    assert rel_err(to_nchw(dx, 3), ar.grad) < BF16_TOL and float(dx[..., 3].float().abs().max()) == 0.0
    n, _, h, w = lm.shape
    buf = torch.zeros((n, h, w, 112), dtype=torch.bfloat16, device="cuda")
    loss = ops.loss_landmark(lm.cuda(), hm.cuda(), 0.3, buf, 11)
    assert abs(loss.item() - gd["values"][1]) < F32_TOL * abs(gd["values"][1])
    loss = ops.loss_ce2d(lg.cuda(), lb.cuda(), 1.3, buf, 0)
    assert abs(loss.item() - gd["values"][2]) < F32_TOL * abs(gd["values"][2])
    assert rel_err(to_nchw(buf[..., 11:108]), lmr.grad) < BF16_TOL
    assert rel_err(to_nchw(buf[..., :11]), lgr.grad) < BF16_TOL
    assert float(buf[..., 108:].float().abs().max()) == 0.0


@pytest.mark.parametrize("n,h,w,ld,coff", [(1, 3, 5, 104, 0), (3, 7, 9, 112, 11), (2, 8, 8, 100, 2), (5, 5, 7, 99, 1)])
def test_landmark_gradient_rows_ragged(cuda, n, h, w, ld, coff):
    """The landmark loss writes each pixel's 97 equal gradients as one row of the heads' gradient buffer, a warp per 32 pixels:
    pixel counts that are no multiple of the warp, rows that start on odd and even elements, odd row pitches; everything
    outside the rows stays untouched."""
    ops = _ops()
    g = torch.Generator().manual_seed(n * 100 + coff)
    lm = torch.randn(n, 97, h, w, generator=g)
    hm = torch.rand(n, h, w, generator=g)
    lmr = lm.clone().requires_grad_(True)
    (0.3 * ((lmr.sum(1) - hm) ** 2).mean() * 97.0).backward()
    buf = torch.full((n, h, w, ld), 7.0, dtype=torch.bfloat16, device="cuda")
    loss = ops.loss_landmark(lm.cuda(), hm.cuda(), 0.3, buf, coff)
    ref = (((lm.sum(1) - hm) ** 2).mean() * 97.0).item()
    assert abs(loss.item() - ref) < F32_TOL * abs(ref)
    assert rel_err(to_nchw(buf[..., coff:coff + 97]), lmr.grad) < BF16_TOL
    rest = torch.cat([buf[..., :coff], buf[..., coff + 97:]], -1).float()
    assert bool((rest == 7.0).all())


def test_loss_modules_dropin(cuda):
    """MSELossFunc / MSELoss_Landmark / CrossEntropyLoss2d keep the reference call signature and autograd behaviour."""
    from crfr_b200.loss import CrossEntropyLoss2d, MSELoss_Landmark, MSELossFunc
    from oracle import fsrnet_oracle as FO
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 3, 32, 32, generator=g); t = torch.randn(2, 3, 32, 32, generator=g)
    lm = torch.randn(2, 97, 8, 8, generator=g); hm = torch.rand(2, 8, 8, generator=g)
    lg = torch.randn(2, 11, 8, 8, generator=g); lb = torch.randint(0, 11, (2, 1, 8, 8), generator=g)
    refs = []
    for fn, (p, q) in ((FO.mse97, (x, t)), (FO.landmark_loss, (lm, hm)), (FO.ce2d, (lg, lb))):
        pr = p.clone().requires_grad_(True)
        v = fn(pr, q)
        (2.0 * v).backward()
        refs.append((v.item(), pr.grad))
    for mod, (p, q), (v_ref, g_ref) in zip((MSELossFunc(), MSELoss_Landmark(), CrossEntropyLoss2d()),
                                           ((x, t), (lm, hm), (lg, lb)), refs):
        pc = p.cuda().requires_grad_(True)
        v = mod(pc, q.cuda())
        (2.0 * v).backward()
        assert abs(v.item() - v_ref) < F32_TOL * abs(v_ref)
        assert rel_err(pc.grad, g_ref) < BF16_TOL


def test_kd_loss(cuda):
    """distill_main.py:63,68-70: MSE(s, t) and MSE(t - s, a), fp32 embeddings and bf16 stage maps."""
    ops = _ops()
    g = torch.Generator().manual_seed(21)
    for dtype, shape in ((torch.float32, (16, 512)), (torch.bfloat16, (4, 14, 14, 256))):
        t, s, a = (bf16_round(torch.randn(shape, generator=g)) for _ in range(3))
        sr, ar = s.clone().requires_grad_(True), a.clone().requires_grad_(True)
        ref = F.mse_loss(t - sr, ar)
        ref.backward()
        loss, (dt, ds, da) = ops.loss_kd(t.to(dtype).cuda(), s.to(dtype).cuda(), a.to(dtype).cuda())
        assert abs(loss.item() - ref.item()) < F32_TOL * abs(ref.item())
        tol = F32_TOL if dtype == torch.float32 else BF16_TOL
        assert rel_err(ds.float(), sr.grad) < tol and rel_err(da.float(), ar.grad) < tol
        # student term: MSE(s_emb, t_emb) == mean(((t) - 0) - s)^2 with s := NULL slot
        loss2, _ = ops.loss_kd(t.to(dtype).cuda(), None, s.to(dtype).cuda(), want=(False, False, True))
        assert abs(loss2.item() - F.mse_loss(s, t).item()) < F32_TOL * F.mse_loss(s, t).item()


def test_rmsprop_matches_torch(cuda):
    """torch.optim.RMSprop(lr, alpha=.99, eps=1e-8, weight_decay=1e-5) as at FSR_main.py:185."""
    ops = _ops()
    g = torch.Generator().manual_seed(17)
    p0 = torch.randn(10007, generator=g)
    p_ref = p0.clone().requires_grad_(True)
    opt = torch.optim.RMSprop([p_ref], lr=1e-3, alpha=0.99, weight_decay=1e-5)
    p = p0.clone().cuda()
    p = torch.cat([p, torch.zeros(1, device="cuda")])[:10007]      # keep 16B alignment explicit
    sq = torch.zeros_like(p)
    for _ in range(3):
        gr = torch.randn(10007, generator=g)
        p_ref.grad = gr.clone()
        opt.step()
        ops.rmsprop_step(p, (gr * 2).cuda(), sq, 1e-3, 0.99, 1e-8, 1e-5, gscale=0.5)
    assert rel_err(p, p_ref) < 1e-6


def test_bicubic_bit_exact(cuda, golden_dir):
    import os
    ops = _ops()
    gd = np.load(os.path.join(golden_dir, "bicubic.npz"))
    from oracle import bicubic_oracle as BO
    for key in gd.files:
        if not key.startswith("src_"):
            continue
        _, s, o = key.split("_")
        src, dst = gd[key], gd["dst_%s_%s" % (s, o)]
        got, f32 = ops.bicubic_u8(torch.from_numpy(src).cuda(), int(o), int(o), want_f32=True)
        assert np.array_equal(got.cpu().numpy(), dst), key
        assert np.array_equal(f32.cpu().numpy(), BO.normalise_to_input(dst)), key
    # BASELINE size: a batch of 128 faces 16 -> 128, checked against the numpy oracle
    rng = np.random.default_rng(1)
    src = rng.integers(0, 256, (128, 16, 16, 3), dtype=np.uint8)
    got, _ = ops.bicubic_u8(torch.from_numpy(src).cuda(), 128, 128)
    assert np.array_equal(got.cpu().numpy(), BO.bicubic_u8(src, 128, 128))


def test_landmark_heatmap(cuda, golden_dir):
    """Device-side landmark heat-map target (helen_loader.py:118-143) against the reference's own generate_hm."""
    ops = _ops()
    g = np.load(os.path.join(golden_dir, "heatmap.npz"))
    hm = ops.landmark_heatmap(torch.from_numpy(g["landmarks"]).cuda(), 32, 32, 1.3).cpu().numpy()
    np.testing.assert_allclose(hm, g["hm"], rtol=1e-6, atol=1e-7)    # fp64 exp: last-ulp libm differences only
    from oracle import bicubic_oracle as BO
    lm = torch.rand(5, 97, 2) * 32
    got = ops.landmark_heatmap(lm.cuda(), 32, 32).cpu().numpy()
    want = np.stack([BO.landmark_heatmap(l.numpy(), 32, 32) for l in lm])
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-7)


def test_eval_dropins(cuda, golden_dir):
    import os
    from crfr_b200.utils import accuracy, calculate_accuracy, calculate_roc
    from oracle import eval_oracle as EO
    gd = np.load(os.path.join(golden_dir, "eval.npz"))
    sc, tg = torch.from_numpy(gd["scores"]).cuda(), torch.from_numpy(gd["target"]).cuda()
    r = accuracy(sc, tg, topk=(1, 5))
    assert abs(r[0].item() - gd["top1"]) < 1e-5 and abs(r[1].item() - gd["top15"][1]) < 1e-5
    ops = _ops()
    _, idx = ops.topk_rows(sc, 5)
    assert np.array_equal(idx.cpu().numpy(), gd["top5_idx"])
    # ties -> lowest index, k > number of distinct maxima
    t = torch.tensor([[1.0, 3.0, 3.0, 3.0, 0.0], [5.0, 5.0, 5.0, 5.0, 5.0]], device="cuda")
    assert ops.topk_rows(t, 3)[1].tolist() == [[1, 2, 3], [0, 1, 2]]
    dist = EO.pair_sqdist(gd["e1"], gd["e2"])
    for thr, ref in zip(gd["thr"], gd["calc_acc"]):
        assert np.allclose(calculate_accuracy(thr, dist, gd["same"]), ref)
    d_gpu, same = ops.pair_verify(torch.from_numpy(gd["e1"]).cuda(), torch.from_numpy(gd["e2"]).cuda(), 30.0)
    assert rel_err(d_gpu, torch.from_numpy(dist)) < 1e-5
    assert np.array_equal(same.cpu().numpy(), dist < 30.0)          # margins >> fp32 summation-order noise
    tpr, fpr, acc, best = calculate_roc(gd["thr"], gd["e1"], gd["e2"], gd["same"], nrof_folds=10, seed=0)
    o = EO.calculate_roc(gd["thr"], gd["e1"], gd["e2"], gd["same"], nrof_folds=10, seed=0)
    assert np.allclose(tpr, o[0]) and np.allclose(fpr, o[1]) and abs(acc - o[2]) < 1e-12 and np.array_equal(best, o[3])


def test_verify_sweep_4000_thresholds(cuda):
    """The threshold sweep of the verification protocol (utils/utils.py:70-82; distill_main.test sweeps 4000 thresholds)
    as one launch per fold: bit-exact counts against numpy, with and without a K-fold subset."""
    ops = _ops()
    rng = np.random.RandomState(3)
    n = 6000
    dist = (rng.rand(n) * 4).astype(np.float32)
    same = rng.rand(n) < 0.5
    thr = np.arange(0, 4, 0.001).astype(np.float32)
    sub = np.sort(rng.permutation(n)[:5400]).astype(np.int32)
    d, s, t = torch.from_numpy(dist).cuda(), torch.from_numpy(same).cuda(), torch.from_numpy(thr).cuda()
    for subset in (None, sub):
        got = ops.verify_sweep(d, s, t, None if subset is None else torch.from_numpy(subset).cuda()).cpu().numpy()
        dd, ss = (dist, same) if subset is None else (dist[subset], same[subset])
        pred = dd[None, :] < thr[:, None]
        want = np.stack([(pred & ss).sum(1), (pred & ~ss).sum(1), (~pred & ~ss).sum(1), (~pred & ss).sum(1)], 1)
        assert np.array_equal(got, want)
