"""crfr_conv_dgrad_norm_bwd: the backward across `conv(PReLU(InstanceNorm(y) (+ res)))` as one operation - the first pass of
the normalisation backward runs inside the epilogue of the row-streaming dgrad kernel (rowconv2.cu, FUSE = 1).

ref: model/FSRnet.py:91-97 (_Residual_Block.forward: in1 -> relu -> conv2, and in2 -> add -> relu_out -> next conv1)."""
import pytest
import torch
import torch.nn.functional as F

from tests.util import bf16_round, nhwc_from, rel_err, to_nchw

pytestmark = pytest.mark.gpu


def _case(n, h, res, second, seed):
    g = torch.Generator().manual_seed(seed)
    c, w_ = 64, 128
    y = bf16_round(torch.randn(n, c, h, w_, generator=g) * 1.3 + 0.2)
    r = bf16_round(torch.randn(n, c, h, w_, generator=g)) if res else None
    dxb = bf16_round(torch.randn(n, c, h, w_, generator=g) * 0.5) if second else None
    wgt = bf16_round(torch.randn(c, c, 3, 3, generator=g) * 0.05)
    dout = bf16_round(torch.randn(n, c, h, w_, generator=g))
    gamma, beta = torch.rand(c, generator=g) + 0.5, torch.randn(c, generator=g) * 0.3
    alpha = torch.rand(c, generator=g) * 0.5 - 0.05
    return y, r, dxb, wgt, dout, gamma, beta, alpha


@pytest.mark.parametrize("n,h,res,second", [(2, 1, False, False), (2, 2, True, True), (6, 3, True, False),
                                            (40, 16, False, True), (8, 50, True, True), (2, 128, False, False),
                                            (34, 128, True, True), (300, 1, True, True)])
def test_fused_dgrad_norm_bwd(cuda, n, h, res, second):
    """Fused against unfused (option fuse_norm_bwd): dz is the same arithmetic per element -> identical bits; dy and the
    parameter gradients differ only through the association of the fp32 sums.  Both against fp32 autograd of the chain
    conv(prelu(instance_norm(y) + res)) with the extra gradient dx_b added at the convolution's input."""
    from crfr_b200 import _lib as L, ops
    y, r, dxb, wgt, dout, gamma, beta, alpha = _case(n, h, res, second, 900 + n + h)
    c = 64
    yg = nhwc_from(y)
    stats = ops.norm_stats(yg)
    wt = ops.pack_conv_weight(wgt.cuda(), for_dgrad=True)
    rg = nhwc_from(r) if res else None
    bg = nhwc_from(dxb) if second else None
    out = {}
    try:
        for mode in (0, 1):
            ops.set_option("fuse_norm_bwd", mode)
            out[mode] = ops.conv_dgrad_norm_bwd(nhwc_from(dout), wt, yg, stats, c, c, 3, 1, 1, gamma.cuda(), beta.cuda(),
                                                alpha.cuda(), res=rg, dx_b=bg, engine=L.ENGINE_TCGEN05)
            torch.cuda.synchronize()
    finally:
        ops.set_option("fuse_norm_bwd", 1)
    dz0, dy0, dg0, db0, da0 = out[0]
    dz1, dy1, dg1, db1, da1 = out[1]
    assert torch.equal(dz0, dz1), "dz differs: %.3e" % rel_err(dz1.float(), dz0.float())
    assert rel_err(dy1.float(), dy0.float()) < 2e-3
    for a, b in ((dg1, dg0), (db1, db0), (da1, da0)):
        assert rel_err(a, b) < 1e-4
    # fp32 autograd of the same chain
    yr, gr, br, ar = (t.clone().requires_grad_(True) for t in (y, gamma, beta, alpha))
    rr = r.clone().requires_grad_(True) if res else None
    z = F.instance_norm(yr, weight=gr, bias=br, eps=1e-5)
    if res:
        z = z + rr
    x = F.prelu(z, ar)
    x.retain_grad()
    o = F.conv2d(x, wgt, None, 1, 1)
    o.backward(dout, retain_graph=True)
    if second:
        x.backward(dxb)
    assert rel_err(to_nchw(dy1), yr.grad) < 1e-2          # three bf16 roundings (dgrad output, dz, dy)
    if res:
        assert rel_err(to_nchw(dz1), rr.grad) < 1e-2
    assert rel_err(dg1, gr.grad) < 1e-2 and rel_err(db1, br.grad) < 1e-2 and rel_err(da1, ar.grad) < 1e-2


def test_fused_dgrad_norm_bwd_deterministic(cuda):
    from crfr_b200 import _lib as L, ops
    n, h = 10, 37
    y, r, dxb, wgt, dout, gamma, beta, alpha = _case(n, h, True, True, 7)
    yg = nhwc_from(y)
    stats = ops.norm_stats(yg)
    wt = ops.pack_conv_weight(wgt.cuda(), for_dgrad=True)
    a = ops.conv_dgrad_norm_bwd(nhwc_from(dout), wt, yg, stats, 64, 64, 3, 1, 1, gamma.cuda(), beta.cuda(), alpha.cuda(),
                                res=nhwc_from(r), dx_b=nhwc_from(dxb), engine=L.ENGINE_TCGEN05)
    b = ops.conv_dgrad_norm_bwd(nhwc_from(dout), wt, yg, stats, 64, 64, 3, 1, 1, gamma.cuda(), beta.cuda(), alpha.cuda(),
                                res=nhwc_from(r), dx_b=nhwc_from(dxb), engine=L.ENGINE_TCGEN05)
    torch.cuda.synchronize()
    for u, v in zip(a, b):
        assert torch.equal(u, v)


def test_fused_dgrad_norm_bwd_other_shapes_fall_back(cuda):
    """Shapes the row-streaming kernel does not take (here 128 channels at 32 x 32, odd image count) run dgrad + the
    normalisation backward as two calls with the same contract."""
    from crfr_b200 import _lib as L, ops
    g = torch.Generator().manual_seed(3)
    n, c, h = 3, 128, 32
    y = bf16_round(torch.randn(n, c, h, h, generator=g))
    wgt = bf16_round(torch.randn(c, c, 3, 3, generator=g) * 0.05)
    dout = bf16_round(torch.randn(n, c, h, h, generator=g))
    alpha = torch.full((c,), 0.25)
    yg = nhwc_from(y)
    stats = ops.norm_stats(yg)
    dz, dy, _, _, da = ops.conv_dgrad_norm_bwd(nhwc_from(dout), ops.pack_conv_weight(wgt.cuda(), for_dgrad=True), yg, stats,
                                               c, c, 3, 1, 1, alpha=alpha.cuda(), engine=L.ENGINE_TCGEN05)
    yr, ar = y.clone().requires_grad_(True), alpha.clone().requires_grad_(True)
    o = F.conv2d(F.prelu(F.instance_norm(yr, eps=1e-5), ar), wgt, None, 1, 1)
    o.backward(dout)
    assert rel_err(to_nchw(dy), yr.grad) < 2e-2 and rel_err(da, ar.grad) < 1e-2

