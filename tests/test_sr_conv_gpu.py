"""Tensor-core paths for the convolution shapes of the SUPER_RESOLUTION FSRNet variant (SUPER_RESOLUTION/model/FSRnet.py:
251-416 of the reference): 3x3 stride-1 and stride-2 convolutions with padding 0 on reflection-padded maps, 3x3 stride-2
transposed convolutions, 1x1 convolutions, and the padding-0 stems and image heads.

Every shape class runs forward (with and without bias), dgrad and wgrad (with the bias gradient) on ENGINE_TCGEN05 at the
variant's shapes and at one ragged shape, against fp64 PyTorch on bf16-representable inputs (norm-wise 5e-3) and
against ENGINE_DIRECT, the CUDA-core kernels.  Then the support table, deterministic weight gradients, under-sized
workspaces, and the four sub-networks against the fp32 and bf16 oracles."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from tests.util import bf16_round, rel_err

pytestmark = pytest.mark.gpu

TOL = 5e-3
EUNSUPPORTED, EWORKSPACE = 4, 3

# (name, cin, cout, k, stride, pad, transposed, input size, batch); transposed layers: ConvTranspose2d(3, 2, 1, 1)
SR_SHAPES = [
    ("valid3_64_130", 64, 64, 3, 1, 0, False, 130, 2),
    ("valid3_128_130", 128, 128, 3, 1, 0, False, 130, 2),
    ("valid3_128_66", 128, 128, 3, 1, 0, False, 66, 2),
    ("valid3_256_66", 256, 256, 3, 1, 0, False, 66, 2),
    ("valid3_256_34", 256, 256, 3, 1, 0, False, 34, 2),
    ("valid3_512_34", 512, 512, 3, 1, 0, False, 34, 2),
    ("s2p0_64_130", 64, 128, 3, 2, 0, False, 130, 2),
    ("s2p0_128_130", 128, 256, 3, 2, 0, False, 130, 2),
    ("s2p0_128_66", 128, 256, 3, 2, 0, False, 66, 2),
    ("s2p0_256_66", 256, 512, 3, 2, 0, False, 66, 2),
    ("deconv_512_32", 512, 256, 3, 2, 1, True, 32, 2),
    ("deconv_256_32", 256, 128, 3, 2, 1, True, 32, 2),
    ("deconv_256_64", 256, 128, 3, 2, 1, True, 64, 2),
    ("deconv_128_64", 128, 64, 3, 2, 1, True, 64, 2),
    ("pw_128", 64, 64, 1, 1, 0, False, 128, 2),
    ("pw_64", 64, 64, 1, 1, 0, False, 64, 2),
    ("pw_32", 64, 64, 1, 1, 0, False, 32, 2),
    ("pw_16", 64, 64, 1, 1, 0, False, 16, 2),
    ("pw_8", 64, 64, 1, 1, 0, False, 8, 2),
    ("stem7_134", 3, 64, 7, 1, 0, False, 134, 2),
    ("stem3_130", 3, 64, 3, 1, 0, False, 130, 2),
    ("head_64_130", 64, 3, 3, 1, 0, False, 130, 2),
    ("head_128_130", 128, 3, 3, 1, 0, False, 130, 2),
]
# one ragged case per class: batch 1 or 3, a spatial size that does not divide the tile
RAGGED = [
    ("valid3_ragged", 128, 128, 3, 1, 0, False, 37, 3),
    ("s2p0_ragged", 64, 128, 3, 2, 0, False, 45, 1),
    ("deconv_ragged", 128, 64, 3, 2, 1, True, 13, 3),
    ("pw_ragged", 128, 64, 1, 1, 0, False, 11, 3),
    ("stem7_ragged", 3, 64, 7, 1, 0, False, 41, 1),
    ("stem3_ragged", 3, 64, 3, 1, 0, False, 23, 3),
    ("head_ragged", 128, 3, 3, 1, 0, False, 23, 3),
]
ALL = SR_SHAPES + RAGGED


def _no_tf32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def _stem_dgrad_direct(cin, k):
    """The 3x3 stem's dgrad (3 input channels) stays on the direct kernel: recipe 1 has no dgrad."""
    return cin == 3 and k == 3


class Layer:
    """One convolution on the native ops with seeded bf16-representable operands and its fp64 reference."""

    def __init__(self, cin, cout, k, stride, pad, transposed, size, batch, seed=0):
        from crfr_b200 import ops
        g = torch.Generator().manual_seed(seed)
        self.cfg = (cin, cout, k, stride, pad, transposed)
        self.size, self.batch = size, batch
        x = bf16_round(torch.randn(batch, cin, size, size, generator=g))
        wshape = (cin, cout, k, k) if transposed else (cout, cin, k, k)
        w = bf16_round(torch.randn(wshape, generator=g) / (cin * k * k) ** 0.5)
        self.bias = (0.5 * torch.randn(cout, generator=g)).cuda()
        if transposed:
            o = (size - 1) * stride - 2 * pad + k + 1
        else:
            o = (size + 2 * pad - k) // stride + 1
        self.o = o
        dy = bf16_round(torch.randn(batch, cout, o, o, generator=g))
        self.x, self.w, self.dy = x.cuda(), w.cuda(), dy.cuda()
        self.in_ld = 4 if cin < 8 else cin
        self.out_ld = 4 if cout < 8 else cout
        self.x4 = ops.nchw_to_nhwc(self.x, ld=self.in_ld)
        self.dy4 = ops.nchw_to_nhwc(self.dy, ld=self.out_ld)

    def ref(self):
        _no_tf32()
        cin, cout, k, stride, pad, transposed = self.cfg
        x = self.x.double().requires_grad_(True)
        w = self.w.double().requires_grad_(True)
        b = self.bias.double().requires_grad_(True)
        if transposed:
            y = F.conv_transpose2d(x, w, b, stride, pad, 1)
        else:
            y = F.conv2d(x, w, b, stride, pad)
        y.backward(self.dy.double())
        return y.detach(), x.grad, w.grad, b.grad

    def fwd(self, engine, bias=True):
        from crfr_b200 import ops
        cin, cout, k, stride, pad, transposed = self.cfg
        wp = ops.pack_conv_weight(self.w, transposed=transposed, s_pad=self.in_ld if cin < 8 else None)
        y, _, _ = ops.conv_fwd(self.x4, wp, cin, cout, k, stride, pad, bias=self.bias if bias else None, engine=engine,
                               transposed=transposed, out_hw=(self.o, self.o), out_ld=self.out_ld)
        return y[..., :cout].float().permute(0, 3, 1, 2)

    def dgrad(self, engine):
        from crfr_b200 import ops
        cin, cout, k, stride, pad, transposed = self.cfg
        wt = ops.pack_conv_weight(self.w, for_dgrad=True, transposed=transposed)
        dx = ops.conv_dgrad(self.dy4, wt, tuple(self.x4.shape), cin, cout, k, stride, pad, engine=engine,
                            transposed=transposed)
        return dx[..., :cin].float().permute(0, 3, 1, 2)

    def wgrad(self, engine):
        from crfr_b200 import ops
        cin, cout, k, stride, pad, transposed = self.cfg
        return ops.conv_wgrad(self.x4, self.dy4, cin, cout, k, stride, pad, engine=engine, transposed=transposed,
                              want_bias=True)

    def desc(self):
        from crfr_b200 import _lib as L
        cin, cout, k, stride, pad, transposed = self.cfg
        return L.ConvDesc(self.batch, self.size, self.size, cin, cout, k, stride, pad, self.o, self.o, self.in_ld,
                          self.out_ld, int(transposed))


@pytest.mark.parametrize("name,cin,cout,k,stride,pad,transposed,size,batch", ALL, ids=[c[0] for c in ALL])
def test_sr_conv_tcgen05_against_fp64_and_direct(cuda, name, cin, cout, k, stride, pad, transposed, size, batch):
    from crfr_b200 import _lib as L
    lay = Layer(cin, cout, k, stride, pad, transposed, size, batch, seed=sum(map(ord, name)))
    y_ref, dx_ref, dw_ref, db_ref = lay.ref()
    tc = L.ENGINE_TCGEN05
    y = lay.fwd(tc)
    y_nb = lay.fwd(tc, bias=False)
    dx = lay.dgrad(L.ENGINE_AUTO if _stem_dgrad_direct(cin, k) else tc)
    dw, db = lay.wgrad(tc)
    y_d, dx_d, (dw_d, db_d) = lay.fwd(L.ENGINE_DIRECT), lay.dgrad(L.ENGINE_DIRECT), lay.wgrad(L.ENGINE_DIRECT)
    torch.cuda.synchronize()
    y_ref_nb = y_ref - lay.bias.double().view(1, -1, 1, 1)
    errs = {"fwd": rel_err(y, y_ref), "fwd_nobias": rel_err(y_nb, y_ref_nb), "dgrad": rel_err(dx, dx_ref),
            "wgrad": rel_err(dw, dw_ref), "dbias": rel_err(db, db_ref)}
    direct = {"fwd": rel_err(y, y_d), "dgrad": rel_err(dx, dx_d), "wgrad": rel_err(dw, dw_d), "dbias": rel_err(db, db_d)}
    print("%s: vs fp64 %s | vs ENGINE_DIRECT %s" % (name, {k2: "%.2e" % v for k2, v in errs.items()},
                                                     {k2: "%.2e" % v for k2, v in direct.items()}))
    for key, e in errs.items():
        assert e < TOL, (name, key, e)
    for key, e in direct.items():
        assert e < 2 * TOL, (name, key, e)


def test_sr_conv_engine_support_table(cuda):
    from crfr_b200 import _lib as L
    sup = lambda op, h, cin, cout, k, s, p: bool(L.lib().crfr_conv_engine_supported(L.ENGINE_TCGEN05, op, h, h, cin, cout, k, s, p))
    for name, cin, cout, k, stride, pad, transposed, size, _ in ALL:
        if transposed:          # the query has no transposed flag: the transposed layers are checked by running them
            continue
        for op in (0, 1, 2):
            want = not (op == 1 and _stem_dgrad_direct(cin, k))
            assert sup(op, size, cin, cout, k, stride, pad) == want, (name, op)
    for cout in (11, 13, 68):   # 1x1 layers stop at output channels that are a multiple of 64
        for op in (0, 1, 2):
            assert not sup(op, 32, 64, cout, 1, 1, 0) and not sup(op, 32, 128, cout, 1, 1, 0)


def test_sr_conv_transposed_runs_on_tcgen05_only_for_its_shape(cuda):
    """ConvTranspose2d(3, 2, 1, 1) is accepted by ENGINE_TCGEN05; a 3x3 stride-2 transposed layer without output padding
    is not."""
    from crfr_b200 import _lib as L
    lay = Layer(128, 64, 3, 2, 1, True, 8, 1)
    d = lay.desc()
    d.oh = d.ow = 15
    wsb = L.lib().crfr_conv_workspace_bytes(C.byref(d))
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    y = torch.empty((1, 15, 15, 64), dtype=torch.bfloat16, device="cuda")
    from crfr_b200 import ops
    wp = ops.pack_conv_weight(lay.w, transposed=True)
    rc = L.lib().crfr_conv_fwd(L.ENGINE_TCGEN05, C.byref(d), ops.ptr(lay.x4), ops.ptr(wp), 128, None, ops.ptr(y), None,
                               None, 1e-5, ops.ptr(ws), wsb, ops.stream())
    assert rc == EUNSUPPORTED


@pytest.mark.parametrize("name,cin,cout,k,stride,pad,transposed,size,batch", RAGGED + [SR_SHAPES[5], SR_SHAPES[9], SR_SHAPES[10]],
                         ids=[c[0] for c in RAGGED + [SR_SHAPES[5], SR_SHAPES[9], SR_SHAPES[10]]])
def test_sr_conv_wgrad_is_deterministic(cuda, name, cin, cout, k, stride, pad, transposed, size, batch):
    from crfr_b200 import _lib as L
    lay = Layer(cin, cout, k, stride, pad, transposed, size, batch, seed=3)
    dw1, db1 = lay.wgrad(L.ENGINE_TCGEN05)
    dw2, db2 = lay.wgrad(L.ENGINE_TCGEN05)
    assert torch.equal(dw1, dw2) and torch.equal(db1, db2), name


@pytest.mark.parametrize("name,cin,cout,k,stride,pad,transposed,size,batch", RAGGED, ids=[c[0] for c in RAGGED])
def test_sr_conv_undersized_workspace(cuda, name, cin, cout, k, stride, pad, transposed, size, batch):
    """A workspace too small for the layer returns CRFR_EWORKSPACE and writes nothing past it (nor into the outputs).
    The forward of the tile-engine and 1x1 layers needs no workspace: only the calls that use one are checked."""
    from crfr_b200 import _lib as L
    from crfr_b200 import ops
    lay = Layer(cin, cout, k, stride, pad, transposed, size, batch, seed=4)
    d = lay.desc()
    small = 256
    buf = torch.full((1 << 20,), 0x5A, dtype=torch.uint8, device="cuda")
    lib, st = L.lib(), ops.stream()
    calls = []
    dw = torch.zeros((cin, cout, k, k) if transposed else (cout, cin, k, k), dtype=torch.float32, device="cuda")
    calls.append(("wgrad", lambda: lib.crfr_conv_wgrad(L.ENGINE_TCGEN05, C.byref(d), ops.ptr(lay.x4), ops.ptr(lay.dy4),
                                                       ops.ptr(dw), None, ops.ptr(buf), small, st), dw))
    if stride == 2 or cin == 3 or cout == 3:        # the lowered forms stage an im2col / product matrix
        y = torch.zeros((batch, lay.o, lay.o, lay.out_ld), dtype=torch.bfloat16, device="cuda")
        wp = ops.pack_conv_weight(lay.w, transposed=transposed, s_pad=lay.in_ld if cin < 8 else None)
        calls.append(("fwd", lambda: lib.crfr_conv_fwd(L.ENGINE_TCGEN05, C.byref(d), ops.ptr(lay.x4), ops.ptr(wp), wp.shape[2],
                                                       None, ops.ptr(y), None, None, 1e-5, ops.ptr(buf), small, st), y))
    if stride == 2 or k == 7 or cout == 3:
        dx = torch.zeros_like(lay.x4)
        wt = ops.pack_conv_weight(lay.w, for_dgrad=True, transposed=transposed)
        calls.append(("dgrad", lambda: lib.crfr_conv_dgrad(L.ENGINE_TCGEN05, C.byref(d), ops.ptr(lay.dy4), ops.ptr(wt),
                                                           wt.shape[2], ops.ptr(dx), ops.ptr(buf), small, st), dx))
    for op, fn, out in calls:
        assert fn() == EWORKSPACE, (name, op)
        torch.cuda.synchronize()
        assert bool((buf[small:] == 0x5A).all()), (name, op, "wrote past the workspace")
        assert not bool(out.float().abs().sum() > 0), (name, op, "wrote the output")


# ------------------------------------------------------------------------------------------------ module level
SLACK = 1.6
MODULES = [("coarse", "Coarse_SR_Network", 700, 64), ("encoder", "Fine_SR_Encoder", 701, 64),
           ("prior", "Prior_Estimation_Network", 702, 64), ("decoder", "Fine_SR_Decoder", 703, 64),
           ("decoder", "Fine_SR_Decoder", 703, 128)]


def _build(cls_name, seed):
    from crfr_b200.SUPER_RESOLUTION.model import FSRnet as M
    torch.manual_seed(seed)
    net = getattr(M, cls_name)()
    with torch.no_grad():
        for _, p in net.named_parameters():
            if p.dim() == 1:
                p.add_(0.2 * torch.randn_like(p))
    return net


@pytest.mark.parametrize("name,cls_name,seed,size", MODULES, ids=["%s_%d" % (m[0], m[3]) for m in MODULES])
def test_sr_subnetwork_gradients_against_oracle(cuda, name, cls_name, seed, size):
    """Outputs, input gradient and every parameter gradient within 1.6 x the bf16 oracle's own deviation from fp32 + 2e-2
    (the bound of tests/test_sr_variant_gpu.py), batch 2.  The oracle runs on the GPU in fp32 without TF32."""
    from oracle import fsrnet_oracle as FO
    from oracle import sr_oracle as SO
    _no_tf32()
    net = _build(cls_name, seed)
    sd = {k: v.detach().clone().cuda() for k, v in net.state_dict().items()}
    net = net.cuda().train()
    g = torch.Generator().manual_seed(9)
    cin = 128 if name == "decoder" else 3
    x = bf16_round(torch.randn(2, cin, size, size, generator=g)).cuda()
    fwd = {"coarse": SO.coarse_forward, "encoder": SO.encoder_forward, "prior": SO.prior_forward,
           "decoder": SO.decoder_forward}[name]
    xg = x.clone().requires_grad_(True)
    outs = net(xg)
    outs = outs if isinstance(outs, tuple) else (outs,)
    dys = [torch.randn(o.shape, generator=g).cuda() for o in outs]
    torch.autograd.backward(outs, dys)
    res = {}
    for tag, pr in (("ref", FO.FP32), ("emu", FO.Precision("bf16"))):
        leaves = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        xr = x.clone().requires_grad_(True)
        o = fwd(leaves, xr, "", pr)
        o = o if isinstance(o, tuple) else (o,)
        torch.autograd.backward(o, dys)
        res[tag] = ([t.detach() for t in o], xr.grad, {k: v.grad for k, v in leaves.items()})
    ref, emu = res["ref"], res["emu"]
    for i, o in enumerate(outs):
        bound = SLACK * rel_err(emu[0][i], ref[0][i]) + 2e-2
        assert rel_err(o, ref[0][i]) < bound, (name, "output", i, rel_err(o, ref[0][i]), bound)
    bound = SLACK * rel_err(emu[1], ref[1]) + 2e-2
    assert rel_err(xg.grad, ref[1]) < bound, (name, "dx", rel_err(xg.grad, ref[1]), bound)
    worst = (0.0, None)
    for k, p in net.named_parameters():
        r, e = ref[2][k], emu[2][k]
        assert p.grad is not None, k
        err, bound = rel_err(p.grad, r), SLACK * rel_err(e, r) + 2e-2
        assert err < bound, (name, k, err, rel_err(e, r))
        worst = max(worst, (err, k))
    print("%s %d: worst parameter gradient %.2e (%s)" % (name, size, worst[0], worst[1]))
