"""The SUPER_RESOLUTION FSRNet variant's network program (crfr_srnet_*, csrc/srnet.cu) behind the modules of
crfr_b200/SUPER_RESOLUTION/model/FSRnet.py: against the fp32 / bf16 oracle (oracle/sr_oracle.py), against the op-by-op
composition it replaces (oracle/sr_composed.py), one op deep on its own stored tensors (crfr_srnet_tape), and its
invariants (bit-identical repeats and graph replay, the tape inside the workspace, workspace and shape rejections)."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from tests.util import bf16_round, rel_err

pytestmark = pytest.mark.gpu

SLACK = 1.6                      # the module bound of tests/test_sr_variant_gpu.py: SLACK x the bf16 oracle's deviation + 2e-2
EINVAL, EWORKSPACE = 1, 3
K_CONV, K_NORM, K_POOL, K_UPADD, K_CAT, K_HEADS, K_PAD, K_ADD, K_TANH = 0, 1, 2, 3, 4, 5, 20, 21, 22


def _no_tf32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def _net(seed=5):
    from crfr_b200.SUPER_RESOLUTION.model.FSRnet import SRNetwork
    torch.manual_seed(seed)
    net = SRNetwork()
    with torch.no_grad():                       # non-trivial affine / bias parameters, as tests/test_sr_variant_gpu.py
        for _, p in net.named_parameters():
            if p.dim() == 1:
                p.add_(0.2 * torch.randn_like(p))
    return net.cuda().train()


def _grads(net):
    return {k: (None if p.grad is None else p.grad.detach().clone()) for k, p in net.named_parameters()}


def _run(net, x, dys, fwd=None):
    net.zero_grad(set_to_none=True)
    xg = x.clone().requires_grad_(True)
    outs = (fwd or net)(xg)
    torch.autograd.backward(outs, dys)
    return [o.detach() for o in outs], xg.grad.detach(), _grads(net)


@pytest.mark.parametrize("size", [32, 64])
def test_srnet_against_oracle(cuda, size):
    """All four outputs, the input gradient and all 1108 parameter gradients within 1.6 x the bf16 oracle's deviation from
    fp32 + 2e-2, batch 2."""
    from oracle import fsrnet_oracle as FO
    from oracle import sr_oracle as SO
    _no_tf32()
    net = _net()
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    g = torch.Generator().manual_seed(3)
    x = bf16_round(torch.randn(2, 3, size, size, generator=g)).cuda()
    shapes = [(2, 3, size, size), (2, 3, size, size), (2, 68, size, size), (2, 13, size, size)]
    dys = [torch.randn(s, generator=g).cuda() for s in shapes]
    outs, dx, grads = _run(net, x, dys)
    assert len(grads) == 1108
    res = {}
    for tag, pr in (("ref", FO.FP32), ("emu", FO.Precision("bf16"))):
        leaves = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        xr = x.clone().requires_grad_(True)
        o = SO.sr_forward(leaves, xr, pr)
        torch.autograd.backward(o, dys)
        res[tag] = ([t.detach() for t in o], xr.grad, {k: v.grad for k, v in leaves.items()})
    ref, emu = res["ref"], res["emu"]
    for i, o in enumerate(outs):
        bound = SLACK * rel_err(emu[0][i], ref[0][i]) + 2e-2
        assert rel_err(o, ref[0][i]) < bound, ("output", i, rel_err(o, ref[0][i]), bound)
    assert rel_err(dx, ref[1]) < SLACK * rel_err(emu[1], ref[1]) + 2e-2, ("dx", rel_err(dx, ref[1]))
    worst = (0.0, None)
    for k, gk in grads.items():
        r, e = ref[2][k], emu[2][k]
        assert gk is not None, k
        err, bound = rel_err(gk, r), SLACK * rel_err(e, r) + 2e-2
        assert err < bound, (k, err, rel_err(e, r))
        worst = max(worst, (err, k))
    print("SRNetwork %d x %d: worst parameter gradient %.3e (%s)" % (size, size, worst[0], worst[1]))


def test_srnet_against_oracle_at_128(cuda):
    """Batch 32 at 128 x 128 (the timed size): the program against the fp32 / bf16 oracle with the module bound, all four
    outputs, the input gradient and all 1108 parameter gradients.  The composition the modules ran before
    (oracle/sr_composed.py) is evaluated on the same weights, inputs and output gradients and its distances printed."""
    from oracle import fsrnet_oracle as FO
    from oracle import sr_composed as SC
    from oracle import sr_oracle as SO
    _no_tf32()
    net = _net()
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    g = torch.Generator(device="cuda").manual_seed(11)
    x = bf16_round(torch.randn(32, 3, 128, 128, device="cuda", generator=g))
    shapes = [(32, 3, 128, 128), (32, 3, 128, 128), (32, 68, 128, 128), (32, 13, 128, 128)]
    dys = [torch.randn(s, device="cuda", generator=g) for s in shapes]
    prog = _run(net, x, dys)
    comp = _run(net, x, dys, fwd=lambda t: SC.network(net, t))
    res = {}
    for tag, pr in (("ref", FO.FP32), ("emu", FO.Precision("bf16"))):
        leaves = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        xr = x.clone().requires_grad_(True)
        o = SO.sr_forward(leaves, xr, pr)
        torch.autograd.backward(o, dys)
        res[tag] = ([t.detach() for t in o], xr.grad.detach(), {k: v.grad.detach() for k, v in leaves.items()})
        del leaves, xr, o
        torch.cuda.empty_cache()
    ref, emu = res["ref"], res["emu"]
    pairs = [("output %d" % i, prog[0][i], comp[0][i], ref[0][i], emu[0][i]) for i in range(4)]
    pairs.append(("dx", prog[1], comp[1], ref[1], emu[1]))
    pairs += [(k, prog[2][k], comp[2][k], ref[2][k], emu[2][k]) for k in prog[2]]
    bad, worst, worst_c = [], (0.0, None), (0.0, None)
    for k, p, c, r, e in pairs:
        err, bound = rel_err(p, r), SLACK * rel_err(e, r) + 2e-2
        if not err < bound:
            bad.append((k, err, bound))
        worst = max(worst, (err / bound, k))
        worst_c = max(worst_c, (rel_err(c, r) / bound, k))
    print("128 x 128 batch 32: worst error / bound %.3f (%s); the composed path's %.3f (%s)" % (*worst, *worst_c))
    assert not bad, bad[:10]


def test_srnet_unreached_heads_get_no_gradient(cuda):
    net = _net()
    x = torch.randn(2, 3, 32, 32, device="cuda")
    coarse, out, lm, ps = net(x)
    (out.square().mean() + coarse.mean()).backward()
    p = net._prior_estimation_network
    assert p.fc.weight.grad is None and p.fc.bias.grad is None and p.fc_landmark.weight.grad is None
    assert p.model[1].weight.grad is not None and net._fine_sr_decoder.out[1].weight.grad is not None
    net.zero_grad(set_to_none=True)
    _, _, lm, _ = net(x)
    lm.sum().backward()
    assert p.fc.weight.grad is None and p.fc_landmark.weight.grad is not None
    assert net._fine_sr_decoder.out[1].weight.grad is None and net._fine_sr_encoder.model[1].weight.grad is None
    assert net._coarse_sr_network.model[1].weight.grad is not None


# ------------------------------------------------------------------------------------------------ the C ABI directly
def _params(net):
    sd = dict(net.named_parameters())
    return [sd[k].detach() for k in net.state_dict().keys()]


def _table(ts):
    return (C.c_void_p * len(ts))(*[None if t is None else t.data_ptr() for t in ts])


def _io(section, x, outs):
    from crfr_b200 import _lib as L
    io = L.SrnetIO()
    io.section, io.batch, io.h, io.w = section, x.shape[0], x.shape[2], x.shape[3]
    io.x = x.data_ptr()
    for i, o in enumerate(outs):
        io.out[i] = o.data_ptr()
    return io


def _outs(b, h, w):
    return [torch.zeros(s, device="cuda") for s in [(b, 3, h, w), (b, 3, h, w), (b, 68, h, w), (b, 13, h, w)]]


def _forward_c(net, x, ws, training=1):
    from crfr_b200 import _lib as L
    from crfr_b200 import ops
    params = _params(net)
    outs = _outs(*x.shape[:1], *x.shape[2:])
    io = _io(L.SRNET_NETWORK, x, outs)
    rc = L.lib().crfr_srnet_forward(L.ENGINE_AUTO, _table(params), C.byref(io), training, ws.data_ptr(), ws.numel(),
                                    ops.stream())
    return rc, outs, params, io


def _tape(section, b, h, w):
    from crfr_b200 import _lib as L
    n = L.lib().crfr_srnet_tape(section, b, h, w, 1, None, 0)
    arr = (L.TapeEntry * n)()
    assert L.lib().crfr_srnet_tape(section, b, h, w, 1, arr, n) == n
    return list(arr)


def test_srnet_repeat_and_graph_replay_are_bit_identical(cuda):
    from crfr_b200 import _lib as L
    from crfr_b200 import ops
    net = _net()
    b, s = 2, 32
    x = torch.randn(b, 3, s, s, device="cuda")
    dys = [torch.randn(t.shape, device="cuda") for t in _outs(b, s, s)]
    ws = torch.empty(L.lib().crfr_srnet_workspace_bytes(L.SRNET_NETWORK, b, s, s, 1), dtype=torch.uint8, device="cuda")
    params = _params(net)
    grads = [torch.zeros_like(p) for p in params]
    dx = torch.zeros_like(x)
    outs = _outs(b, s, s)
    io = _io(L.SRNET_NETWORK, x, outs)
    darr = _table(dys)

    def step():
        for t in grads:
            t.zero_()
        L.call("crfr_srnet_forward", L.ENGINE_AUTO, _table(params), C.byref(io), 1, ws.data_ptr(), ws.numel(),
               ops.stream())
        L.call("crfr_srnet_backward", L.ENGINE_AUTO, _table(params), _table(grads), C.byref(io), darr, dx.data_ptr(),
               ws.data_ptr(), ws.numel(), ops.stream())

    def snap():
        torch.cuda.synchronize()
        return [t.clone() for t in outs + grads + [dx]]

    step()
    first = snap()
    step()
    second = snap()
    assert all(torch.equal(a, b_) for a, b_ in zip(first, second))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()                                   # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    for t in outs + grads + [dx]:
        t.fill_(7.0)
    graph.replay()
    replayed = snap()
    assert all(torch.equal(a, b_) for a, b_ in zip(first, replayed))


def test_srnet_tape_inside_workspace_and_disjoint(cuda):
    from crfr_b200 import _lib as L
    for sec, (b, h, w) in [(L.SRNET_NETWORK, (2, 32, 48)), (L.SRNET_PRIOR, (2, 32, 32)), (L.SRNET_COARSE, (1, 13, 9)),
                           (L.SRNET_ENCODER, (2, 20, 20)), (L.SRNET_DECODER, (1, 16, 24))]:
        size = L.lib().crfr_srnet_workspace_bytes(sec, b, h, w, 1)
        spans = {}
        for e in _tape(sec, b, h, w):
            if e.out_off < 0 or (e.ld > 4 and e.c < e.ld):   # the concat halves are views of the concat buffer
                continue
            lo, hi = e.out_off, e.out_off + (e.n * e.h * e.w * e.ld) * 2
            assert 0 <= lo and hi <= size, (sec, e.kind, lo, hi, size)
            assert lo not in spans, (sec, e.kind, lo)
            spans[lo] = hi
            if e.kind == K_NORM:
                assert 0 <= e.stats_off and e.stats_off + e.n * e.c * 8 <= size
        ivs = sorted(spans.items())
        for (a0, a1), (b0, b1) in zip(ivs, ivs[1:]):
            assert a1 <= b0, (sec, a0, a1, b0, b1)


def test_srnet_undersized_workspace_and_rejections(cuda):
    from crfr_b200 import _lib as L
    from crfr_b200 import ops
    from crfr_b200.SUPER_RESOLUTION.model.FSRnet import Fine_SR_Decoder, Prior_Estimation_Network, SRNetwork
    net = _net()
    b, s = 2, 32
    x = torch.randn(b, 3, s, s, device="cuda")
    need = L.lib().crfr_srnet_workspace_bytes(L.SRNET_NETWORK, b, s, s, 1)
    small = need // 2
    buf = torch.full((small + (1 << 20),), 0x5A, dtype=torch.uint8, device="cuda")
    rc, outs, params, io = _forward_c(net, x, buf[:small])
    torch.cuda.synchronize()
    assert rc == EWORKSPACE
    assert bool((buf == 0x5A).all()), "wrote into or past the undersized workspace"
    assert all(not bool(o.abs().sum() > 0) for o in outs), "wrote the outputs"
    grads = [torch.zeros_like(p) for p in params]
    rc = L.lib().crfr_srnet_backward(L.ENGINE_AUTO, _table(params), _table(grads), C.byref(io), _table(outs[:1]), None,
                                     buf.data_ptr(), small, ops.stream())
    torch.cuda.synchronize()
    assert rc == EWORKSPACE and bool((buf == 0x5A).all()) and all(not bool(g.abs().sum() > 0) for g in grads)
    # shapes the program does not take: EINVAL before any launch, ValueError / RuntimeError from the modules
    ws = torch.full((need,), 0x5A, dtype=torch.uint8, device="cuda")
    for bad in [(2, 3, 40, 32), (2, 3, 8, 8)]:
        xb = torch.randn(bad, device="cuda")
        rc, outs, _, _ = _forward_c(net, xb, ws)
        torch.cuda.synchronize()
        assert rc == EINVAL and bool((ws == 0x5A).all())
        with pytest.raises(ValueError):
            net(xb)
    assert L.lib().crfr_srnet_workspace_bytes(L.SRNET_PRIOR, 2, 24, 32, 1) == 0
    assert L.lib().crfr_srnet_workspace_bytes(L.SRNET_COARSE, 2, 4, 32, 1) == 0
    assert L.lib().crfr_srnet_tape(L.SRNET_NETWORK, 2, 40, 32, 1, None, 0) == -1
    with pytest.raises(ValueError):
        Prior_Estimation_Network().cuda()(torch.randn(1, 3, 24, 24, device="cuda"))
    with pytest.raises(ValueError):
        Fine_SR_Decoder().cuda()(torch.randn(1, 64, 16, 16, device="cuda"))
    with pytest.raises(RuntimeError):
        SRNetwork()(torch.randn(1, 3, 32, 32))


def test_srnet_sections_odd_sizes_against_oracle(cuda):
    """The sub-networks at sizes that are not multiples of 4 (their outputs are 4 * ceil(h / 4) high) and with h != w:
    outputs, input gradient and every parameter gradient against the fp32 / bf16 oracle with the module bound."""
    from oracle import fsrnet_oracle as FO
    from oracle import sr_oracle as SO
    from crfr_b200.SUPER_RESOLUTION.model import FSRnet as M
    _no_tf32()
    fwds = {"Coarse_SR_Network": SO.coarse_forward, "Fine_SR_Encoder": SO.encoder_forward,
            "Prior_Estimation_Network": SO.prior_forward, "Fine_SR_Decoder": SO.decoder_forward}
    g = torch.Generator().manual_seed(4)
    for cls, cin, (h, w) in [("Coarse_SR_Network", 3, (13, 22)), ("Fine_SR_Encoder", 3, (18, 11)),
                             ("Fine_SR_Decoder", 128, (9, 16)), ("Prior_Estimation_Network", 3, (32, 48))]:
        torch.manual_seed(2)
        m = getattr(M, cls)()
        sd = {k: v.detach().clone().cuda() for k, v in m.state_dict().items()}
        m = m.cuda().train()
        x = bf16_round(torch.randn(2, cin, h, w, generator=g)).cuda()
        xg = x.clone().requires_grad_(True)
        outs = m(xg)
        outs = outs if isinstance(outs, tuple) else (outs,)
        dys = [torch.randn(o.shape, generator=g).cuda() for o in outs]
        torch.autograd.backward(outs, dys)
        res = {}
        for tag, pr in (("ref", FO.FP32), ("emu", FO.Precision("bf16"))):
            leaves = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
            xr = x.clone().requires_grad_(True)
            o = fwds[cls](leaves, xr, "", pr)
            o = o if isinstance(o, tuple) else (o,)
            torch.autograd.backward(o, dys)
            res[tag] = ([t.detach() for t in o], xr.grad, {k: v.grad for k, v in leaves.items()})
        ref, emu = res["ref"], res["emu"]
        checks = [("output %d" % i, o, ref[0][i], emu[0][i]) for i, o in enumerate(outs)]
        checks.append(("dx", xg.grad, ref[1], emu[1]))
        checks += [(k, p.grad, ref[2][k], emu[2][k]) for k, p in m.named_parameters()]
        for k, p, r, e in checks:
            assert p is not None and p.shape == r.shape, (cls, k)
            assert rel_err(p, r) < SLACK * rel_err(e, r) + 2e-2, (cls, (h, w), k, rel_err(p, r), rel_err(e, r))


# ------------------------------------------------------------------------------------------------ one op deep
class Stored:
    """The tensors a training forward left in its workspace, read through crfr_srnet_tape, as float64 NCHW."""

    def __init__(self, net, b, h, w):
        from crfr_b200 import _lib as L
        self.L = L
        self.b, self.h, self.w = b, h, w
        g = torch.Generator().manual_seed(21)
        self.x = torch.randn(b, 3, h, w, generator=g).cuda()
        self.ws = torch.empty(L.lib().crfr_srnet_workspace_bytes(L.SRNET_NETWORK, b, h, w, 1), dtype=torch.uint8,
                              device="cuda")
        rc, self.outs, self.params, _ = _forward_c(net, self.x, self.ws)
        assert rc == 0
        torch.cuda.synchronize()
        self.keys = list(net.state_dict().keys())
        self.mods = dict(net.named_modules())
        self.tape = _tape(L.SRNET_NETWORK, b, h, w)

    def dims_of(self, i, off):
        """(n, h, w, c, ld) of the tensor at off as op i reads it: the last earlier op that wrote there."""
        for j in range(i - 1, -1, -1):
            e = self.tape[j]
            if e.out_off == off:
                return e.n, e.h, e.w, e.c, e.ld
        return self.b, self.h, self.w, 3, 4                  # the network input, NHWC4

    def read(self, off, dims):
        n, h, w, c, ld = dims
        t = self.ws[off:off + n * h * w * ld * 2].view(torch.bfloat16).view(n, h, w, ld)[..., :c]
        return t.permute(0, 3, 1, 2).double().cpu()

    def raw(self, off, dims):
        """the stored bf16 NHWC tensor itself (device, dense copy of its channels)"""
        n, h, w, c, ld = dims
        return self.ws[off:off + n * h * w * ld * 2].view(torch.bfloat16).view(n, h, w, ld)[..., :c].contiguous()

    def out(self, i):
        e = self.tape[i]
        return self.read(e.out_off, (e.n, e.h, e.w, e.c, e.ld))

    def inp(self, i, off=None):
        off = self.tape[i].in_off if off is None else off
        return self.read(off, self.dims_of(i, off))

    def param(self, idx):
        return self.params[idx].double().cpu()

    def module_of(self, idx):
        return self.mods[self.keys[idx].rsplit(".", 1)[0]]


def _in(y, w=None, b=None):
    return F.instance_norm(y, None, None, w, b, True, 0.0, 1e-5)


def _check(kind_errs, tol, planted):
    worst = max(kind_errs)
    assert worst < tol, (worst, tol)
    assert planted > tol, ("a planted error passes the bound", planted, tol)
    return worst


def test_srnet_forward_one_op_deep(cuda):
    """Every op kind the program records, on its own stored bf16 input replayed in float64 against its stored output.
    Each class of check rejects a planted error in the float64 reference."""
    st = Stored(_net(), 2, 32, 32)
    T = st.tape
    kinds = {e.kind for e in T}
    assert kinds == {K_CONV, K_NORM, K_POOL, K_UPADD, K_CAT, K_HEADS, K_PAD, K_ADD, K_TANH}, kinds
    errs = {k: [] for k in kinds}
    planted = {}
    fref = {}                                                # float64 references of the ops, by tape index
    conv_cls = set()
    for i, e in enumerate(T):
        if e.kind == K_PAD:
            x = st.inp(i)
            ref = F.pad(x, (e.w_idx,) * 4, mode="reflect")
            errs[K_PAD].append(rel_err(st.out(i), ref))
            if K_PAD not in planted:                         # reflection off by one: replicate the edge instead
                planted[K_PAD] = rel_err(st.out(i), F.pad(x, (e.w_idx,) * 4, mode="replicate"))
        elif e.kind == K_CONV:
            m = st.module_of(e.w_idx)
            x = st.inp(i)
            wgt = st.param(e.w_idx)
            bias_key = st.keys[e.w_idx].rsplit(".", 1)[0] + ".bias"
            bias = st.param(e.w_idx + 1) if e.w_idx + 1 < len(st.keys) and st.keys[e.w_idx + 1] == bias_key else None
            wq = bf16_round(wgt.float()).double()
            if isinstance(m, torch.nn.ConvTranspose2d):
                ref = F.conv_transpose2d(x, wq, bias, m.stride, m.padding, m.output_padding)
                cls = "transposed"
            else:
                ref = F.conv2d(x, wq, bias, m.stride, m.padding)
                cls = "%dx%d s%d p%d cin%s cout%s" % (m.kernel_size[0], m.kernel_size[0], m.stride[0], m.padding[0],
                                                      "3" if m.in_channels == 3 else "", "3" if m.out_channels == 3 else "")
            conv_cls.add(cls)
            errs[K_CONV].append(rel_err(st.out(i), ref))
            if K_CONV not in planted and m.kernel_size[0] == 3 and m.padding[0] == 0:   # the pad-0 conv read one pixel off
                planted[K_CONV] = rel_err(st.out(i), F.conv2d(torch.roll(x, 1, 3), wq, bias, m.stride, 0))
        elif e.kind == K_NORM:
            y = st.inp(i)
            # affine / PReLU: the _Residual_Block norms, found by their position after the block's convolutions
            conv_key = None
            if T[i - 1].kind == K_CONV and T[i - 1].w_idx >= 0:
                conv_key = st.keys[T[i - 1].w_idx]
            z = _in(y)
            if conv_key and conv_key.endswith("conv1.weight") and ".hg." not in conv_key:
                p = conv_key[:-len("conv1.weight")]
                idx = st.keys.index(p + "in1.weight")
                z = _in(y, st.param(idx), st.param(idx + 1))
                ref = F.prelu(z, st.param(idx + 2))
            elif conv_key and conv_key.endswith("conv2.weight") and ".hg." not in conv_key and e.has_res:
                p = conv_key[:-len("conv2.weight")]
                idx = st.keys.index(p + "in2.weight")
                res = st.inp(i - 3)
                ref = _in(y, st.param(idx), st.param(idx + 1)) + res
            else:
                ref = F.relu(z)
            fref[i] = ref
            errs[K_NORM].append(rel_err(st.out(i), ref))
            if K_NORM not in planted and e.has_res:          # the residual dropped
                planted[K_NORM] = rel_err(st.out(i), ref - st.inp(i - 3))
        elif e.kind == K_ADD:
            ref = st.inp(i) + st.inp(i, e.stats_off)
            errs[K_ADD].append(rel_err(st.out(i), ref))
            planted.setdefault(K_ADD, rel_err(st.out(i), st.inp(i)))
        elif e.kind == K_POOL:
            ref = F.max_pool2d(st.inp(i), 2, 2)
            errs[K_POOL].append(rel_err(st.out(i), ref))
            planted.setdefault(K_POOL, rel_err(st.out(i), F.avg_pool2d(st.inp(i), 2, 2)))
        elif e.kind == K_UPADD:
            up, low = st.inp(i), st.inp(i, e.stats_off)
            ref = up + F.interpolate(low, scale_factor=2)
            fref[i] = ref
            errs[K_UPADD].append(rel_err(st.out(i), ref))
            planted.setdefault(K_UPADD, rel_err(st.out(i), F.interpolate(low, scale_factor=2)))   # skip dropped
        elif e.kind == K_CAT:
            # the reference of each half comes from its producer's own inputs: the prior network's last up-add and the
            # encoder's last InstanceNorm + ReLU
            cat = st.read(e.out_off, (e.n, e.h, e.w, e.c, e.ld))
            prod = lambda off: max(j for j in range(i) if T[j].out_off == off and T[j].kind in (K_UPADD, K_NORM))
            jp, je = prod(e.in_off), prod(e.stats_off)
            assert T[jp].kind == K_UPADD and T[je].kind == K_NORM
            errs[K_CAT].append(rel_err(cat, torch.cat((fref[jp], fref[je]), 1)))
            planted[K_CAT] = rel_err(cat, torch.cat((fref[je], fref[jp]), 1))
        elif e.kind == K_HEADS:
            f = st.read(e.in_off, (e.n, e.h, e.w, 64, 128))
            wp = bf16_round(st.param(e.w_idx).float()).double()
            wl = bf16_round(st.param(e.w_idx + 2).float()).double()
            parsing = F.conv2d(f, wp, st.param(e.w_idx + 1))
            landmark = F.conv2d(f, wl)
            lm, ps = st.outs[2].double().cpu(), st.outs[3].double().cpu()
            errs[K_HEADS] += [rel_err(lm, landmark), rel_err(ps, parsing)]
            w_all = torch.cat((wp, wl), 0)                   # the 13 / 68 split shifted by one channel
            shifted = F.conv2d(f, w_all[1:14])
            planted[K_HEADS] = rel_err(ps, shifted + st.param(e.w_idx + 1).view(1, -1, 1, 1))
        elif e.kind == K_TANH:
            y = st.inp(i)
            out = st.outs[0 if e.out_off >= 0 else 1].double().cpu()
            errs[K_TANH].append(rel_err(out, torch.tanh(y)))
            planted.setdefault(K_TANH, rel_err(out, y))
            if e.out_off >= 0:                               # the bf16 copy the encoder and the prior network read
                errs[K_TANH].append(rel_err(st.out(i), bf16_round(torch.tanh(y).float()).double()))
    tols = {K_PAD: 0.0 + 1e-12, K_CONV: 5e-3, K_NORM: 8e-3, K_ADD: 4e-3, K_POOL: 1e-12, K_UPADD: 4e-3, K_CAT: 8e-3,
            K_HEADS: 5e-3, K_TANH: 1e-5}
    report = {}
    for k, tol in tols.items():
        report[k] = _check(errs[k], tol, planted[k])
    assert {"transposed", "1x1 s1 p0 cin cout", "3x3 s1 p1 cin cout", "3x3 s2 p0 cin cout", "3x3 s1 p0 cin cout",
            "7x7 s1 p0 cin3 cout", "3x3 s1 p0 cin3 cout", "3x3 s1 p0 cin cout3"} <= conv_cls, conv_cls
    print("one op deep, worst per kind:", report, "planted:", planted)


K_GOUT, K_GIN = 30, 31


def _grad_tape(b, h, w):
    from crfr_b200 import _lib as L
    n = L.lib().crfr_srnet_grad_tape(L.SRNET_NETWORK, b, h, w, 15, 1, None, 0)
    arr = (L.TapeEntry * n)()
    assert L.lib().crfr_srnet_grad_tape(L.SRNET_NETWORK, b, h, w, 15, 1, arr, n) == n
    return list(arr)


def _ad(fn, inputs, g):
    """float64 autograd of fn at the given inputs against the output gradient g."""
    leaves = [t.clone().requires_grad_(True) for t in inputs]
    torch.autograd.backward(fn(*leaves), g)
    return [t.grad for t in leaves]


def test_srnet_backward_one_op_deep(cuda):
    """Every op kind of the backward on its own stored tensors (crfr_srnet_grad_tape): the summed gradient an op consumed
    for its output, pushed through the op in float64 from its stored forward inputs, against the gradient it stored for
    each input.  Then the consumer sums: the gradient every producer consumed is the sum of what its consumers produced
    (the coarse image's two consumers, Bottleneck and hourglass inputs, the concat halves, the heads' input gradient).
    Each class of check rejects a planted error, among them one consumer slot of the coarse image left out."""
    from crfr_b200 import _lib as L
    from crfr_b200 import ops
    net = _net()
    b, h, w = 2, 32, 32
    st = Stored(net, b, h, w)
    T = st.tape
    g = torch.Generator().manual_seed(23)
    dys = [torch.randn(o.shape, generator=g).cuda() for o in st.outs]
    grads = [torch.zeros_like(p) for p in st.params]
    dx = torch.zeros_like(st.x)
    io = _io(L.SRNET_NETWORK, st.x, st.outs)
    L.call("crfr_srnet_backward", L.ENGINE_AUTO, _table(st.params), _table(grads), C.byref(io), _table(dys), dx.data_ptr(),
           st.ws.data_ptr(), st.ws.numel(), ops.stream())
    torch.cuda.synchronize()
    G = _grad_tape(b, h, w)
    rd = lambda e: st.read(e.out_off, (e.n, e.h, e.w, e.c, e.ld))
    gout = {}
    gin = {}
    for e in G:
        (gout if e.kind == K_GOUT else gin).setdefault(e.w_idx, []).append(e)
    kinds = {T[i].kind for i in gout}
    assert kinds == {K_CONV, K_NORM, K_POOL, K_UPADD, K_CAT, K_HEADS, K_PAD, K_ADD, K_TANH}, kinds
    errs, planted = {k: [] for k in kinds}, {}
    d_img = {True: dys[0].double().cpu(), False: dys[1].double().cpu()}   # coarse image / SR output gradients
    where = {k: [] for k in kinds}
    for i, outs in gout.items():
        e = T[i]
        n_before = {k: len(v) for k, v in errs.items()}
        go = sum(rd(o) for o in outs)
        ins = sorted(gin.get(i, []), key=lambda t: t.has_res)
        if e.kind == K_PAD:
            x = st.inp(i)
            ref, = _ad(lambda t: F.pad(t, (e.w_idx,) * 4, mode="reflect"), [x], go)
            errs[K_PAD].append(rel_err(rd(ins[0]), ref))
            if K_PAD not in planted:
                bad, = _ad(lambda t: F.pad(t, (e.w_idx,) * 4, mode="replicate"), [x], go)
                planted[K_PAD] = rel_err(rd(ins[0]), bad)
        elif e.kind == K_CONV:
            if not ins:                                   # the stem convolution without an input gradient
                continue
            m = st.module_of(e.w_idx)
            x = st.inp(i)
            wq = bf16_round(st.param(e.w_idx).float()).double()
            if isinstance(m, torch.nn.ConvTranspose2d):
                fn = lambda t, wt=wq: F.conv_transpose2d(t, wt, None, m.stride, m.padding, m.output_padding)
            else:
                fn = lambda t, wt=wq: F.conv2d(t, wt, None, m.stride, m.padding)
            ref, = _ad(fn, [x], go)
            errs[K_CONV].append(rel_err(rd(ins[0]), ref))
            if K_CONV not in planted and m.kernel_size[0] == 3 and not isinstance(m, torch.nn.ConvTranspose2d):
                bad, = _ad(lambda t: fn(t, wq.flip(2, 3)), [x], go)   # the kernel not flipped in the dgrad
                planted[K_CONV] = rel_err(rd(ins[0]), bad)
        elif e.kind == K_NORM:
            # against the single-op entry point (crfr_norm_act_bwd) on the same stored tensors: the program's wiring
            # (which map, statistics, parameters, residual and slots reach the kernel, where its results go).  The
            # kernel's own accuracy is the single-op path's (DESIGN 6f: it loses accuracy where a channel's mean is large
            # against its spread, as in the deepest hourglass levels, so a float64 reference does not bound it here).
            conv_key = st.keys[T[i - 1].w_idx] if T[i - 1].kind == K_CONV else ""
            rb = conv_key.endswith(("conv1.weight", "conv2.weight")) and ".hg." not in conv_key
            gamma = beta = alpha = res = None
            if rb and conv_key.endswith("conv1.weight"):
                idx = st.keys.index(conv_key[:-len("conv1.weight")] + "in1.weight")
                gamma, beta, alpha = (st.params[idx + j] for j in range(3))
            elif rb and e.has_res:
                idx = st.keys.index(conv_key[:-len("conv2.weight")] + "in2.weight")
                gamma, beta = st.params[idx], st.params[idx + 1]
                res = st.raw(T[i - 3].in_off, st.dims_of(i - 3, T[i - 3].in_off))
            y = st.raw(e.in_off, st.dims_of(i, e.in_off))
            stats = st.ws[e.stats_off:e.stats_off + e.n * e.c * 8].view(torch.float32).view(e.n, e.c, 2)
            slots = [st.raw(o.out_off, (o.n, o.h, o.w, o.c, o.ld)) for o in outs]
            relu = alpha is None and not e.has_res
            dz, dyk, *_ = ops.norm_act_bwd(slots[0], y, stats, gamma, beta, alpha, relu, res,
                                           slots[1] if len(slots) > 1 else None)
            nchw = lambda t: t.permute(0, 3, 1, 2).double().cpu()
            errs[K_NORM].append(rel_err(rd(ins[0]), nchw(dyk)))
            if e.has_res:
                errs[K_NORM].append(rel_err(rd(ins[1]), nchw(dz)))
            if K_NORM not in planted and relu:                 # the ReLU mask left out
                _, bad, *_ = ops.norm_act_bwd(slots[0], y, stats, None, None, None, False, None,
                                              slots[1] if len(slots) > 1 else None)
                planted[K_NORM] = rel_err(rd(ins[0]), nchw(bad))
        elif e.kind == K_ADD:
            errs[K_ADD] += [rel_err(rd(ins[0]), go), rel_err(rd(ins[1]), go)]
            planted.setdefault(K_ADD, rel_err(rd(ins[1]), 2 * go))
        elif e.kind == K_POOL:
            x = st.inp(i)
            ref, = _ad(lambda t: F.max_pool2d(t, 2, 2), [x], go)
            errs[K_POOL].append(rel_err(rd(ins[0]), ref))
            bad, = _ad(lambda t: F.avg_pool2d(t, 2, 2), [x], go)
            planted.setdefault(K_POOL, rel_err(rd(ins[0]), bad))
        elif e.kind == K_UPADD:
            low = st.inp(i, e.stats_off)
            ref, = _ad(lambda t: F.interpolate(t, scale_factor=2), [low], go)
            errs[K_UPADD] += [rel_err(rd(ins[0]), go), rel_err(rd(ins[1]), ref)]
            planted.setdefault(K_UPADD, rel_err(rd(ins[1]), ref / 4))     # averaged instead of summed
        elif e.kind == K_CAT:
            errs[K_CAT] += [rel_err(rd(ins[0]), go[:, :64]), rel_err(rd(ins[1]), go[:, 64:])]
            planted[K_CAT] = rel_err(rd(ins[0]), go[:, 64:])
        elif e.kind == K_HEADS:
            # the gathered output gradient: parsing in channels 0..12, landmark in 13..80, zeros after
            want = torch.zeros_like(go)
            want[:, :13], want[:, 13:81] = dys[3].double().cpu(), dys[2].double().cpu()
            errs[K_HEADS].append(rel_err(go, bf16_round(want.float()).double()))
            shifted = torch.zeros_like(go)
            shifted[:, :13], shifted[:, 14:82] = dys[3].double().cpu(), dys[2].double().cpu()
            planted[K_HEADS] = rel_err(go, shifted)
            f = st.read(e.in_off, (e.n, e.h, e.w, 64, 128))
            wc = torch.cat((bf16_round(st.param(e.w_idx).float()), bf16_round(st.param(e.w_idx + 2).float())), 0).double()
            ref, = _ad(lambda t: F.conv2d(t, wc), [f], go[:, :81])
            errs[K_HEADS].append(rel_err(rd(ins[0]), ref))
        elif e.kind == K_TANH:
            coarse = e.out_off >= 0
            y = st.inp(i)
            tot = d_img[coarse] + go                    # the caller's gradient + the coarse copy's consumer slots
            ref, = _ad(torch.tanh, [y], tot)
            errs[K_TANH].append(rel_err(rd(ins[0]), ref))
            # the tanh derivative left out (a dropped consumer slot of the coarse image is the consumer-sum check's
            # planted error below: here the caller's own gradient dominates the sum)
            planted.setdefault(K_TANH, rel_err(rd(ins[0]), tot))
        for k in errs:
            where[k] += [(i, st.keys[e.w_idx] if e.kind == K_CONV else e.h)] * (len(errs[k]) - n_before[k])
    for k in errs:
        if errs[k]:
            j = max(range(len(errs[k])), key=lambda t: errs[k][t])
            print("kind %d worst %.3e at op %s" % (k, errs[k][j], where[k][j]))
    tols = {K_PAD: 4e-3, K_CONV: 5e-3, K_NORM: 1e-3, K_ADD: 0.0 + 1e-12, K_POOL: 1e-2, K_UPADD: 4e-3,
            K_CAT: 1e-12, K_HEADS: 5e-3, K_TANH: 4e-3}
    report = {k: _check(errs[k], tol, planted[k]) for k, tol in tols.items()}

    # consumer sums: per tensor (offset, channels), the consumed gradient against the sum of the produced ones
    produced, consumed = {}, {}
    for e in G:
        if e.in_off < 0:
            continue
        key = (e.in_off, e.c)
        (produced if e.kind == K_GIN else consumed).setdefault(key, []).append(e)
    # where the producer reads its consumers' own buffers (no sum materialised), they must be exactly those buffers;
    # where the slots were summed into a new buffer, that buffer must be their sum.  (Magnitudes of the slots can differ
    # by many orders - the prior network's gradient at the coarse image dwarfs the encoder's - so a missing slot is
    # looked for by buffer, not by a norm-wise sum.)
    def consumer_sum_error(outs, ins):
        co, pi = sorted(o.out_off for o in outs), sorted(t.out_off for t in ins)
        if set(co) <= set(pi):
            return 0.0 if co == pi else 1.0
        return rel_err(sum(rd(o) for o in outs), sum(rd(t) for t in ins))

    sums = []
    multi = 0
    for key, outs in consumed.items():
        ins = produced.get(key, [])
        assert ins, ("a consumed gradient no consumer produced", key)
        multi += len(ins) > 1
        sums.append(consumer_sum_error(outs, ins))
    assert multi > 100, multi                           # Bottleneck / hourglass inputs, the coarse copy, the features
    c4 = [k for k, v in consumed.items() if T[v[0].w_idx].kind == K_TANH]
    assert len(c4) == 1 and len(produced[c4[0]]) == 2   # the coarse image: one slot per consumer
    dropped = consumer_sum_error(consumed[c4[0]][:1], produced[c4[0]])    # one consumer slot of the coarse image left out
    report["sums"] = _check(sums, 5e-3, dropped)
    print("backward one op deep, worst per kind:", report, "planted:", planted, "dropped coarse slot:", dropped)
