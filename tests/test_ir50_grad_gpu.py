"""IR_50's gradient with respect to the input image (crfr_ir50_backward through the autograd path of model_irse.Backbone):
parity with fp32 autograd through the oracle, batch independence, determinism, unchanged no-grad outputs, and the
composition with FSRNet that an identity / perceptual loss on a super-resolved face needs."""
import pytest
import torch
import torch.nn.functional as F

from tests.util import rel_err

pytestmark = pytest.mark.gpu

STAGE_ENDS = (2, 6, 20, 23)


def _gscale(v, k):
    """v in the forward, its gradient multiplied by k (used to plant known errors into the reference)."""
    return v * k - (v * (k - 1)).detach()


def _ir50_ref(sd, x, pr, feed=None, mutate=None):
    """``oracle.resnet_oracle.ir50_forward`` with the gradient roundings (``pr.qg``) at the points where the native
    backward stores a bf16 gradient: the conv-input gradients of res_layer.3 and of the stem, the PReLU output gradient,
    the gradient entering each unit through res_layer.0 and through a conv shortcut, each unit's summed output gradient,
    the seeds, and the head's input gradient.  BatchNorm scales folded into dgrad weights have no rounding of their own.
    Forward values are those of the oracle (``test_ir50_grad_ref.py`` checks that), or with ``feed`` (the stored tensors
    in the order of ``crfr_ir50_tape``) those of another implementation, straight-through for the gradient.
    ``mutate``: (kind, unit[, factor]) plants a known error into the gradient - "drop_s4" / "drop_s0" leave out the
    folded scale of res_layer.4 / res_layer.0, "scale" multiplies the residual branch's gradient by factor.
    -> (embedding, [x1, x2, x3, x4])."""
    from oracle.resnet_oracle import BN_EPS, ir50_block_specs
    q, qg = pr.q, pr.qg
    feed = None if feed is None else iter(feed)

    def st(v):   # a stored activation
        if feed is None:
            return q(v)
        f = next(feed)
        return v + (f.reshape(v.shape) - v).detach()

    def scale(p):
        return (sd[p + "weight"] / torch.sqrt(sd[p + "running_var"] + BN_EPS)).view(1, -1, 1, 1)

    def bn(y, p, res=None):
        shape = (1, -1, 1, 1) if y.dim() == 4 else (1, -1)
        z = (y - sd[p + "running_mean"].view(shape)) / torch.sqrt(sd[p + "running_var"].view(shape) + BN_EPS)
        z = z * sd[p + "weight"].view(shape) + sd[p + "bias"].view(shape)
        return z if res is None else z + res

    def prelu(z, a):
        a = a.view(1, -1, 1, 1)
        return torch.clamp(z, min=0) + a * torch.clamp(z, max=0)

    def conv(v, w, stride, pad):
        return st(F.conv2d(v, q(w), None, stride, pad))

    kind, mu = (mutate[0], mutate[1]) if mutate else (None, -1)
    y0 = qg(conv(qg(q(x)), sd["input_layer.0.weight"], 1, 1))
    a = st(prelu(bn(y0, "input_layer.1."), sd["input_layer.2.weight"]))
    feats = []
    for i, (cin, d, stride) in enumerate(ir50_block_specs()):
        p = "body.%d." % i
        if cin != d:
            sc = st(bn(conv(qg(a), sd[p + "shortcut_layer.0.weight"], stride, 0), p + "shortcut_layer.1."))
        else:
            sc = a[:, :, ::stride, ::stride]
            if stride == 2:
                sc = st(sc)
        a_r = qg(a)
        if i == mu and kind == "drop_s0":
            a_r = _gscale(a_r, 1 / scale(p + "res_layer.0."))
        r = st(bn(a_r, p + "res_layer.0."))
        y1 = qg(conv(r, sd[p + "res_layer.1.weight"], 1, 1))
        r2 = qg(st(prelu(y1, sd[p + "res_layer.2.weight"])))
        y3 = conv(r2, sd[p + "res_layer.3.weight"], stride, 1)
        if i == mu and kind == "drop_s4":
            y3 = _gscale(y3, 1 / scale(p + "res_layer.4."))
        if i == mu and kind == "scale":
            y3 = _gscale(y3, mutate[2])
        a = qg(st(bn(y3, p + "res_layer.4.", res=sc)))
        if i in STAGE_ENDS:   # the seed and the gradient from downstream are stored apart, then summed
            feats.append(qg(a))
            a = qg(a)
    o = st(bn(qg(a), "output_layer.0.")).reshape(a.shape[0], -1)
    y = st(F.linear(o, q(sd["output_layer.3.weight"]), sd["output_layer.3.bias"]))
    emb = qg(st(bn(y, "output_layer.4.")))
    if feed is not None:
        assert next(feed, None) is None, "the reference consumed fewer stored tensors than the tape lists"
    return emb, feats


def _net(sd):
    from crfr_b200.model.model_irse import IR_50
    net = IR_50([112, 112])
    net.load_state_dict(sd)
    return net.cuda().eval()


def _state():
    from oracle import resnet_oracle as RO
    return RO.randomize_bn_everywhere(RO.build_ir50_state_dict(91), 191)


def _seeds(b, seed=77):
    g = torch.Generator().manual_seed(seed)
    shapes = ((b, 512), (b, 64, 56, 56), (b, 128, 28, 28), (b, 256, 14, 14), (b, 512, 7, 7))
    return [torch.randn(s, generator=g) for s in shapes]


CASES = {"emb": (0,), "features": (1, 2, 3, 4), "all": (0, 1, 2, 3, 4)}


def _native_dx(net, x, seeds, which, **kw):
    x = x.cuda().requires_grad_(True)
    outs = net.forward_features(x)
    return torch.autograd.grad([outs[k] for k in which], x, [seeds[k].cuda() for k in which], **kw)[0]


def test_ir50_input_grad_parity(cuda):
    from oracle import resnet_oracle as RO
    sd = _state()
    net = _net(sd)
    x = RO.synthetic_faces(4, seed=4322)
    seeds = _seeds(4)
    ref = {}
    for name in ("fp32", "bf16"):
        xr = x.clone().requires_grad_(True)
        emb, feats = _ir50_ref(sd, xr, RO.Precision(name))
        outs = (emb,) + tuple(feats)
        ref[name] = {c: torch.autograd.grad([outs[k] for k in ks], xr, [seeds[k] for k in ks], retain_graph=True)[0]
                     for c, ks in CASES.items()}
    for c, ks in CASES.items():
        dx = _native_dx(net, x, seeds, ks).cpu()
        exact, emu = ref["fp32"][c], ref["bf16"][c]
        assert dx.shape == (4, 3, 112, 112) and torch.isfinite(dx).all()
        err, err_bf16 = rel_err(dx, exact), rel_err(emu, exact)
        # free-running, the bf16-stored forward flips PReLU masks of values near zero (the bf16 oracle is ~0.17 from the
        # exact gradient at this depth): this bound is coarse, test_ir50_input_grad_teacher_forced is the tight one
        assert err <= 1.4 * err_bf16 + 2e-3, (c, err, err_bf16)


def _tape(b):
    from crfr_b200 import _lib as L
    n = L.lib().crfr_ir50_tape(b, 112, None, 0)
    assert n > 0
    arr = (L.TapeEntry * n)()
    assert L.lib().crfr_ir50_tape(b, 112, arr, n) == n
    return list(arr)


def _stored(ws, e):
    v = torch.as_strided(ws.view(torch.bfloat16), (e.n, e.h, e.w, e.c), (e.h * e.w * e.ld, e.w * e.ld, e.ld, 1), e.out_off // 2)
    return v.float().permute(0, 3, 1, 2).contiguous().cpu()


def test_ir50_tape_lists_every_storage_point(cuda):
    tape = _tape(4)
    # stem conv + BN/PReLU, 24 units x (BN, conv, PReLU, conv, BN) + 3 x (shortcut conv, BN) + 1 subsampling, head BN,
    # linear, BN1d
    assert len(tape) == 2 + 24 * 5 + 3 * 2 + 1 + 3
    kinds = [e.kind for e in tape]
    assert kinds.count(0) == 1 + 24 * 2 + 3 and kinds.count(8) == 24 and kinds.count(9) == 1 and kinds[-2] == 7


def _native_forced(net, x, seeds):
    """crfr_ir50_forward into a grad-sized workspace, then crfr_ir50_backward for each case -> ({case: dx}, stored
    tensors in tape order, (emb, feats))."""
    import ctypes as C
    from crfr_b200 import _lib as L
    from crfr_b200 import ops
    b = x.shape[0]
    xg = x.cuda().contiguous()
    ws = torch.empty(L.lib().crfr_ir50_grad_workspace_bytes(b, 112), dtype=torch.uint8, device="cuda")
    emb, feats, (ptab, btab), io = net._launch(xg, True, ws)
    gs = [t.cuda().contiguous() for t in seeds]
    dxs = {}
    for c, ks in CASES.items():
        dfeat = (C.c_void_p * 4)(*[gs[k].data_ptr() if k in ks else None for k in (1, 2, 3, 4)])
        dx = torch.empty_like(xg)
        L.call("crfr_ir50_backward", net.engine, ptab.arr, btab.arr, C.byref(io), gs[0].data_ptr() if 0 in ks else None,
               dfeat, dx.data_ptr(), ws.data_ptr(), ws.numel(), ops.stream())
        dxs[c] = dx.cpu()
    torch.cuda.synchronize()
    return dxs, [_stored(ws, e) for e in _tape(b)], (emb.cpu(), [f.cpu() for f in feats])


_FORCED_REF = {}


def _forced_refs(sd, x, seeds, stored):
    """Exact and bf16 gradients of the reference on the native program's stored forward, cached per stored forward."""
    from oracle import resnet_oracle as RO
    key = stored[-1].numpy().tobytes()
    if key not in _FORCED_REF:
        ref = {}
        for name in ("fp32", "bf16"):
            xr = x.clone().requires_grad_(True)
            emb, feats = _ir50_ref(sd, xr, RO.Precision(name), feed=stored)
            outs = (emb,) + tuple(feats)
            ref[name] = ({c: torch.autograd.grad([outs[k] for k in ks], xr, [seeds[k] for k in ks], retain_graph=True)[0]
                          for c, ks in CASES.items()}, outs)
        mutants = {}
        for m in (("drop_s4", 22), ("drop_s0", 4), ("drop_s0", 15), ("scale", 5, 1.25), ("scale", 12, 0.8),
                  ("scale", 22, 1.1)):
            xr = x.clone().requires_grad_(True)
            emb, feats = _ir50_ref(sd, xr, RO.Precision("bf16"), feed=stored, mutate=m)
            outs = (emb,) + tuple(feats)
            mutants[m] = {c: torch.autograd.grad([outs[k] for k in ks], xr, [seeds[k] for k in ks], retain_graph=True)[0]
                          for c, ks in CASES.items()}
        _FORCED_REF[key] = (ref, mutants)
    return _FORCED_REF[key]


def test_ir50_input_grad_teacher_forced(cuda):
    """The reference replays the native program's stored bf16 activations (``crfr_ir50_tape``), so both see the same PReLU
    masks and the backward - linear once the forward is fixed - is compared without the chaos of free-running rounding
    flips.  The same bound must reject a reference with one known error planted (a folded BatchNorm scale left out, one
    unit's residual gradient scaled)."""
    from oracle import resnet_oracle as RO
    sd = _state()
    net = _net(sd)
    x = RO.synthetic_faces(4, seed=4322)
    seeds = _seeds(4)
    dxs, stored, (emb, feats) = _native_forced(net, x, seeds)
    assert len(stored) == len(_tape(4))
    (ref, mutants) = _forced_refs(sd, x, seeds, stored)
    for a, b in zip((emb,) + tuple(feats), ref["fp32"][1]):   # the forced forward reproduces the native outputs
        assert rel_err(a, b) < 1e-6
    for c in CASES:
        dx, exact, emu = dxs[c], ref["fp32"][0][c], ref["bf16"][0][c]
        assert torch.isfinite(dx).all()
        err, err_bf16 = rel_err(dx, exact), rel_err(emu, exact)
        cos = F.cosine_similarity(dx.double().reshape(-1), exact.double().reshape(-1), dim=0).item()
        print("IR_50 dx teacher-forced (%s): %.2e to the exact backward (bf16 reference %.2e), cosine %.6f"
              % (c, err, err_bf16, cos))
        bound = 1.4 * err_bf16 + 2e-3
        assert err <= bound, (c, err, err_bf16)
        assert cos > 0.999, (c, cos)
        for m, dm in mutants.items():   # the bound is tight enough to see each planted error
            assert rel_err(dm[c], exact) > bound, (c, m, rel_err(dm[c], exact), bound)


def test_ir50_input_grad_batch_independent(cuda):
    from oracle import resnet_oracle as RO
    net = _net(_state())
    x = RO.synthetic_faces(8, seed=4322)
    seeds = _seeds(8)
    full = _native_dx(net, x, seeds, CASES["all"])
    halves = [_native_dx(net, x[h], [s[h] for s in seeds], CASES["all"]) for h in (slice(0, 4), slice(4, 8))]
    assert torch.equal(full, torch.cat(halves))


def test_ir50_input_grad_deterministic_and_repeatable(cuda):
    from oracle import resnet_oracle as RO
    net = _net(_state())
    x = RO.synthetic_faces(4, seed=4322)
    seeds = _seeds(4)
    a = _native_dx(net, x, seeds, CASES["all"])
    b = _native_dx(net, x, seeds, CASES["all"])
    assert torch.equal(a, b)
    xg = x.cuda().requires_grad_(True)
    outs = net.forward_features(xg)
    loss = sum((o * s.cuda()).sum() for o, s in zip(outs, seeds))
    loss.backward(retain_graph=True)
    g1 = xg.grad.clone()
    xg.grad = None
    loss.backward(retain_graph=True)
    assert torch.equal(g1, xg.grad)
    assert torch.equal(g1, a)


def test_ir50_no_grad_outputs_unchanged(cuda):
    from oracle import resnet_oracle as RO
    net = _net(_state())
    x = RO.synthetic_faces(4, seed=4322).cuda()
    plain = net.forward_features(x)
    emb = net(x)
    with_grad = net.forward_features(x.clone().requires_grad_(True))
    assert with_grad[0].grad_fn is not None and plain[0].grad_fn is None
    for p, g in zip(plain, with_grad):
        assert torch.equal(p, g)
    assert torch.equal(emb, net(x.clone().requires_grad_(True)))
    with torch.no_grad():
        assert net(x.clone().requires_grad_(True)).grad_fn is None
    # parameters stay frozen even when they require a gradient
    assert all(p.requires_grad for p in net.parameters())
    net(x.clone().requires_grad_(True)).sum().backward()
    assert all(p.grad is None for p in net.parameters())
    net.train()
    with pytest.raises(RuntimeError):
        net(x.clone().requires_grad_(True))


def test_ir50_workspace_prefix(cuda):
    from crfr_b200 import _lib as L
    lib = L.lib()
    # the forward's arena, and so the KD step's layout, is the one it was before the backward existed
    assert [lib.crfr_ir50_workspace_bytes(b, 112) for b in (1, 4, 256)] == [155848704, 273567744, 10161967104]
    for b in (1, 4, 256):
        assert lib.crfr_ir50_grad_workspace_bytes(b, 112) > lib.crfr_ir50_workspace_bytes(b, 112)
    assert lib.crfr_ir50_grad_workspace_bytes(4, 96) == 0


def test_ir50_identity_loss_drives_fsrnet(cuda):
    """An identity / perceptual loss on IR_50 features of FSRNet's output (cropped to 112) reaches FSRNet's parameters
    exactly as IR_50's input gradient fed to FSRNet's backward does; IR_50's parameters receive nothing."""
    from crfr_b200.model.FSRnet import OverallNetwork, weights_init
    from oracle import resnet_oracle as RO
    torch.manual_seed(1234)
    fsr = OverallNetwork()
    fsr.apply(weights_init)
    fsr = fsr.cuda().train()
    ir50 = _net(_state())
    g = torch.Generator().manual_seed(5)
    lr = torch.rand(2, 3, 128, 128, generator=g).cuda()
    hr = RO.synthetic_faces(2, seed=4323).cuda()
    with torch.no_grad():
        f_hr = ir50.forward_features(hr)

    def crop():
        return fsr(lr)[1][:, :, 8:120, 8:120]

    sr = crop()
    loss = F.mse_loss(sr, hr) + sum(F.mse_loss(a, b) for a, b in zip(ir50.forward_features(sr), f_hr))
    loss.backward()
    got = {k: p.grad.clone() for k, p in fsr.named_parameters() if p.grad is not None}   # (not every head reaches out[1])
    assert got
    assert all(p.grad is None for p in ir50.parameters())

    sr_leaf = sr.detach().requires_grad_(True)
    id_loss = sum(F.mse_loss(a, b) for a, b in zip(ir50.forward_features(sr_leaf), f_hr))
    d_sr = torch.autograd.grad(id_loss, sr_leaf)[0]
    assert d_sr.abs().sum() > 0
    fsr.zero_grad(set_to_none=True)
    sr2 = crop()
    torch.autograd.backward([sr2, F.mse_loss(sr2, hr)], [d_sr, None])
    assert {k for k, p in fsr.named_parameters() if p.grad is not None} == set(got)
    for k, g in got.items():
        assert rel_err(fsr.get_parameter(k).grad, g) < 1e-5, k
    # the identity term does contribute
    fsr.zero_grad(set_to_none=True)
    F.mse_loss(crop(), hr).backward()
    assert any(rel_err(fsr.get_parameter(k).grad, g) > 1e-4 for k, g in got.items())
