"""IR_101 / IR_152 and the squeeze-excitation teachers IR_SE_50 / 101 / 152 on the GPU (crfr_irnet_* through
model_irse.Backbone): forward parity, the excitation of every SE unit, the teacher-forced input gradient with planted
errors, batch independence and determinism, and the KD step with these teachers."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from tests.irnet_oracle import (bn_affine, build_irnet_state_dict, irnet_block_specs, irnet_forward, se_excitation,
                                se_from_pooled, stage_ends)
from tests.test_ir50_grad_gpu import CASES, _gscale, _seeds, _stored
from tests.test_resnet_gpu import SLACK
from tests.util import rel_err

pytestmark = pytest.mark.gpu

# constructor name -> (num_layers, se)
VARIANTS = {"IR_SE_50": (50, 1), "IR_101": (100, 0), "IR_SE_101": (100, 1), "IR_152": (152, 0), "IR_SE_152": (152, 1)}
# the gradient seeds of the teacher-forced checks: those of the IR_50 tests, and one on x4 alone (7 x 7 pixels: the SE
# squeeze path dpool / hw is largest relative to e * g there)
GRAD_CASES = dict(CASES, x4=(4,))


def _state(name):
    from oracle import resnet_oracle as RO
    return RO.randomize_bn_everywhere(build_irnet_state_dict(91, *VARIANTS[name]), 191)


def _net(name, sd):
    from crfr_b200.model import model_irse as M
    net = getattr(M, name)([112, 112])
    net.load_state_dict(sd)
    return net.cuda().eval()


@pytest.mark.parametrize("name", sorted(VARIANTS))
def test_irnet_forward_parity(cuda, name):
    from oracle import resnet_oracle as RO
    sd = _state(name)
    net = _net(name, sd)
    x = RO.synthetic_faces(4, seed=4322)
    with torch.no_grad():
        outs = net.forward_features(x.cuda())
        emb = net(x.cuda())
        ref_emb, ref = irnet_forward(sd, x, want_features=True)
        emu_emb, emu = irnet_forward(sd, x, pr=RO.Precision("bf16"), want_features=True)
    assert torch.equal(outs[0], emb)
    with_grad = net.forward_features(x.cuda().requires_grad_(True))
    assert with_grad[0].grad_fn is not None
    for a, b in zip(outs, with_grad):
        assert torch.equal(a, b)
    shapes = ((512,), (64, 56, 56), (128, 28, 28), (256, 14, 14), (512, 7, 7))
    for k, (o, r, e, shape) in enumerate(zip(outs, [ref_emb] + ref, [emu_emb] + emu, shapes)):
        assert tuple(o.shape) == (4,) + shape and torch.isfinite(o).all()
        err, err_bf16 = rel_err(o, r), rel_err(e, r)
        print("%s output %d: %.2e from the fp32 oracle (bf16 oracle %.2e)" % (name, k, err, err_bf16))
        assert err < SLACK * err_bf16 + 1e-2, (name, k, err, err_bf16)


def _tape(num_layers, se, b):
    from crfr_b200 import _lib as L
    n = L.lib().crfr_irnet_tape(num_layers, se, b, 112, None, 0)
    assert n > 0
    arr = (L.TapeEntry * n)()
    assert L.lib().crfr_irnet_tape(num_layers, se, b, 112, arr, n) == n
    return list(arr)


def _native_forced(name, net, x, seeds, cases):
    """crfr_irnet_forward into a grad-sized workspace, then crfr_irnet_backward for each case -> ({case: dx}, the tape,
    the workspace, (emb, feats))."""
    from crfr_b200 import _lib as L
    from crfr_b200 import ops
    num_layers, se = net._variant
    assert name not in VARIANTS or VARIANTS[name] == net._variant
    b = x.shape[0]
    xg = x.cuda().contiguous()
    ws = torch.empty(L.lib().crfr_irnet_grad_workspace_bytes(num_layers, se, b, 112), dtype=torch.uint8, device="cuda")
    emb, feats, (ptab, btab), io = net._launch(xg, True, ws)
    gs = [t.cuda().contiguous() for t in seeds]
    dxs = {}
    for c, ks in cases.items():
        dfeat = (C.c_void_p * 4)(*[gs[k].data_ptr() if k in ks else None for k in (1, 2, 3, 4)])
        dx = torch.empty_like(xg)
        L.call("crfr_irnet_backward", net.engine, num_layers, se, ptab.arr, btab.arr, C.byref(io),
               gs[0].data_ptr() if 0 in ks else None, dfeat, dx.data_ptr(), ws.data_ptr(), ws.numel(), ops.stream())
        dxs[c] = dx.cpu()
    torch.cuda.synchronize()
    return dxs, _tape(num_layers, se, b), ws, (emb.cpu(), [f.cpu() for f in feats])


def test_irnet_excitation_exact(cuda):
    """Teacher-forced from the tape: the native excitation e [n][c] of every SE unit of IR_SE_50 equals the fp32 SE of the
    oracle computed from the stored res_layer.3 output."""
    from oracle import resnet_oracle as RO
    sd = _state("IR_SE_50")
    net = _net("IR_SE_50", sd)
    x = RO.synthetic_faces(4, seed=4322)
    _, tape, ws, _ = _native_forced("IR_SE_50", net, x, _seeds(4), {})
    by_out = {e.out_off: e for e in tape}
    se_ops = [e for e in tape if e.kind == 10]
    assert len(se_ops) == len(irnet_block_specs(50))
    worst = 0.0
    for i, e in enumerate(se_ops):
        conv = by_out[e.in_off]
        assert conv.kind == 0 and conv.c == e.c
        y = _stored(ws, conv)
        native = ws[e.stats_off:e.stats_off + 4 * e.n * e.c].view(torch.float32).view(e.n, e.c).cpu()
        ref = se_excitation(sd, "body.%d." % i, y)
        err = rel_err(native, ref)
        worst = max(worst, err)
        assert err <= 1e-5, (i, err)
    print("IR_SE_50 excitation: worst unit %.2e from the fp32 oracle on the stored res_layer.3 outputs" % worst)


def _ir_ref(sd, x, pr, num_layers, se, feed=None, mutate=None):
    """``tests.test_ir50_grad_gpu._ir50_ref`` for every variant: the forward of ``irnet_forward`` with the gradient
    roundings (``pr.qg``) where the native backward stores a bf16 gradient.  In an SE unit that is the gradient at the SE
    input z = BN_4(y) (dr = e * g + dpool / hw, one stored map) besides the unit's output gradient.  ``feed``: the stored
    tensors in tape order, straight-through for the gradient.  ``mutate``: (kind, unit[, factor]) plants a known error -
    "drop_s4" leaves out res_layer.4's folded scale, "scale" scales the unit's residual gradient, and in an SE unit
    "no_squeeze" leaves out the squeeze path (dpool / hw) and "no_e" the factor e of dr.  -> (embedding, [x1 .. x4])."""
    from oracle.resnet_oracle import BN_EPS
    q, qg = pr.q, pr.qg
    feed = None if feed is None else iter(feed)
    ends = stage_ends(num_layers)

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

    def excite(z, p):
        return se_from_pooled(sd, p, z.mean(dim=(2, 3)))[:, :, None, None]

    kind, mu = (mutate[0], mutate[1]) if mutate else (None, -1)
    y0 = qg(conv(qg(q(x)), sd["input_layer.0.weight"], 1, 1))
    a = st(prelu(bn(y0, "input_layer.1."), sd["input_layer.2.weight"]))
    feats = []
    for i, (cin, d, stride) in enumerate(irnet_block_specs(num_layers)):
        p = "body.%d." % i
        if cin != d:
            sc = st(bn(conv(qg(a), sd[p + "shortcut_layer.0.weight"], stride, 0), p + "shortcut_layer.1."))
        else:
            sc = a[:, :, ::stride, ::stride]
            if stride == 2:
                sc = st(sc)
        r = st(bn(qg(a), p + "res_layer.0."))
        y1 = qg(conv(r, sd[p + "res_layer.1.weight"], 1, 1))
        r2 = qg(st(prelu(y1, sd[p + "res_layer.2.weight"])))
        y3 = conv(r2, sd[p + "res_layer.3.weight"], stride, 1)
        if i == mu and kind == "drop_s4":
            y3 = _gscale(y3, 1 / scale(p + "res_layer.4."))
        if i == mu and kind == "scale":
            y3 = _gscale(y3, mutate[2])
        if se:   # z = BN_4(y3) as s * y3 + t (the oracle's form)
            s4, t4 = bn_affine(sd, p + "res_layer.4.")
            z = qg(y3 * s4.view(1, -1, 1, 1) + t4.view(1, -1, 1, 1))
            if i == mu and kind == "no_squeeze":
                out = z * excite(z.detach(), p)
            elif i == mu and kind == "no_e":
                out = z.detach() * excite(z, p) + (z - z.detach())
            else:
                out = z * excite(z, p)
            a = qg(st(out + sc))
        else:
            a = qg(st(bn(y3, p + "res_layer.4.", res=sc)))
        if i in ends:   # the seed and the gradient from downstream are stored apart, then summed
            feats.append(qg(a))
            a = qg(a)
    o = st(bn(qg(a), "output_layer.0.")).reshape(a.shape[0], -1)
    y = st(F.linear(o, q(sd["output_layer.3.weight"]), sd["output_layer.3.bias"]))
    emb = qg(st(bn(y, "output_layer.4.")))
    if feed is not None:
        assert next(feed, None) is None, "the reference consumed fewer stored tensors than the tape lists"
    return emb, feats


# planted errors per variant: e left out of dr in a 14 x 14 unit, the squeeze path left out in a 7 x 7 unit.  In IR_SE_50 the
# squeeze term dpool / hw of any single unit stays inside the bf16 noise that the bound allows, for every seed including one on
# x4 alone (at most 0.99 of the bound: unit 22, x4 seed; the bf16 reference replaying its own stored forward, which reproduces
# the native distances to 1 %), so that mutant is planted in IR_SE_152, where it exceeds the bound 1.8-2.6x on every seed.
MUTANTS = {"IR_SE_50": (("no_e", 12),), "IR_SE_152": (("no_squeeze", 48), ("no_e", 30))}


@pytest.mark.parametrize("name", ["IR_SE_50", "IR_SE_152"])
def test_irnet_input_grad_teacher_forced(cuda, name):
    """As test_ir50_input_grad_teacher_forced: the reference replays the native program's stored activations, so both
    see the same PReLU masks and excitations, and dx must be within 1.4x the bf16 reference's distance to the exact
    backward (+ 2e-3), cosine > 0.999, for seeds on the embedding, the features, both, and x4 alone.  The same bound must
    reject a reference with one planted error (MUTANTS): e left out of dr, or the squeeze path dpool / hw of one unit left
    out."""
    from oracle import resnet_oracle as RO
    num_layers, se = VARIANTS[name]
    sd = _state(name)
    net = _net(name, sd)
    x = RO.synthetic_faces(4, seed=4322)
    seeds = _seeds(4)
    dxs, tape, ws, (emb, feats) = _native_forced(name, net, x, seeds, GRAD_CASES)
    stored = [_stored(ws, e) for e in tape]
    ref = {}
    for prec in ("fp32", "bf16"):
        xr = x.clone().requires_grad_(True)
        o = _ir_ref(sd, xr, RO.Precision(prec), num_layers, se, feed=stored)
        outs = (o[0],) + tuple(o[1])
        ref[prec] = ({c: torch.autograd.grad([outs[k] for k in ks], xr, [seeds[k] for k in ks], retain_graph=True)[0]
                      for c, ks in GRAD_CASES.items()}, outs)
    for a, b in zip((emb,) + tuple(feats), ref["fp32"][1]):   # the forced forward reproduces the native outputs
        assert rel_err(a, b.detach()) < 1e-5
    mutants = {}
    for m in MUTANTS[name]:
        xr = x.clone().requires_grad_(True)
        o = _ir_ref(sd, xr, RO.Precision("bf16"), num_layers, se, feed=stored, mutate=m)
        outs = (o[0],) + tuple(o[1])
        mutants[m] = {c: torch.autograd.grad([outs[k] for k in ks], xr, [seeds[k] for k in ks], retain_graph=True)[0]
                      for c, ks in GRAD_CASES.items()}
    for c in GRAD_CASES:
        dx, exact, emu = dxs[c], ref["fp32"][0][c], ref["bf16"][0][c]
        assert torch.isfinite(dx).all()
        err, err_bf16 = rel_err(dx, exact), rel_err(emu, exact)
        cos = F.cosine_similarity(dx.double().reshape(-1), exact.double().reshape(-1), dim=0).item()
        bound = 1.4 * err_bf16 + 2e-3
        print("%s dx teacher-forced (%s): %.2e to the exact backward (bf16 reference %.2e), cosine %.6f; mutants %s"
              % (name, c, err, err_bf16, cos, {m[0]: "%.2e" % rel_err(dm[c], exact) for m, dm in mutants.items()}))
        assert err <= bound, (c, err, err_bf16)
        assert cos > 0.999, (c, cos)
        for m, dm in mutants.items():
            assert rel_err(dm[c], exact) > bound, (c, m, rel_err(dm[c], exact), bound)


def _native_dx(net, x, seeds, which):
    x = x.cuda().requires_grad_(True)
    outs = net.forward_features(x)
    return torch.autograd.grad([outs[k] for k in which], x, [seeds[k].cuda() for k in which])[0]


@pytest.mark.parametrize("name", ["IR_SE_50", "IR_101"])
def test_irnet_input_grad_batch_independent_and_deterministic(cuda, name):
    from oracle import resnet_oracle as RO
    net = _net(name, _state(name))
    x = RO.synthetic_faces(4, seed=4322)
    seeds = _seeds(4)
    full = _native_dx(net, x, seeds, CASES["all"])
    singles = [_native_dx(net, x[i:i + 1], [s[i:i + 1] for s in seeds], CASES["all"]) for i in range(4)]
    assert torch.equal(full, torch.cat(singles))
    with torch.no_grad():
        outs = net.forward_features(x.cuda())
        for i in range(4):
            one = net.forward_features(x[i:i + 1].cuda())
            assert all(torch.equal(a[i:i + 1], b) for a, b in zip(outs, one))
    # two full runs, and repeated backward calls on one forward
    assert torch.equal(full, _native_dx(net, x, seeds, CASES["all"]))
    xg = x.cuda().requires_grad_(True)
    outs = net.forward_features(xg)
    loss = sum((o * s.cuda()).sum() for o, s in zip(outs, seeds))
    loss.backward(retain_graph=True)
    g1 = xg.grad.clone()
    xg.grad = None
    loss.backward(retain_graph=True)
    assert torch.equal(g1, xg.grad) and torch.equal(g1, full)
    assert all(p.grad is None for p in net.parameters())


@pytest.mark.parametrize("name", ["IR_SE_50", "IR_152"])
def test_kd_step_irnet_teacher(cuda, name):
    """test_kd_step_hr_teacher_lr_student with an IR_SE_50 / IR_152 teacher: the native crfr_kd_train_step equals the same
    step composed from the drop-in modules, the loss modules and autograd."""
    from crfr_b200.loss import MSELoss, ResidualKDLoss
    from crfr_b200.model.resnet import kd_train_step
    from oracle import resnet_oracle as RO
    from tests.test_resnet_gpu import B, _nets
    (_, student, assistant), sds = _nets()
    teacher = _net(name, _state(name))
    student.train(); assistant.train()
    x_hr = RO.synthetic_faces(B).cuda()
    x_lr = RO.synthetic_faces(B, seed=999).cuda()
    with torch.no_grad():
        t_outs = teacher.forward_features(x_hr)
    s_outs, a_outs = student(x_lr), assistant(x_lr)
    mse, kd = MSELoss(), ResidualKDLoss()
    l_s = mse(s_outs[0], t_outs[0])
    l_a = sum(kd(t_outs[k], s_outs[k], a_outs[k]) for k in (1, 2, 3, 4)) + kd(t_outs[0], s_outs[0], a_outs[0])
    (l_s + l_a).backward()
    ref_s = [p.grad.clone() for p in student.parameters()]
    ref_a = [p.grad.clone() for p in assistant.parameters()]
    for net, sd in zip((student, assistant), sds[1:]):
        net.load_state_dict(sd)
        net.zero_grad(set_to_none=True)
    losses = kd_train_step(teacher, student, assistant, x_hr, x_lr=x_lr)
    torch.cuda.synchronize()
    assert abs(losses[0].item() - l_s.item()) < 1e-4 * abs(l_s.item())
    assert abs(losses[1].item() - l_a.item()) < 1e-4 * abs(l_a.item())
    names = [k for k, _ in student.named_parameters()]
    for tag, net, ref in (("s", student, ref_s), ("a", assistant, ref_a)):
        fo, fr = [], []
        for k, p, r in zip(names, net.parameters(), ref):
            if k in RO.RESNET_NULL_GRAD:
                continue
            assert rel_err(p.grad, r) < 6e-2, (tag, k, rel_err(p.grad, r))
            fo.append(p.grad.flatten().double()); fr.append(r.flatten().double())
        a, b = torch.cat(fo), torch.cat(fr)
        assert float(a @ b / (a.norm() * b.norm())) > 0.999, tag


def test_kd_trainer_irse50_teacher(cuda):
    """One KDTrainer step with an IR_SE_50 teacher gives the losses and gradients of kd_train_step."""
    from crfr_b200.model.resnet import kd_train_step
    from crfr_b200.trainer import KDTrainer
    from oracle import resnet_oracle as RO
    from tests.test_resnet_gpu import B, _nets
    x_hr, x_lr = RO.synthetic_faces(B).cuda(), RO.synthetic_faces(B, seed=5).cuda()
    (_, student, assistant), _ = _nets()
    teacher = _net("IR_SE_50", _state("IR_SE_50"))
    student.train(); assistant.train()
    ref_losses = kd_train_step(teacher, student, assistant, x_hr, x_lr=x_lr).clone()
    ref_g = [[p.grad.clone() for p in n.parameters()] for n in (student, assistant)]
    (_, student2, assistant2), _ = _nets()
    student2.train(); assistant2.train()
    tr = KDTrainer(teacher, student2, assistant2, lr=1e-4)
    losses = tr.step(x_hr, x_lr)
    torch.cuda.synchronize()
    assert torch.allclose(losses, ref_losses, rtol=1e-5)
    for f, r in zip((tr.S, tr.A), ref_g):
        for gv, g in zip(f.grad_views, r):
            assert rel_err(gv, g) < 1e-3
