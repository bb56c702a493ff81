"""Per-layer teacher-forced forward and per-unit backward parity of the IR / IR-SE teachers (crfr_irnet_*), as
tests/test_resnet_forced_gpu.py does for ResNet_34.

The end-to-end checks of tests/test_irnet_gpu.py compare five outputs and dx; with every stored tensor substituted, an early
layer or one unit's gradient can be a few percent wrong without moving them past their bf16-noise bounds.  Here every
comparison is one operation deep: each stored forward tensor (``crfr_irnet_tape``) is recomputed in float64 from the stored
tensors that feed it, and each stored gradient of the backward (``crfr_irnet_grad_tape``) from the native gradient one step
downstream.  Where the native kernel rounds to bf16 the reference rounds at the same points, so the remaining difference is
the order of fp32 sums.  Every bound is also checked to reject a reference with one known error planted (``_Report.mutant``): the SE shift
left out of dr, the last pixel of each reduction chunk dropped, e in place of e(1 - e), the hidden ReLU mask inverted, the
PReLU slope of channel c + 1 used for channel c, the odd pixel in the stride-2 gather, res_layer.0's folded scale left
out."""
import pytest
import torch
import torch.nn.functional as F
from torch.nn.grad import conv2d_input

from tests.irnet_oracle import build_irnet_state_dict, irnet_block_specs
from tests.test_ir50_grad_gpu import CASES, _seeds
from tests.test_irnet_gpu import _native_forced, _net
from tests.test_resnet_forced_gpu import LAYER_TOL
from tests.util import rel_err

pytestmark = pytest.mark.gpu

VARIANTS = {"IR_50": (50, 0), "IR_SE_50": (50, 1), "IR_101": (100, 0), "IR_SE_101": (100, 1), "IR_152": (152, 0),
            "IR_SE_152": (152, 1)}
# (variant, batch, images checked): batch 4 / 2, and IR_SE_50 at the benchmark's batch of 256, where the first two, the
# last two and one middle image cover the tile and persistent-grid edges that a small batch never reaches
SHAPES = [(n, 2 if v[0] == 152 else 4, None) for n, v in VARIANTS.items()] + [("IR_SE_50", 256, (0, 1, 127, 254, 255))]
# the upstream gradients of the backward checks: every output, the 7 x 7 stage output alone, the embedding alone
GRAD_CASES = {"all": (CASES["all"], 31), "x4": ((4,), 16), "emb": ((0,), 1)}

# Bounds, from the worst value over all variants, shapes and seeds measured on a B200 (in brackets) and the least error
# of a planted error that the bound must reject:
GRAD_TOL = 1e-3       # ||native - bf16(reference with the native roundings)|| / ||.|| of a gradient one dgrad deep
                      # [2.2e-4 (d_r2); mutants >= 0.10]
SHIFT_TOL = 1e-5      # the SE squeeze gradient shift[n][c] (fp32) against float64 [3.5e-7; mutants >= 3e-2]
TIE_FRAC = 2e-4       # element-wise passes: the fraction of elements more than one bf16 ulp away, where the fp32 sum
                      # cancels (s * y + t + res near 0) [3.0e-5]
EXCITE_TOL = 1e-5     # the fp32 excitation against float64 [1.3e-7]
BN_EPS = 1e-5


def _state(name):
    """The parameters of tests/test_irnet_gpu.py (seeded construction, random BatchNorms), with per-channel PReLU slopes:
    the constructors' uniform 0.25 would hide a channel index error of the PReLU passes.  The seed keeps every SE unit's
    squeeze path live on these images (some hidden unit of each has pre > 0): with many seeds a 4-wide hidden layer of
    stage 1 is dead for every image, its shift is exactly 0, and no error in that path could show."""
    from oracle import resnet_oracle as RO
    sd = RO.randomize_bn_everywhere(build_irnet_state_dict(91, *VARIANTS[name]), 191)
    g = torch.Generator().manual_seed(303)
    for k in sd:
        if k.endswith(("input_layer.2.weight", "res_layer.2.weight")):
            sd[k] = 0.05 + 0.4 * torch.rand(sd[k].shape, generator=g)
    return sd


def q(t):
    """bf16 rounding (of the fp32 value, as the native kernels round), back in float64."""
    return t.float().bfloat16().double()


def _ulps(native, ref):
    """|native - ref| in bf16 ulps of ref, element-wise."""
    a = ref.abs().clamp_min(2.0 ** -126)
    return (native - ref).abs() / torch.exp2(torch.floor(torch.log2(a)) - 7)


class _Run:
    """One native forward + backward in its workspace: stored tensors read back for the checked images, in float64 NCHW
    on the GPU."""

    def __init__(self, ws, idx):
        self.ws, self.idx = ws, idx

    def t(self, e, off=None):
        v = torch.as_strided(self.ws.view(torch.bfloat16), (e.n, e.h, e.w, e.c), (e.h * e.w * e.ld, e.w * e.ld, e.ld, 1),
                             (e.out_off if off is None else off) // 2)
        return v[self.idx].double().permute(0, 3, 1, 2)

    def f32(self, off, e):
        return self.ws[off:off + 4 * e.n * e.c].view(torch.float32).view(e.n, e.c)[self.idx].double()


def _program(tape, num_layers):
    """The forward tape grouped as the program records it: stem, units, head."""
    it = iter(tape)
    take = lambda *kinds: [next(it) for _ in kinds]
    stem = dict(zip(("conv", "bn"), take(0, 1)))
    units = []
    for cin, d, stride in irnet_block_specs(num_layers):
        u = dict(cin=cin, d=d, stride=stride)
        if cin != d:
            u["sc_conv"], u["sc_bn"] = take(0, 1)
        elif stride == 2:
            u["sub"], = take(9)
        u.update(zip(("bn0", "conv1", "prelu", "conv2", "bn4"), take(1, 0, 8, 0, 1)))
        units.append(u)
    head = dict(zip(("bn0", "lin", "bn1"), take(1, 7, 1)))
    assert next(it, None) is None
    kinds = [stem["conv"].kind, stem["bn"].kind, head["bn0"].kind, head["lin"].kind, head["bn1"].kind]
    assert kinds == [0, 1, 1, 7, 1], kinds
    for u in units:
        assert [u[k].kind for k in ("bn0", "conv1", "prelu", "conv2")] == [1, 0, 8, 0]
        assert u["bn4"].kind in (1, 10) and ("sub" not in u or u["sub"].kind == 9)
    return stem, units, head


def _grad_tape(num_layers, se, b, mask):
    from crfr_b200 import _lib as L
    n = L.lib().crfr_irnet_grad_tape(num_layers, se, b, 112, mask, None, 0)
    assert n > 0
    arr = (L.TapeEntry * n)()
    assert L.lib().crfr_irnet_grad_tape(num_layers, se, b, 112, mask, arr, n) == n
    return list(arr)


class _Params:
    """float64 (and fp32) views of the state on the GPU, and the BatchNorm scales as the native program forms them."""

    def __init__(self, sd):
        self.d = {k: v.cuda().double() for k, v in sd.items()}
        self.f = {k: v.cuda().float() for k, v in sd.items()}

    def affine(self, p):   # BN(y) = s * y + t, float64
        s = self.d[p + "weight"] / torch.sqrt(self.d[p + "running_var"] + BN_EPS)
        return s, self.d[p + "bias"] - self.d[p + "running_mean"] * s

    def scale32(self, p):  # gamma * rsqrt(var + eps) in fp32: the scale folded into a weight pack
        return self.f[p + "weight"] * torch.rsqrt(self.f[p + "running_var"] + BN_EPS)

    def fold(self, w, cout_scale=None, cin_scale=None):   # bf16(fp32(W) * s): the dgrad pack with a folded scale
        w = self.f[w]
        if cout_scale is not None:
            w = w * cout_scale.view(-1, *([1] * (w.dim() - 1)))
        if cin_scale is not None:
            w = w * cin_scale.view(1, -1, *([1] * (w.dim() - 2)))
        return q(w)


def _c(v):   # per-channel vector as [1, C, 1, 1]
    return v.view(1, -1, 1, 1)


class _Report:
    """Worst error per check, and the planted errors each check rejects or, wrongly, accepts."""

    def __init__(self, tag):
        self.tag, self.worst, self.fails, self.rejected = tag, {}, [], {}

    def err(self, check, value, bound, where):
        self.worst[check] = max(self.worst.get(check, (0.0, None)), (value, where), key=lambda t: t[0])
        if not value <= bound:
            self.fails.append((check, where, value, bound))

    def mutant(self, name, value, bound, where, required=True):
        ok = value > bound
        n_ok, n, least = self.rejected.get(name, (0, 0, float("inf")))
        self.rejected[name] = (n_ok + ok, n + 1, min(least, value if required else float("inf")))
        if required and not ok:
            self.fails.append(("mutant " + name, where, value, bound))

    def finish(self):
        for check, (v, where) in sorted(self.worst.items()):
            print("%s %-24s worst %.3e at %s" % (self.tag, check, v, where))
        for name, (n_ok, n, least) in sorted(self.rejected.items()):
            print("%s mutant %-24s rejected in %d of %d checks (least error where required %.3e)"
                  % (self.tag, name, n_ok, n, least))
        assert not self.fails, self.fails[:20]


def _check_forward(run, P, x, stem, units, head, rep):
    """Every stored forward tensor recomputed from the stored tensors that feed it."""
    def conv(e, inp, w, stride):
        k = P.d[w].shape[-1]
        ref = F.conv2d(inp, q(P.d[w]), None, stride, k // 2)
        rep.err("fwd conv", rel_err(run.t(e), q(ref)), LAYER_TOL, w)

    def elementwise(check, e, ref, where):
        u = _ulps(run.t(e).reshape(ref.shape), ref)
        rep.err(check + " >1ulp", (u > 1).double().mean().item(), TIE_FRAC, where)
        rep.err(check + " norm", rel_err(run.t(e).reshape(ref.shape), q(ref)), LAYER_TOL, where)

    def bn(e, inp, p, res=None, alpha=None):
        s, t = P.affine(p)
        shape = (1, -1) if inp.dim() == 2 else (1, -1, 1, 1)
        z = inp * s.view(shape) + t.view(shape)
        if alpha is not None:
            z = torch.where(z > 0, z, z * _c(P.d[alpha]))
        elementwise("fwd bn", e, z if res is None else z + res, p)

    conv(stem["conv"], q(x), "input_layer.0.weight", 1)
    bn(stem["bn"], run.t(stem["conv"]), "input_layer.1.", alpha="input_layer.2.weight")
    a_entry = stem["bn"]
    for i, u in enumerate(units):
        p = "body.%d." % i
        a = run.t(a_entry)
        assert u["bn0"].in_off == a_entry.out_off
        if "sc_conv" in u:
            conv(u["sc_conv"], a, p + "shortcut_layer.0.weight", u["stride"])
            bn(u["sc_bn"], run.t(u["sc_conv"]), p + "shortcut_layer.1.")
            res = run.t(u["sc_bn"])
        elif "sub" in u:
            sub = run.t(u["sub"])
            rep.err("fwd subsample", float(not torch.equal(sub, a[:, :, ::2, ::2])), 0, p)
            rep.mutant("odd pixel (fwd)", float(not torch.equal(sub, a[:, :, 1::2, 1::2])), 0, p)
            res = sub
        else:
            res = a
        bn(u["bn0"], a, p + "res_layer.0.")
        conv(u["conv1"], run.t(u["bn0"]), p + "res_layer.1.weight", 1)
        y1, alpha = run.t(u["conv1"]), _c(P.d[p + "res_layer.2.weight"])
        # PReLU pass: bit-exact (y * alpha is exact in float64; the native pass rounds it to fp32, then to bf16)
        ref = q(torch.where(y1 > 0, y1, y1 * alpha))
        rep.err("fwd prelu", float(not torch.equal(run.t(u["prelu"]), ref)), 0, p)
        rep.mutant("alpha c+1 (fwd)", float(not torch.equal(run.t(u["prelu"]), q(torch.where(
            y1 > 0, y1, y1 * torch.roll(alpha, -1, 1))))), 0, p)
        conv(u["conv2"], run.t(u["prelu"]), p + "res_layer.3.weight", u["stride"])
        y = run.t(u["conv2"])
        if u["bn4"].kind == 10:   # res + e * (s * y + t), one rounding; e from the stored y against float64 first
            e_nat = run.f32(u["bn4"].stats_off, u["bn4"])
            s, t = P.affine(p + "res_layer.4.")
            pooled = y.mean(dim=(2, 3)) * s + t
            e_ref = torch.sigmoid(torch.relu(pooled @ P.d[p + "res_layer.5.fc1.weight"].flatten(1).t())
                                  @ P.d[p + "res_layer.5.fc2.weight"].flatten(1).t())
            rep.err("fwd excitation", rel_err(e_nat, e_ref), EXCITE_TOL, p)
            elementwise("fwd se apply", u["bn4"], res + e_nat[:, :, None, None] * (y * _c(s) + _c(t)), p)
        else:
            bn(u["bn4"], y, p + "res_layer.4.", res=res)
        a_entry = u["bn4"]
    assert head["bn0"].in_off == a_entry.out_off
    bn(head["bn0"], run.t(a_entry), "output_layer.0.")
    o = run.t(head["bn0"]).reshape(len(run.idx), -1)
    ref = o @ q(P.d["output_layer.3.weight"]).t() + P.d["output_layer.3.bias"]
    rep.err("fwd linear", rel_err(run.t(head["lin"]).reshape(ref.shape), q(ref)), LAYER_TOL, "output_layer.3")
    bn(head["bn1"], run.t(head["lin"]).reshape(ref.shape), "output_layer.4.")


def _chunk_ends(hw):
    """The last pixel of each chunk of se_bwd_reduce_kernel (chunks of at most 256 pixels, split evenly)."""
    chunks = (hw + 255) // 256
    return [hw * (k + 1) // chunks - 1 for k in range(chunks)]


def _se_shift(P, p, y, g, e, mutate=None):
    """The part of dr that every pixel of an (image, channel) shares: (1/hw) W1^T(relu'(pre) * W2^T(e(1-e) * sum g r))
    with r = s y + t, pre = W1 (s mean(y) + t) from the stored y; float64."""
    s, t = P.affine(p + "res_layer.4.")
    w1 = P.d[p + "res_layer.5.fc1.weight"].flatten(1)   # [Hd, C]
    w2 = P.d[p + "res_layer.5.fc2.weight"].flatten(1)   # [C, Hd]
    hw = y.shape[2] * y.shape[3]
    gr = (g * (y * _c(s) + _c(t))).flatten(2)
    if mutate == "chunk":
        keep = torch.ones(hw, dtype=torch.bool, device=y.device)
        keep[_chunk_ends(hw)] = False
        gr = gr[:, :, keep]
    de = gr.sum(2)
    pre = (y.mean(dim=(2, 3)) * s + t) @ w1.t()
    u = de * (e if mutate == "e" else e * (1 - e))
    mask = (pre <= 0) if mutate == "relu" else (pre > 0)
    return ((u @ w2) * mask) @ w1 / hw


def _check_backward(run, P, x, seeds, dx, stem, units, head, gtape, mask, rep):
    """Every stored gradient of the IR backward from the native gradient one step downstream."""
    by = {(e.kind, e.w_idx): e for e in gtape}
    assert len(by) == len(gtape)
    if mask & 1:   # head: da = s_o0 * W^T (s_emb * d_emb), the scales folded into the bf16 pack
        e = by[(11, -1)]
        assert e.in_off == head["bn0"].in_off
        de = q(seeds[0][list(run.idx)].cuda().double())
        w = P.f["output_layer.3.weight"].view(512, 512, 49) * P.scale32("output_layer.4.").view(-1, 1, 1)
        w = q(w * P.scale32("output_layer.0.").view(1, -1, 1))
        ref = (de @ w.view(512, -1)).view(-1, 512, 7, 7)
        rep.err("bwd head da", rel_err(run.t(e), q(ref)), GRAD_TOL, "output_layer")
    for i in reversed(range(len(units))):
        u, p = units[i], "body.%d." % i
        if (12, i) not in by:
            continue
        eg, ed2, ein = by[(12, i)], by[(14, i)], by[(15, i)]
        assert eg.in_off == u["bn4"].out_off and ed2.in_off == u["conv1"].out_off and ein.in_off == u["bn0"].in_off
        g = run.t(eg)
        dz = g
        if u["bn4"].kind == 10:   # res_layer.5: the squeeze gradient, then dr = e * g + shift
            edr = by[(13, i)]
            assert edr.in_off == u["conv2"].out_off
            y, e_nat = run.t(u["conv2"]), run.f32(u["bn4"].stats_off, u["bn4"])
            shift = run.f32(edr.stats_off, edr)
            ref = _se_shift(P, p, y, g, e_nat)
            rep.err("bwd se shift", rel_err(shift, ref), SHIFT_TOL, p)
            for m in ("e", "relu"):
                rep.mutant("se " + m, rel_err(shift, _se_shift(P, p, y, g, e_nat, m)), SHIFT_TOL, p)
            hw = y.shape[2] * y.shape[3]
            rep.mutant("se chunk end", rel_err(shift, _se_shift(P, p, y, g, e_nat, "chunk")), SHIFT_TOL, p,
                       required=hw == 56 * 56)
            dz = run.t(edr)
            ref = e_nat[:, :, None, None] * g + shift[:, :, None, None]
            rep.err("bwd se dr ulps", _ulps(dz, ref).max().item(), 1, p)
            rep.mutant("se no shift", _ulps(dz, e_nat[:, :, None, None] * g).max().item(), 1, p)
        # res_layer.4 + .3: conv2's dgrad with res_layer.4's scale folded over its output channels, then the PReLU mask
        y1 = run.t(u["conv1"])
        w2 = P.fold(p + "res_layer.3.weight", cout_scale=P.scale32(p + "res_layer.4."))
        d = q(conv2d_input(y1.shape, w2, dz, u["stride"], 1))
        alpha = _c(P.d[p + "res_layer.2.weight"])
        d_r2 = run.t(ed2)
        rep.err("bwd d_r2", rel_err(d_r2, q(torch.where(y1 > 0, d, d * alpha))), GRAD_TOL, p)
        rep.mutant("alpha c+1", rel_err(d_r2, q(torch.where(y1 > 0, d, d * torch.roll(alpha, -1, 1)))), GRAD_TOL, p)
        # res_layer.1 + .0: conv1's dgrad with res_layer.0's scale folded over its input channels, plus the shortcut
        shape = run.t(u["bn0"]).shape   # the unit input's
        w1 = P.fold(p + "res_layer.1.weight", cin_scale=P.scale32(p + "res_layer.0."))
        d1 = q(conv2d_input(shape, w1, d_r2, 1, 1))
        if "sc_conv" in u:
            wsc = P.fold(p + "shortcut_layer.0.weight", cout_scale=P.scale32(p + "shortcut_layer.1."))
            sc = q(conv2d_input(shape, wsc, g, u["stride"], 0))
        elif "sub" in u:
            sc = torch.zeros(shape, dtype=g.dtype, device=g.device)
            sc[:, :, ::2, ::2] = g
            odd = torch.zeros_like(sc)
            odd[:, :, 1::2, 1::2] = g
        else:
            sc = g
        d_in = run.t(ein)
        rep.err("bwd d_in", rel_err(d_in, q(d1 + sc)), GRAD_TOL, p)
        d1_no_s0 = q(conv2d_input(shape, P.fold(p + "res_layer.1.weight"), d_r2, 1, 1))
        rep.mutant("no s0 fold", rel_err(d_in, q(d1_no_s0 + sc)), GRAD_TOL, p)
        if "sub" in u:
            rep.mutant("odd pixel", rel_err(d_in, q(d1 + odd)), GRAD_TOL, p)
    # stem: BatchNorm + PReLU element-wise on the gradient of the stem's output (unit 0's d_in), then conv's dgrad
    e0 = by[(16, -1)]
    assert e0.in_off == stem["conv"].out_off
    g0, y0 = run.t(by[(15, 0)]), run.t(stem["conv"])
    s, t = P.affine("input_layer.1.")
    z = y0 * _c(s) + _c(t)
    dy0 = run.t(e0)
    alpha = _c(P.d["input_layer.2.weight"])
    rep.err("bwd stem dy0", rel_err(dy0, q(g0 * _c(s) * torch.where(z > 0, 1.0, alpha))), GRAD_TOL, "input_layer")
    rep.mutant("alpha c+1 (stem)", rel_err(dy0, q(g0 * _c(s) * torch.where(z > 0, 1.0, torch.roll(alpha, -1, 1)))),
               GRAD_TOL, "input_layer")
    ref = conv2d_input((dy0.shape[0], 3, 112, 112), q(P.d["input_layer.0.weight"]), dy0, 1, 1)
    rep.err("bwd stem dx", rel_err(dx[list(run.idx)].cuda().double(), q(ref)), GRAD_TOL, "input_layer.0")


@pytest.mark.parametrize("name,batch,images", SHAPES, ids=["%s-%d" % s[:2] for s in SHAPES])
def test_irnet_forced_layers(cuda, name, batch, images):
    """Forward: every stored tensor against float64 on the stored inputs - convolutions and the linear head norm-wise
    (LAYER_TOL), BatchNorm and the SE output within one bf16 ulp but for a counted fraction, the PReLU pass and the
    subsampling bit-exact, the excitation at fp32 level.  Backward, for seeds on every output, on x4 alone and on the
    embedding alone: per unit g -> (SE: shift and dr) -> d_r2 -> d_in, the head and the stem, each from the native
    gradient one step downstream."""
    from oracle import resnet_oracle as RO
    num_layers, se = VARIANTS[name]
    sd = _state(name)
    net = _net(name, sd)
    P = _Params(sd)
    x = RO.synthetic_faces(batch, seed=4322)
    seeds = _seeds(batch)
    idx = tuple(images) if images else tuple(range(batch))
    xi = x[list(idx)].cuda().double()
    rep = _Report("%s b%d" % (name, batch))
    for c, (ks, mask) in GRAD_CASES.items():
        dxs, tape, ws, _ = _native_forced(name, net, x, seeds, {c: ks})
        stem, units, head = _program(tape, num_layers)
        run = _Run(ws, list(idx))
        if c == "all":
            _check_forward(run, P, xi, stem, units, head, rep)
        gtape = _grad_tape(num_layers, se, batch, mask)
        _check_backward(run, P, xi, seeds, dxs[c], stem, units, head, gtape, mask, rep)
        del ws
    rep.finish()
