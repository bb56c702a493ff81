"""Teacher-forced, one-operation-deep parity of the FSRNet identity step (crfr_fsrnet_id_train_step), from the two crops
to the decoder's output gradient.

tests/test_fsrnet_identity_gpu.py checks the step end to end (parameter gradients within 6e-2 of autograd, the identity
contribution within 3e-2 at a weight where it dominates).  Here the glue between the three programs is checked on its
own, through the step's tape (crfr_fsrnet_id_tape): the crops each teacher program reads, both teacher forwards, the
feature terms and losses[5] / losses[0], the bf16 seed slots, the stage-end sums of the teacher backward, its input
gradient dx4, the output-image gradient d_out4 it joins, conv_out.bias, and every FSRNet parameter gradient against the
forced oracle with dx4 as an added output gradient.  Each bound is shown to reject a planted error (``_Report.mutant``):
crop windows one pixel off, id_scale inside losses[5], a term left out, gscale without id_scale, unselected terms
seeded, the stage-end seed dropped or doubled, the window one pixel off, the pixel term dropped inside the window, the
window sums left out of the bias, and the gradient G placed at (7, 8)."""
import ctypes as C
import time

import pytest
import torch

from tests.test_fsrnet_forced_gpu import CANCELLING, EXACT_SLACK, REASSOC_TOL_DEEP, _tol
from tests.test_fsrnet_identity_gpu import W_BIG
from tests.test_irnet_forced_gpu import (TIE_FRAC, _check_backward, _check_forward, _Params, _program, _Report, _Run,
                                         _stage_ends, _state, _ulps)
from tests.test_irnet_forced_gpu import VARIANTS as IR_VARIANTS
from tests.util import rel_err

S, CROP, SIZE = 128, 8, 112
ALL = ("A", "B", "C", "D", "E", "F", "G", "H", "I", "J")
# (teacher, batch, w_id, id_scale, global batch, terms, checks, images of C / F / G (None: all))
CONFIGS = {
    "IR_50-w1": ("IR_50", 2, 1.0, 1.0, 2, (31,), ALL, None),
    "IR_50-wbig": ("IR_50", 2, W_BIG["IR_50"], 1.0, 2, (31,), ALL, None),
    "IR_SE_50-w1": ("IR_SE_50", 2, 1.0, 1.0, 2, (31,), ALL, None),
    "IR_SE_50-wbig": ("IR_SE_50", 2, W_BIG["IR_SE_50"], 1.0, 2, (31,), ALL, None),
    "IR_50-chunk": ("IR_50", 2, W_BIG["IR_50"], 0.5, 4, (31,), "ABDEHI", None),
    "IR_152-terms": ("IR_152", 2, 1.0, 1.0, 2, (1, 16, 0b01010), "AEFG", None),
    "IR_SE_50-terms": ("IR_SE_50", 2, 1.0, 1.0, 2, (1, 16, 0b01010), "AEFG", None),
    # the benchmark's shape: C, F and G on the first two, the last two and one middle image; J is the plain step's
    "IR_50-b128": ("IR_50", 128, W_BIG["IR_50"], 1.0, 128, (31,), "ABCDEFGHI", (0, 1, 63, 126, 127)),
}
LOSS_TOL = 1e-6     # losses[5], losses[0] against float64 on the stored features
WINDOW_FRAC = 1e-6  # d_out4 inside the window: the fraction of elements off the float64 reference's rounding
BIAS_TOL = 1e-5     # conv_out.bias against float64, relative to the sum of the magnitudes of its terms


def _tape(layers, se, b, terms):
    from crfr_b200 import _lib as L
    fn = L.lib().crfr_fsrnet_id_tape
    n = fn(layers, se, b, S, terms, None, 0)
    assert n > 0, n
    arr = (L.TapeEntry * n)()
    assert fn(layers, se, b, S, terms, arr, n) == n
    return list(arr)


def _plain_tape(fn, *args):
    n = fn(*args, None, 0)
    assert n > 0
    from crfr_b200 import _lib as L
    arr = (L.TapeEntry * n)()
    assert fn(*args, arr, n) == n
    return list(arr)


FIELDS = ("kind", "n", "h", "w", "c", "ld", "out_off", "in_off", "stats_off", "w_idx", "has_res")


def _shifted(e, base):
    d = {f: getattr(e, f) for f in FIELDS}
    for f in ("out_off", "in_off", "stats_off"):
        if d[f] >= 0:
            d[f] += base
    return d


def _round4096(n):
    return (n + 4095) & ~4095


class _Sections:
    """The id tape split into its seven sections, checked against the existing tapes (check A)."""

    def __init__(self, layers, se, b, terms):
        from crfr_b200 import _lib as L
        lib = L.lib()
        t = _tape(layers, se, b, terms)
        fsr = _plain_tape(lib.crfr_fsrnet_tape, b, S, 1)
        ir = _plain_tape(lib.crfr_irnet_tape, layers, se, b, SIZE)
        self.base_h = _round4096(lib.crfr_fsrnet_workspace_bytes(b, S, 1))
        self.base_s = self.base_h + _round4096(lib.crfr_irnet_workspace_bytes(layers, se, b, SIZE))
        self.ws_bytes = lib.crfr_fsrnet_id_workspace_bytes(layers, se, b, S)
        i = 0
        self.fsr = t[i:i + len(fsr)]
        i += len(fsr)
        self.d_out4 = t[i]
        i += 1
        self.hr = t[i:i + len(ir)]
        self.sr = t[i + len(ir):i + 2 * len(ir)]
        i += 2 * len(ir)
        self.seeds = []
        while t[i].kind == 17:
            self.seeds.append(t[i])
            i += 1
        self.grads = t[i:-1]
        self.dx4 = t[-1]
        self.fsr_ref, self.ir_ref, self.layers, self.terms, self.b = fsr, ir, layers, terms, b

    def check(self):
        """Sections 1, 3 and 4 are the existing tapes shifted; 2 and 5-7 lie inside the workspace and overlap neither a
        stored forward tensor nor each other, except that a unit's summed output gradient (kind 12) is the buffer of its
        only incoming gradient (kind 15 of the next unit, the head's kind 11 or a kind-17 seed)."""
        b = self.b
        assert [_shifted(e, 0) for e in self.fsr] == [_shifted(e, 0) for e in self.fsr_ref]
        assert [_shifted(e, 0) for e in self.hr] == [_shifted(e, self.base_h) for e in self.ir_ref]
        assert [_shifted(e, 0) for e in self.sr] == [_shifted(e, self.base_s) for e in self.ir_ref]
        d = self.d_out4
        assert (d.kind, d.n, d.h, d.w, d.c, d.ld) == (19, b, S, S, 3, 4)
        stem, units, head = _program(self.sr, self.layers)
        outs = [head["bn1"]] + [units[i]["bn4"] for i in _ends(units)]
        assert [e.w_idx for e in self.seeds] == [k for k in range(5) if self.terms >> k & 1]
        for e in self.seeds:
            o = outs[e.w_idx]
            assert e.in_off == o.out_off and (e.n, e.h, e.w, e.c, e.ld) == (o.n, o.h, o.w, o.c, o.ld)
        assert self.grads and all(11 <= e.kind <= 16 for e in self.grads)
        x = self.dx4
        assert (x.kind, x.n, x.h, x.w, x.c, x.ld, x.in_off) == (18, b, SIZE, SIZE, 3, 4, stem["conv"].in_off)

        def region(e):
            return e.out_off, e.out_off + 2 * e.n * e.h * e.w * e.ld
        stored = [region(e) for e in self.fsr + self.hr + self.sr if e.out_off >= 0]
        new = [region(e) for e in [self.d_out4] + self.seeds + self.grads + [self.dx4]]
        new += [(e.stats_off, e.stats_off + 4 * e.n * e.c) for e in self.grads if e.kind == 13]
        for lo, hi in new:
            assert 0 <= lo < hi <= self.ws_bytes, (lo, hi, self.ws_bytes)
        shared = {region(e) for e in self.grads if e.kind in (11, 15)} | {region(e) for e in self.seeds}
        own = [region(e) for e in [self.d_out4] + self.seeds + self.grads + [self.dx4]
               if not (e.kind == 12 and region(e) in shared)]
        own = sorted(own + [(e.stats_off, e.stats_off + 4 * e.n * e.c) for e in self.grads if e.kind == 13])
        for (_, hi), (lo, _) in zip(own, own[1:]):
            assert hi <= lo, "two gradient regions overlap"
        s_lo = torch.tensor([r[0] for r in stored], dtype=torch.int64)
        s_hi = torch.tensor([r[1] for r in stored], dtype=torch.int64)
        for lo, hi in own:
            assert not bool(((s_lo < hi) & (lo < s_hi)).any()), ("overlaps a stored forward tensor", lo, hi)
        return stem, units, head


def _ends(units):   # each stage's last unit, in stage order
    return sorted(_stage_ends(units))


@pytest.mark.parametrize("cfg", sorted(CONFIGS))
def test_id_tape_sections(cfg):
    """Check A without a device: the tape is a dry run."""
    name, b, _, _, _, terms_list, checks, _ = CONFIGS[cfg]
    for terms in terms_list:
        _Sections(*IR_VARIANTS[name], b, terms).check()


def test_id_tape_rejections():
    from crfr_b200 import _lib as L
    fn = L.lib().crfr_fsrnet_id_tape
    assert fn(50, 0, 2, S, 0, None, 0) == -1 and fn(50, 0, 2, S, 32, None, 0) == -1
    assert fn(50, 0, 2, 64, 31, None, 0) == -1 and fn(34, 0, 2, S, 31, None, 0) == -1 and fn(50, 2, 2, S, 31, None, 0) == -1


def _bf16_eq(a, b):
    return torch.equal(a.view(torch.int16), b.view(torch.int16))


class _Step:
    """One crfr_fsrnet_id_train_step, called directly, on a fresh workspace and zeroed gradients."""

    def __init__(self, teacher, batch, w_id, id_scale, loss_div, terms):
        from crfr_b200 import _lib as L
        from crfr_b200 import ops
        from crfr_b200.model import FSRnet as M
        from crfr_b200.trainer import FSRNetTrainer
        from oracle import forced_check as FC
        self.x, self.hr, self.hm, self.lbl = batch
        self.w_id, self.id_scale, self.loss_div, self.terms = w_id, id_scale, loss_div, terms
        self.net = FC.make_net()
        tr = FSRNetTrainer(self.net, lr=0.0, chunk=self.x.shape[0], identity_net=teacher)
        layers, se = teacher._variant
        b = self.x.shape[0]
        self.ws = torch.zeros(L.lib().crfr_fsrnet_id_workspace_bytes(layers, se, b, S), dtype=torch.uint8, device="cuda")
        self.outs = M.alloc_outputs(self.x)
        io = M._io(self.x, self.outs, (self.hr, self.hm, self.lbl), loss_div=loss_div, w_pix=5.0)
        ptab, btab, _ = tr._id_tabs
        idio = L.FsrnetIdIO(layers, se, C.cast(ptab.arr, C.c_void_p), C.cast(btab.arr, C.c_void_p), w_id, terms, id_scale)
        self.losses = torch.zeros(6, device="cuda")
        tr.flat_g.zero_()
        torch.cuda.synchronize()
        n0 = L.lib().crfr_launch_count()
        t0 = time.perf_counter()
        L.call("crfr_fsrnet_id_train_step", L.ENGINE_AUTO, tr.ptable.arr, tr.gtable.arr, C.byref(io), C.byref(idio),
               self.losses.data_ptr(), self.ws.data_ptr(), self.ws.numel(), ops.stream())
        torch.cuda.synchronize()
        self.seconds, self.launches = time.perf_counter() - t0, L.lib().crfr_launch_count() - n0
        self.grads = {k: g for (k, _), g in zip(self.net.named_parameters(), tr.grad_views)}
        self.tr = tr

    def nhwc4(self, e):
        """The bf16 NHWC tensor of a 3-channel entry with its padding channel: [n, h, w, 4] on the device."""
        return torch.as_strided(self.ws.view(torch.bfloat16), (e.n, e.h, e.w, 4), (e.h * e.w * 4, e.w * 4, 4, 1),
                                e.out_off // 2)


def _nchw3(v):   # [n, h, w, 4] bf16 -> [n, 3, h, w] float64
    return v[..., :3].double().permute(0, 3, 1, 2)


def _crop(t, y=CROP, x=CROP):
    return t[:, :, y:y + SIZE, x:x + SIZE]


def _check_crop(st, sec, rep):
    """B: each program's stem input is the window of the fp32 image read in place, rounded to bf16; channel 3 zero."""
    for tag, src, tape in (("hr", st.hr, sec.hr), ("sr", st.outs[1], sec.sr)):
        e = tape[0]
        x4 = torch.as_strided(st.ws.view(torch.bfloat16), (e.n, SIZE, SIZE, 4),
                              (SIZE * SIZE * 4, SIZE * 4, 4, 1), e.in_off // 2)

        def ref(y, x):
            r = torch.zeros_like(x4)
            r[..., :3] = _crop(src, y, x).permute(0, 2, 3, 1).bfloat16()
            return r
        rep.err("B crop", float(not _bf16_eq(x4, ref(CROP, CROP))), 0, tag)
        rep.mutant("B window (7, 8)", float(not _bf16_eq(x4, ref(CROP - 1, CROP))), 0, tag)
        rep.mutant("B window (8, 7)", float(not _bf16_eq(x4, ref(CROP, CROP - 1))), 0, tag)


def _features(run, units, head):
    """The five stored outputs (embedding, x1..x4) of a teacher program, float64 NCHW, all images."""
    return [run.t(head["bn1"])] + [run.t(units[i]["bn4"]) for i in _ends(units)]


def _check_losses(st, f_sr, f_hr, rep):
    """D: losses[5] = w_id sum_k mean((s_k - h_k)^2) over the stored features, losses[0] = the FSRNet share + id_scale
    losses[5]; float64."""
    ks = [k for k in range(5) if st.terms >> k & 1]
    mse = {k: ((f_sr[k] - f_hr[k]) ** 2).mean().item() for k in ks}
    l = st.losses.double().cpu()
    ref5 = st.w_id * sum(mse.values())
    fsr = (5.0 * l[1] + 5.0 * l[2] + l[3] + l[4]).item() / st.loss_div
    rep.err("D losses[5]", abs(l[5].item() - ref5) / ref5, LOSS_TOL, "")
    rep.err("D losses[0]", abs(l[0].item() - (fsr + st.id_scale * ref5)) / abs(fsr + st.id_scale * ref5), LOSS_TOL, "")
    rep.mutant("D id_scale in losses[5]", abs(l[5].item() - st.id_scale * ref5) / ref5, LOSS_TOL, "",
               required=st.id_scale != 1.0)
    for k in ks:
        rep.mutant("D term left out", abs(l[5].item() - (ref5 - st.w_id * mse[k])) / ref5, LOSS_TOL, "k=%d" % k)


def _gcoef_id(st, numel, id_scale=None):
    """crfr_loss_kd's fp32 gradient coefficient for gscale = fp32(w_id * id_scale)."""
    f = lambda v: torch.tensor(v, dtype=torch.float32)
    gscale = f(st.w_id) * f(st.id_scale if id_scale is None else id_scale)
    return f(gscale.item() * 2.0 / numel)


def _check_seeds(st, sec, run_all, units, head, hr_units, hr_head, rep):
    """E: every seed slot is bf16(fp32(gscale 2 / numel) * fp32(s - h)), as kd_kernel computes it; exactly the selected
    terms are seeded."""
    got = [e.w_idx for e in sec.seeds]
    ks = [k for k in range(5) if st.terms >> k & 1]
    rep.err("E seeded terms", float(got != ks), 0, "")
    rep.mutant("E unselected terms seeded", float(got != list(range(5))), 0, "", required=st.terms != 31)
    s_out = [head["bn1"]] + [units[i]["bn4"] for i in _ends(units)]
    h_out = [hr_head["bn1"]] + [hr_units[i]["bn4"] for i in _ends(hr_units)]
    for e in sec.seeds:
        k = e.w_idx
        s, h = run_all.t(s_out[k]).float(), run_all.t(h_out[k]).float()
        numel = s.numel()
        slot = run_all.t(e).float()
        ref = lambda g: (g.cuda() * (s - h)).bfloat16().float()
        rep.err("E seed bits", float(not torch.equal(slot, ref(_gcoef_id(st, numel)))), 0, "k=%d" % k)
        rep.mutant("E gscale without id_scale", float(not torch.equal(slot, ref(_gcoef_id(st, numel, 1.0)))), 0,
                   "k=%d" % k, required=st.id_scale != 1.0)


def _gcoef_pix(st, numel):
    """crfr_loss_mse97_chan's fp32 coefficient: gscale = fp32(w_pix * fp32(1 / loss_div))."""
    f = lambda v: torch.tensor(v, dtype=torch.float32)
    gscale = f(5.0) * (f(1.0) / f(st.loss_div))
    return f(gscale.item() * 2.0 * 97.0 / numel).item()


def _check_out_grad(st, sec, dx4, rep):
    """H: d_out4 outside the window is the plain step's bf16(gcoef (out - hr)); inside, float64 gcoef (out - hr) + dx4
    rounded to fp32, then bf16.  I: conv_out.bias = gcoef sum(out - hr) + the window sums of dx4, float64."""
    got = _nchw3(st.nhwc4(sec.d_out4))
    pad = st.nhwc4(sec.d_out4)[..., 3]
    d = (st.outs[1] - st.hr)                       # fp32, as the kernels form it
    gc = _gcoef_pix(st, d.numel())
    plain = (torch.tensor(gc, dtype=torch.float32, device="cuda") * d).bfloat16().double()
    g = dx4

    def full(y, x, pixel=True):
        r = plain.clone()
        r[:, :, y:y + SIZE, x:x + SIZE] = ((gc * _crop(d, y, x).double() if pixel else 0) + g).float().bfloat16().double()
        return r
    inside = torch.zeros_like(got, dtype=torch.bool)
    inside[:, :, CROP:CROP + SIZE, CROP:CROP + SIZE] = True
    ref = full(CROP, CROP)
    rep.err("H outside differ", float((got != ref)[~inside].sum().item()) + float(pad.abs().max().item()), 0, "")
    rep.err("H inside max ulps", _ulps(got[inside], ref[inside]).max().item(), 1, "")
    rep.err("H inside differ frac", (got != ref)[inside].double().mean().item(), WINDOW_FRAC, "")
    frac = lambda r: (got != r).double().mean().item()
    # a planted error is required to be rejected where it moves the reference past the bound: at w_id = 1 dx4 vanishes in
    # the rounding of d_out4, and at W_BIG with a larger loss_div the pixel term does inside the window
    for name, r in (("H window (8, 9)", full(CROP, CROP + 1)), ("H pixel term dropped", full(CROP, CROP, pixel=False))):
        moved = (r != ref).double().mean().item()
        rep.mutant(name, frac(r), WINDOW_FRAC, "", required=moved > WINDOW_FRAC)
    # I
    bias = st.grads["_fine_sr_decoder.conv_out.bias"].double()
    pix, win = gc * d.double().sum(dim=(0, 2, 3)), g.sum(dim=(0, 2, 3))
    scale = (gc * d.double().abs().sum(dim=(0, 2, 3)) + g.abs().sum(dim=(0, 2, 3)))
    rep.err("I conv_out.bias", ((bias - (pix + win)).abs() / scale).max().item(), BIAS_TOL, "")
    rep.mutant("I window sums left out", ((bias - pix).abs() / scale).max().item(), BIAS_TOL, "",
               required=(win.abs() / scale).max().item() > BIAS_TOL)


def _check_fsrnet_grads(st, sec, dx4, rep):
    """J: every FSRNet parameter gradient against the forced oracle on the stored FSRNet tensors, with the loss plus
    sum(out * G), G the zero-padded dx4: within the bounds of tests/test_fsrnet_forced_gpu.py against the bf16 oracle
    and against the exact backward.  Against the bf16 oracle the deep half takes that file's bound for two bf16
    evaluations of the same backward (REASSOC_TOL_DEEP, 2.5e-2) rather than GRAD_TOL_DEEP (2e-2): at W_BIG, where dx4
    drives the step, the two land 2.36e-2 (IR_50) and 2.27e-2 (IR_SE_50) apart on PReLU slopes and InstanceNorm biases of
    the coarse network (one B200), while the native gradient stays within 1.4 x the oracle's own distance from the exact
    backward there; the planted G at (7, 8) is rejected by the bound of every parameter it moves past it."""
    from oracle import forced_check as FC
    from oracle import fsrnet_oracle as FO
    sd = FO.build_fsrnet_state_dict(1234)
    x, hr, hm, lbl = (t.cpu() for t in (st.x, st.hr, st.hm, st.lbl))

    def oracle(cls, y=CROP, xo=CROP):
        G = torch.zeros_like(x)
        G[:, :, y:y + SIZE, xo:xo + SIZE] = dx4.float().cpu()
        return FO.fsrnet_loss_and_grads(sd, x, hr, hm, lbl, precision=cls(FC.forced_feed(st.ws, sec.fsr)),
                                        out_grad=G)[3]
    gd, gx, gm = oracle(FO.ForcedPrecision), oracle(FO.ForcedExact), oracle(FO.ForcedPrecision, CROP - 1, CROP)
    gnorm = torch.sqrt(sum((g.double() ** 2).sum() for g in gd.values() if g is not None)).item()
    for k, g in st.grads.items():
        if FO.fsrnet_dead_param(k):
            continue
        if k in FO.FSRNET_NULL_GRAD:
            rep.err("J null gradient", g.double().norm().item() / gnorm, 1e-3, k)
            continue
        tol = _tol(k, REASSOC_TOL_DEEP)
        rep.err("J bf16 oracle" + (" (cancelling)" if k in CANCELLING else ""), rel_err(g, gd[k]), tol, k)
        if k not in CANCELLING:
            e_exact, o_exact = rel_err(g, gx[k]), rel_err(gd[k], gx[k])
            rep.err("J exact (bound 1.4 oracle's + 2e-3)", e_exact, EXACT_SLACK * o_exact + 2e-3, k)
        # required where the shift moves the oracle's gradient past the bound: not for conv_out.bias (the plain sum of G
        # wherever it lies) nor the prior network's two heads (only the landmark and parsing losses reach them)
        rep.mutant("J G at (7, 8)", rel_err(g, gm[k]), tol, k, required=rel_err(gm[k], gd[k]) > tol)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", sorted(CONFIGS))
def test_identity_step_forced(cuda, cfg):
    """Checks A - J of the module docstring on one configuration; prints the worst value of each check and, per planted
    error, in how many checks it was rejected."""
    from crfr_b200.trainer import chunk_loss_div
    from oracle import fsrnet_oracle as FO
    from tests.test_irnet_gpu import _net
    name, b, w_id, id_scale, global_b, terms_list, checks, images = CONFIGS[cfg]
    layers, se = IR_VARIANTS[name]
    sd = _state(name)
    teacher = _net(name, sd)
    P = _Params(sd)
    x, hr, lbl, hm = FO.synthetic_batch(b, S, seed=8)
    batch = (x.cuda(), hr.cuda(), hm.cuda(), lbl.cuda().contiguous())
    idx = list(images) if images else list(range(b))
    rep = _Report(cfg)
    big = w_id != 1.0
    for terms in terms_list:
        t0 = time.perf_counter()
        st = _Step(teacher, batch, w_id, id_scale, chunk_loss_div(global_b, b), terms)
        sec = _Sections(layers, se, b, terms)
        stem, units, head = sec.check()                                            # A
        hstem, hunits, hhead = _program(sec.hr, layers)
        run, run_all = _Run(st.ws, idx), _Run(st.ws, list(range(b)))   # both programs' arenas are in st.ws
        dx4 = _nchw3(st.nhwc4(sec.dx4))
        if "B" in checks:
            _check_crop(st, sec, rep)
        if "C" in checks:
            _check_forward(run, P, _crop(st.hr)[idx].double(), hstem, hunits, hhead, rep)
            _check_forward(run, P, _crop(st.outs[1])[idx].double(), stem, units, head, rep)
        if "D" in checks:
            _check_losses(st, _features(run_all, units, head), _features(run_all, hunits, hhead), rep)
        if "E" in checks:
            _check_seeds(st, sec, run_all, units, head, hunits, hhead, rep)
        if "F" in checks or "G" in checks:   # F is the stage-end part of _check_backward
            seeds = [None] * 5
            for e in sec.seeds:
                v = run_all.t(e)
                seeds[e.w_idx] = v.reshape(b, -1) if e.w_idx == 0 else v
            _check_backward(run, P, None, seeds, dx4, stem, units, head, sec.grads, terms, rep)
        if "H" in checks:
            _check_out_grad(st, sec, dx4, rep)
        if "J" in checks and big:
            _check_fsrnet_grads(st, sec, dx4, rep)
        print("%s terms %d: step %.1f ms (first call), %d launches; checks %.1f s"
              % (cfg, terms, 1e3 * st.seconds, st.launches, time.perf_counter() - t0))
        del st
        torch.cuda.empty_cache()
    rep.finish()
