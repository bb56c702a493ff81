"""FSRNet training step with an identity loss through a frozen IR / IR-SE teacher (crfr_fsrnet_id_train_step through
FSRNetTrainer(identity_net=...)): parity with autograd through the drop-in modules, the identity contribution on its own
(against planted errors), the losses, no interference with the plain step at w_id = 0, determinism, graph replay,
chunking, the untouched teacher and the rejections."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from tests.util import rel_err

pytestmark = pytest.mark.gpu

B, CHUNK, S = 4, 2, 128
TERMS = (0, 1, 2, 3, 4)
# On these synthetic batches the FSRNet losses (~5e4, landmark term ~4e5) dwarf the identity term (~170 at w_id = 1): its
# gradient then sits below the bf16 rounding noise of the FSRNet backward, and grad(with) - grad(without) is noise on
# either path.  The contribution is therefore checked at a weight where it dominates the step's gradient (~30x the plain
# gradient for both teachers; the seeded IR_SE_50's features move ~300x less than IR_50's).  Measured on one B200: native
# against module path 1.43e-2 (IR_50) and 1.35e-2 (IR_SE_50); the planted errors land at 9.3e-2 (w_id off by 10 %) and
# 1.17 - 1.38 (crop at (7, 8)).
W_BIG = {"IR_50": 1e4, "IR_SE_50": 3e6}
CONTRIB_BOUND = 3e-2


def _fsr():
    from crfr_b200.model.FSRnet import OverallNetwork, weights_init
    torch.manual_seed(1234)
    net = OverallNetwork()
    net.apply(weights_init)
    return net.cuda().train()


def _teacher(ctor_name="IR_50", seed=91):
    from crfr_b200.model import model_irse as IR
    torch.manual_seed(seed)
    t = getattr(IR, ctor_name)([112, 112])
    with torch.no_grad():   # non-trivial eval statistics
        g = torch.Generator().manual_seed(seed + 1)
        for m in t.modules():
            if isinstance(m, (torch.nn.BatchNorm2d, torch.nn.BatchNorm1d)):
                m.running_mean.copy_(0.1 * torch.randn(m.running_mean.shape, generator=g))
                m.running_var.copy_(1.0 + 0.2 * torch.rand(m.running_var.shape, generator=g))
    return t.cuda().eval()


def _batch(seed=8):
    from oracle import fsrnet_oracle as FO
    x, hr, lbl, hm = FO.synthetic_batch(B, S, seed=seed)
    return x.cuda(), hr.cuda(), hm.cuda(), lbl.cuda()


def _fsr_loss(outs, hr, hm, lbl):
    from crfr_b200.loss import CrossEntropyLoss2d, MSELoss_Landmark, MSELossFunc
    mse, lmk, ce = MSELossFunc(), MSELoss_Landmark(), CrossEntropyLoss2d()
    parts = (mse(outs[1], hr), mse(outs[0], hr), lmk(outs[2], hm), ce(outs[3], lbl))
    return (5. * parts[0] + 5. * parts[1] + parts[2] + parts[3]) / (2.0 * hr.shape[0])


def _module_path(teacher, batch, w_id=1.0, crop=(8, 8), identity=True, chunk=CHUNK):
    """Autograd through the drop-in modules on the loss of crfr_fsrnet_id_train_step -> (grads by name, total, id term).
    The batch runs through FSRNet in chunks of ``chunk`` images, as the trainer runs it: at 128 x 128 the FSRNet forward's
    bf16 bits depend on the images per call (the plain step's losses move by ~7e-4 between 2 and 4), and the loss is the
    global-batch mean either way (each chunk's means weighted by chunk / batch)."""
    x, hr, hm, lbl = batch
    fsr = _fsr()
    total = torch.zeros((), device="cuda")
    idl = torch.zeros((), device="cuda")
    for s0 in range(0, B, chunk):
        sl = slice(s0, s0 + chunk)
        outs = fsr(x[sl])
        total = total + _fsr_loss(outs, hr[sl], hm[sl], lbl[sl]) * (chunk / B) ** 2   # its means, and 1 / (2 B)
        if identity:
            with torch.no_grad():
                f_hr = teacher.forward_features(hr[sl, :, 8:120, 8:120].contiguous())
            y, x0 = crop
            f_sr = teacher.forward_features(outs[1][:, :, y:y + 112, x0:x0 + 112])
            idl = idl + w_id * sum(F.mse_loss(f_sr[k], f_hr[k]) for k in TERMS) * (chunk / B)
    (total + idl).backward()
    grads = {k: p.grad.detach().clone() for k, p in fsr.named_parameters() if p.grad is not None}
    return grads, float((total + idl).detach()), float(idl.detach())


def _trainer(teacher=None, chunk=CHUNK, **kw):
    from crfr_b200.trainer import FSRNetTrainer
    return FSRNetTrainer(_fsr(), lr=0.0, chunk=chunk, identity_net=teacher, **kw)


def _native(tr, batch):
    """One trainer step (lr = 0: the parameters stay put) -> ({name: gradient}, losses)."""
    losses = tr.step(*batch).clone()
    torch.cuda.synchronize()
    names = list(tr.model.state_dict().keys())
    return {k: g.clone() for k, g in zip(names, tr.grad_views)}, losses


def _live(grads):
    from oracle import fsrnet_oracle as FO
    return [k for k in grads if not FO.fsrnet_dead_param(k) and k not in FO.FSRNET_NULL_GRAD]


def _flat(grads, keys):
    return torch.cat([grads[k].double().reshape(-1).cpu() for k in keys])


def test_identity_step_matches_module_path_and_leaves_teacher_untouched(cuda):
    teacher = _teacher()
    bufs = [b.clone() for b in teacher.buffers()]
    batch = _batch()
    ref, ref_total, ref_id = _module_path(teacher, batch)
    got, losses = _native(_trainer(teacher), batch)
    assert losses.shape == (6,)
    assert abs(float(losses[5]) - ref_id) < 1e-4 * abs(ref_id), (float(losses[5]), ref_id)
    assert abs(float(losses[0]) - ref_total) < 1e-4 * abs(ref_total), (float(losses[0]), ref_total)
    for k in _live(ref):
        assert rel_err(got[k], ref[k]) < 6e-2, (k, rel_err(got[k], ref[k]))
    assert all(p.grad is None for p in teacher.parameters())
    assert all(torch.equal(a, b) for a, b in zip(bufs, teacher.buffers()))


@pytest.mark.parametrize("ctor", ["IR_50", "IR_SE_50"])
def test_identity_contribution_rejects_planted_errors(cuda, ctor):
    """grad(with the term) - grad(without), native against the module path; the same bound rejects a crop scattered at
    (7, 8) and w_id off by 10 %."""
    teacher = _teacher(ctor)
    batch = _batch(seed=11)
    w = W_BIG[ctor]
    with_id, _, _ = _module_path(teacher, batch, w_id=w)
    without, _, _ = _module_path(teacher, batch, identity=False)
    keys = _live(with_id)
    ref = _flat(with_id, keys) - _flat(without, keys)
    g1, _ = _native(_trainer(teacher, w_id=w), batch)
    g0, _ = _native(_trainer(teacher, w_id=0.0), batch)
    print("%s: |identity contribution| / |plain gradient| = %.2f" % (ctor, ref.norm() / _flat(without, keys).norm()))
    err = rel_err(_flat(g1, keys) - _flat(g0, keys), ref)
    shifted, _, _ = _module_path(teacher, batch, w_id=w, crop=(7, 8))
    heavier, _, _ = _module_path(teacher, batch, w_id=1.1 * w)
    err_shift = rel_err(_flat(g1, keys) - _flat(g0, keys), _flat(shifted, keys) - _flat(without, keys))
    err_w = rel_err(_flat(g1, keys) - _flat(g0, keys), _flat(heavier, keys) - _flat(without, keys))
    print("%s identity contribution: %.3e (planted: crop %.3e, w_id %.3e)" % (ctor, err, err_shift, err_w))
    assert err < CONTRIB_BOUND, err
    assert err_shift > CONTRIB_BOUND and err_w > CONTRIB_BOUND, (err_shift, err_w)


def test_zero_weight_equals_plain_step_bit_for_bit(cuda):
    batch = _batch()
    tr0 = _trainer(None)
    trz = _trainer(_teacher(), w_id=0.0)
    l0 = tr0.step(*batch).clone()
    lz = trz.step(*batch).clone()
    torch.cuda.synchronize()
    assert torch.equal(tr0.flat_g, trz.flat_g)
    assert torch.equal(l0, lz[:5])


def test_deterministic_graph_chunks_and_lanes(cuda):
    teacher = _teacher("IR_SE_50")
    batch = _batch()
    tr = _trainer(teacher)
    l1 = tr.step(*batch).clone()
    g1 = tr.flat_g.clone()
    l2 = tr.step(*batch).clone()
    torch.cuda.synchronize()
    assert torch.equal(g1, tr.flat_g) and torch.equal(l1, l2)
    trg = _trainer(teacher, use_graph=True)
    trg.step(batch[0] * 0.5, *batch[1:])            # captured on other data, replayed on ours
    lg = trg.step(*batch).clone()
    torch.cuda.synchronize()
    assert trg.replays == 2
    assert torch.equal(trg.flat_g, g1) and torch.equal(lg, l1)
    trl = _trainer(teacher, lanes=2)
    ll = trl.step(*batch).clone()
    torch.cuda.synchronize()
    print("lanes 2 vs 1 (chunk 2): gradients %.3e, losses %.3e" % (rel_err(trl.flat_g, g1), rel_err(ll, l1)))
    assert rel_err(trl.flat_g, g1) < 1e-6 and rel_err(ll, l1) < 1e-6
    # chunk 4 against chunk 2: at 128 x 128 the FSRNet step's own bits depend on the images per call, so the identity
    # step may differ between the two no more than the plain step does (the identity term adds no error of its own)
    tr4 = _trainer(teacher, chunk=4)
    l4 = tr4.step(*batch).clone()
    p2, p4 = _trainer(None), _trainer(None, chunk=4)
    pl2, pl4 = p2.step(*batch).clone(), p4.step(*batch).clone()
    torch.cuda.synchronize()
    e_id, e_plain = rel_err(tr4.flat_g, g1), rel_err(p4.flat_g, p2.flat_g)
    print("chunk 4 vs 2: gradients %.3e (plain step %.3e), losses %.3e (plain %.3e), identity term %.3e"
          % (e_id, e_plain, rel_err(l4[:5], l1[:5]), rel_err(pl4, pl2), rel_err(l4[5], l1[5])))
    assert e_id < 1.5 * e_plain + 1e-4
    assert rel_err(l4[:5], l1[:5]) < 1.5 * rel_err(pl4, pl2) + 1e-5 and rel_err(l4[5], l1[5]) < 1e-2


def test_rejections(cuda):
    from crfr_b200 import _lib as L
    from crfr_b200 import ops
    from crfr_b200.model import FSRnet as M
    from crfr_b200.model import model_irse as IR
    from crfr_b200.trainer import FSRNetTrainer
    teacher = _teacher()
    # a teacher in training mode, a 224 x 224 backbone, not a backbone at all
    with pytest.raises(RuntimeError, match="eval"):
        _trainer(_teacher().train())
    with pytest.raises(NotImplementedError, match="112"):
        _trainer(IR.IR_50([224, 224]).cuda().eval())
    with pytest.raises(TypeError):
        _trainer(torch.nn.Linear(2, 2))
    with pytest.raises(ValueError):
        _trainer(teacher, id_terms=(5,))
    tr = _trainer(teacher)
    teacher.train()
    with pytest.raises(RuntimeError, match="eval"):
        tr.step(*_batch())
    teacher.eval()
    # size 64 and a workspace that is too small: the native error code and message
    lib = L.lib()
    assert lib.crfr_fsrnet_id_workspace_bytes(50, 0, 2, 64) == 0
    assert lib.crfr_fsrnet_id_workspace_bytes(34, 0, 2, 128) == 0
    tr64 = FSRNetTrainer(_fsr(), lr=0.0, chunk=2, identity_net=teacher)
    from oracle import fsrnet_oracle as FO
    x, hr, lbl, hm = (t.cuda() for t in FO.synthetic_batch(2, 64))

    def call(x, hr, hm, lbl, ws_bytes):
        outs = M.alloc_outputs(x)
        io = M._io(x, outs, (hr, hm, lbl), loss_div=4.0, w_pix=5.0)
        ptab, btab, mask = tr64._id_tabs
        idio = L.FsrnetIdIO(50, 0, C.cast(ptab.arr, C.c_void_p), C.cast(btab.arr, C.c_void_p), 1.0, mask, 1.0)
        ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device="cuda")
        losses = torch.zeros(6, device="cuda")
        return lib.crfr_fsrnet_id_train_step(L.ENGINE_AUTO, tr64.ptable.arr, tr64.gtable.arr, C.byref(io), C.byref(idio),
                                             losses.data_ptr(), ws.data_ptr(), ws_bytes, ops.stream())

    assert call(x, hr, hm, lbl, 1 << 20) == 1                       # CRFR_EINVAL
    assert b"size 64" in lib.crfr_last_error()
    with pytest.raises(RuntimeError, match="size 64"):
        tr64.step(x, hr, hm, lbl)
    x, hr, hm, lbl = (t[:2].contiguous() for t in _batch())
    need = lib.crfr_fsrnet_id_workspace_bytes(50, 0, 2, 128)
    assert call(x, hr, hm, lbl, need - 4096) == 3                   # CRFR_EWORKSPACE
    assert b"workspace" in lib.crfr_last_error()
    assert all(p.grad is None for p in teacher.parameters())
