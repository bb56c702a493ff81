"""IR / IR-SE teachers without a GPU: the module mirror of every constructor against the oracle's seeded construction,
the oracle's forward against a plain-torch restatement of the reference modules, and the native size queries."""
import ctypes as C

import pytest
import torch
import torch.nn as nn

from tests.irnet_oracle import build_irnet_state_dict, irnet_forward, stage_ends
from tests.util import rel_err

# constructor name -> (num_layers, se, named_parameters, BatchNorm layers)
VARIANTS = {"IR_SE_50": (50, 1, 235, 54), "IR_101": (100, 0, 362, 104), "IR_SE_101": (100, 1, 460, 104),
            "IR_152": (152, 0, 369, 106), "IR_SE_152": (152, 1, 469, 106)}


@pytest.mark.parametrize("name", sorted(VARIANTS))
def test_irnet_mirror_keeps_reference_interface(name):
    from crfr_b200.model import model_irse as M
    num_layers, se, n_params, n_bn = VARIANTS[name]
    torch.manual_seed(91)
    net = getattr(M, name)([112, 112])
    sd, ref = net.state_dict(), build_irnet_state_dict(91, num_layers, se)
    assert [(k, tuple(v.shape)) for k, v in sd.items()] == [(k, tuple(v.shape)) for k, v in ref.items()]
    assert all(torch.equal(sd[k], ref[k]) for k in ref)               # identical seeded init, draw for draw
    assert len(list(net.named_parameters())) == n_params and len(list(net.named_buffers())) == 3 * n_bn
    if se:
        assert tuple(sd["body.0.res_layer.5.fc1.weight"].shape) == (4, 64, 1, 1)
        assert tuple(sd["body.%d.res_layer.5.fc2.weight" % stage_ends(num_layers)[3]].shape) == (512, 32, 1, 1)
    with pytest.raises(AssertionError):
        M.Backbone([96, 96], num_layers, "ir_se" if se else "ir")    # model_irse.py:132
    net.eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        net(torch.zeros(1, 3, 112, 112))
    with pytest.raises(NotImplementedError):
        M.Backbone([224, 224], num_layers, "ir_se" if se else "ir").eval()(torch.zeros(1, 3, 224, 224))


def test_irnet_oracle_ir50_is_the_pinned_ir50_oracle():
    from oracle import resnet_oracle as RO
    sd, ref = build_irnet_state_dict(91, 50, 0), RO.build_ir50_state_dict(91)
    assert list(sd) == list(ref) and all(torch.equal(sd[k], ref[k]) for k in ref)
    sd = RO.randomize_bn_everywhere(sd, 191)
    x = RO.synthetic_faces(2, seed=4322)
    with torch.no_grad():
        for name in ("fp32", "bf16"):
            pr = RO.Precision(name)
            emb, feats = irnet_forward(sd, x, pr=pr, want_features=True)
            ref_emb, ref_feats = RO.ir50_forward(sd, x, pr=pr, want_features=True)
            assert torch.equal(emb, ref_emb) and all(torch.equal(a, b) for a, b in zip(feats, ref_feats)), name


# ---- a plain-torch restatement of the reference modules (face.evoLVe model_irse.py), with their forward ----
class _SEModule(nn.Module):
    def __init__(self, channels, reduction):
        super().__init__()
        self.avg_pool = nn.AdaptiveAvgPool2d(1)
        self.fc1 = nn.Conv2d(channels, channels // reduction, kernel_size=1, padding=0, bias=False)
        self.relu = nn.ReLU(inplace=True)
        self.fc2 = nn.Conv2d(channels // reduction, channels, kernel_size=1, padding=0, bias=False)
        self.sigmoid = nn.Sigmoid()

    def forward(self, x):
        module_input = x
        x = self.avg_pool(x)
        x = self.fc1(x)
        x = self.relu(x)
        x = self.fc2(x)
        x = self.sigmoid(x)
        return module_input * x


class _Unit(nn.Module):
    def __init__(self, in_channel, depth, stride, se):
        super().__init__()
        if in_channel == depth:
            self.shortcut_layer = nn.MaxPool2d(1, stride)
        else:
            self.shortcut_layer = nn.Sequential(nn.Conv2d(in_channel, depth, (1, 1), stride, bias=False),
                                                nn.BatchNorm2d(depth))
        layers = [nn.BatchNorm2d(in_channel), nn.Conv2d(in_channel, depth, (3, 3), (1, 1), 1, bias=False),
                  nn.PReLU(depth), nn.Conv2d(depth, depth, (3, 3), stride, 1, bias=False), nn.BatchNorm2d(depth)]
        if se:
            layers.append(_SEModule(depth, 16))
        self.res_layer = nn.Sequential(*layers)

    def forward(self, x):
        shortcut = self.shortcut_layer(x)
        res = self.res_layer(x)
        return res + shortcut


class _Flatten(nn.Module):
    def forward(self, x):
        return x.view(x.size(0), -1)


class _Backbone(nn.Module):
    def __init__(self, num_layers, se):
        super().__init__()
        units = {50: (3, 4, 14, 3), 100: (3, 13, 30, 3), 152: (3, 8, 36, 3)}[num_layers]
        self.input_layer = nn.Sequential(nn.Conv2d(3, 64, (3, 3), 1, 1, bias=False), nn.BatchNorm2d(64), nn.PReLU(64))
        self.output_layer = nn.Sequential(nn.BatchNorm2d(512), nn.Dropout(), _Flatten(), nn.Linear(512 * 7 * 7, 512),
                                          nn.BatchNorm1d(512))
        modules, in_ch = [], 64
        for n, depth in zip(units, (64, 128, 256, 512)):
            for u in range(n):
                modules.append(_Unit(in_ch, depth, 2 if u == 0 else 1, se))
                in_ch = depth
        self.body = nn.Sequential(*modules)

    def forward(self, x):
        x = self.input_layer(x)
        x = self.body(x)
        return self.output_layer(x)


@pytest.mark.parametrize("name", ["IR_SE_50", "IR_152"])
def test_irnet_oracle_matches_plain_torch_restatement(name):
    from oracle import resnet_oracle as RO
    num_layers, se = VARIANTS[name][:2]
    sd = RO.randomize_bn_everywhere(build_irnet_state_dict(91, num_layers, se), 191)
    net = _Backbone(num_layers, se)
    net.load_state_dict(sd)
    net.eval()
    feats = []
    for i in stage_ends(num_layers):
        net.body[i].register_forward_hook(lambda m, inp, out: feats.append(out))
    x = RO.synthetic_faces(2, seed=4322)
    with torch.no_grad():
        ref = net(x)
        emb, ofeats = irnet_forward(sd, x, want_features=True)
    assert rel_err(emb, ref) < 1e-5
    assert len(ofeats) == 4 and all(rel_err(a, b) < 1e-5 for a, b in zip(ofeats, feats))


def test_irnet_native_size_queries():
    import crfr_b200
    crfr_b200.build()
    from crfr_b200 import _lib as L
    lib = L.lib()
    for b in (1, 4, 256):
        assert lib.crfr_irnet_workspace_bytes(50, 0, b, 112) == lib.crfr_ir50_workspace_bytes(b, 112)
        assert lib.crfr_irnet_grad_workspace_bytes(50, 0, b, 112) == lib.crfr_ir50_grad_workspace_bytes(b, 112)
    assert lib.crfr_kd_workspace_bytes_ir(64, 112, 50, 0) == lib.crfr_kd_workspace_bytes_ex(64, 112, 1)
    assert L.irnet_sizes(50, 0) == (L.IR50_NPARAMS, L.IR50_NBN)
    for name, (num_layers, se, n_params, n_bn) in VARIANTS.items():
        assert L.irnet_sizes(num_layers, se) == (n_params, n_bn), name
        for b in (1, 4, 256):
            fwd = lib.crfr_irnet_workspace_bytes(num_layers, se, b, 112)
            assert 0 < fwd < lib.crfr_irnet_grad_workspace_bytes(num_layers, se, b, 112), (name, b)
        assert lib.crfr_kd_workspace_bytes_ir(64, 112, num_layers, se) > 0
        assert lib.crfr_irnet_workspace_bytes(num_layers, se, 4, 224) == 0
        assert lib.crfr_irnet_grad_workspace_bytes(num_layers, se, 4, 96) == 0
        assert lib.crfr_irnet_tape(num_layers, se, 0, 112, None, 0) < 0
    for num_layers, se in ((34, 0), (18, 1), (50, 2), (101, 0), (0, 0)):
        assert lib.crfr_irnet_workspace_bytes(num_layers, se, 4, 112) == 0
        assert lib.crfr_irnet_grad_workspace_bytes(num_layers, se, 4, 112) == 0
        assert lib.crfr_kd_workspace_bytes_ir(4, 112, num_layers, se) == 0
        assert lib.crfr_irnet_tape(num_layers, se, 4, 112, None, 0) < 0
        n = C.c_int()
        assert lib.crfr_irnet_sizes(num_layers, se, C.byref(n), None) != 0
        assert b"unsupported IR variant" in lib.crfr_last_error()
        # the calls reject the variant before touching any pointer
        assert lib.crfr_irnet_forward(0, num_layers, se, None, None, None, None, 0, None) != 0
        assert lib.crfr_irnet_backward(0, num_layers, se, None, None, None, None, None, None, None, 0, None) != 0


def test_irnet_tape_lists_the_se_units():
    import crfr_b200
    crfr_b200.build()
    from crfr_b200 import _lib as L
    lib = L.lib()
    for name, (num_layers, se, _, _) in VARIANTS.items():
        units = {50: 24, 100: 49, 152: 50}[num_layers]
        n = lib.crfr_irnet_tape(num_layers, se, 2, 112, None, 0)
        # stem conv + BN/PReLU, units x (BN, conv, PReLU, conv, BN or SE) + 3 x (shortcut conv, BN) + 1 subsampling, head
        assert n == 2 + units * 5 + 3 * 2 + 1 + 3, name
        arr = (L.TapeEntry * n)()
        assert lib.crfr_irnet_tape(num_layers, se, 2, 112, arr, n) == n
        kinds = [e.kind for e in arr]
        assert kinds.count(10) == (units if se else 0) and kinds.count(8) == units, name
        for e in arr:
            if e.kind == 10:
                assert e.stats_off >= 0 and e.has_res == 1 and e.n == 2


def _grad_tape(lib, L, num_layers, se, b, mask):
    n = lib.crfr_irnet_grad_tape(num_layers, se, b, 112, mask, None, 0)
    assert n > 0, (num_layers, se, b, mask)
    arr = (L.TapeEntry * n)()
    assert lib.crfr_irnet_grad_tape(num_layers, se, b, 112, mask, arr, n) == n
    return list(arr)


@pytest.mark.parametrize("name", ["IR_50"] + sorted(VARIANTS))
def test_irnet_grad_tape_layout(name):
    """crfr_irnet_grad_tape: one entry per stored gradient of the IR backward, each inside the grad workspace past the
    forward arena, no two overlapping (except a unit's output gradient that is the very buffer of the gradient flowing
    into it), each naming the stored forward tensor it differentiates."""
    import crfr_b200
    crfr_b200.build()
    from crfr_b200 import _lib as L
    lib = L.lib()
    num_layers, se = (50, 0) if name == "IR_50" else VARIANTS[name][:2]
    units = {50: (3, 4, 14, 3), 100: (3, 13, 30, 3), 152: (3, 8, 36, 3)}[num_layers]
    per_unit = 4 if se else 3
    for b in (2, 5):
        fwd_end = lib.crfr_irnet_workspace_bytes(num_layers, se, b, 112) - 65536   # the forward arena's end
        grad_bytes = lib.crfr_irnet_grad_workspace_bytes(num_layers, se, b, 112)
        nf = lib.crfr_irnet_tape(num_layers, se, b, 112, None, 0)
        ftape = (L.TapeEntry * nf)()
        lib.crfr_irnet_tape(num_layers, se, b, 112, ftape, nf)
        fwd = {e.out_off: e for e in ftape}
        for mask in (1, 2, 4, 8, 16, 17, 30, 31):
            tape = _grad_tape(lib, L, num_layers, se, b, mask)
            # the units up to the deepest seeded output have a gradient
            last_stage = 3 if mask & 1 else max(l for l in range(4) if mask >> (l + 1) & 1)
            n_units = sum(units[:last_stage + 1])
            assert len(tape) == (mask & 1) + n_units * per_unit + 1, (name, mask)
            kinds = [e.kind for e in tape]
            assert kinds[-1] == 16 and (kinds[0] == 11) == bool(mask & 1)
            body = kinds[(mask & 1):-1]
            assert body == ([12, 13, 14, 15] if se else [12, 14, 15]) * n_units, (name, mask)
            assert [e.w_idx for e in tape[(mask & 1):-1]] == [u for u in reversed(range(n_units)) for _ in range(per_unit)]
            spans = []
            for i, e in enumerate(tape):
                f = fwd.get(e.in_off)
                assert f is not None, (name, mask, i, e.kind)   # every gradient is of a stored forward tensor
                assert (e.n, e.h, e.w, e.c) == (f.n, f.h, f.w, f.c) and e.ld >= e.c, (name, mask, i)
                if e.kind == 13:
                    assert f.kind == 0                               # dr is paired with y, res_layer.3's output
                    spans.append((e.stats_off, e.stats_off + 4 * e.n * e.c, i))
                else:
                    assert e.stats_off == -1
                if e.kind == 14:
                    assert f.kind == 0                               # res_layer.1's output
                spans.append((e.out_off, e.out_off + 2 * e.n * e.h * e.w * e.ld, i))
            for lo, hi, i in spans:
                assert fwd_end <= lo < hi <= grad_bytes, (name, mask, i, lo, hi, fwd_end, grad_bytes)
            spans.sort()
            for (lo0, hi0, i0), (lo1, hi1, i1) in zip(spans, spans[1:]):
                if lo1 < hi0:   # only a unit's summed output gradient may alias, and only the buffer that produced it
                    a, c = sorted((i0, i1))
                    assert (lo0, hi0) == (lo1, hi1) and tape[c].kind == 12, (name, mask, i0, i1)
                    assert tape[a].kind in (11, 15) and tape[a].in_off == tape[c].in_off, (name, mask, i0, i1)
    for args in ((num_layers, se, 0, 112, 1), (num_layers, se, 4, 96, 1), (num_layers, se, 4, 112, 0),
                 (num_layers, se, 4, 112, 32), (num_layers, se, 4, 112, -1), (34, 0, 4, 112, 1), (50, 2, 4, 112, 1)):
        assert lib.crfr_irnet_grad_tape(*args, None, 0) == -1, args


def test_irnet_grad_reference_forward_is_the_oracle():
    """The bf16 gradient reference of tests/test_irnet_gpu.py adds gradient roundings to irnet_forward; its forward must
    stay irnet_forward's, for an SE and a plain variant."""
    from oracle import resnet_oracle as RO
    from tests.test_irnet_gpu import VARIANTS as GPU_VARIANTS, _ir_ref, _state
    x = RO.synthetic_faces(2, seed=4322)
    for name in ("IR_SE_50", "IR_101"):
        sd = _state(name)
        with torch.no_grad():
            for prec in ("fp32", "bf16"):
                pr = RO.Precision(prec)
                emb, feats = _ir_ref(sd, x, pr, *GPU_VARIANTS[name])
                ref_emb, ref_feats = irnet_forward(sd, x, pr=pr, want_features=True)
                assert torch.equal(emb, ref_emb) and all(torch.equal(a, b) for a, b in zip(feats, ref_feats)), (name, prec)
