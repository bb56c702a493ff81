"""Drop-in for the reference's SUPER_RESOLUTION/model/FSRnet.py:251-416: the newer face-hallucination network the authors
trained on CelebA-HQ (SURVEY 8f-2) - ReflectionPad convolutions, non-affine InstanceNorm + ReLU, stride-2 encoder /
transposed-conv decoder stages, a prior network of four depth-4 hourglasses of pre-activation Bottleneck blocks, Tanh
image heads.

Same class names, constructor arguments, ``nn.Sequential`` indices and parameter names (identical ``state_dict`` keys;
the parameter-free layers - ReflectionPad2d, InstanceNorm2d, ReLU, Tanh - are kept as containers so the indices match),
same ``forward`` signatures.  ``forward`` never calls the torch layers: ``SRNetwork`` and each sub-network run as one
native network program (crfr_srnet_forward, csrc/srnet.cu) with one autograd node (crfr_srnet_backward).  Inside it
every layer keeps the routing of the single-op entry points (tcgen05 implicit GEMM for the 3x3 stride-1 convolutions;
the lowered tcgen05 recipes for the stride-2, 7x7, 1x1, transposed and 3-channel ones; the 3x3 stem's input gradient on
CUDA cores), the two 1x1 prior heads run as one tensor-core GEMM, and activations stay NHWC bf16 in the program's
workspace.  Module inputs and outputs are fp32 NCHW.

The reference's ``OverallNetwork`` of this file cannot be constructed (it names a class ``Course_SR_Network`` that the
file does not define, :449; SURVEY Appendix C); ``SRNetwork`` below is that wiring with the classes that do exist
(coarse image -> encoder and prior network -> concatenation -> decoder), the one ``train_FHN.py`` drives by hand.
"""
import ctypes as C

import torch
import torch.nn as nn

from ... import _lib as L
from ... import ops


def _check(x, channels, section):
    if not x.is_cuda:
        raise RuntimeError("crfr_b200 SUPER_RESOLUTION networks need CUDA tensors: the hot path has no CPU fallback")
    if x.dim() != 4 or x.shape[1] != channels:
        raise ValueError("expected [B,%d,H,W], got %s" % (channels, tuple(x.shape)))
    if L.lib().crfr_srnet_workspace_bytes(section, x.shape[0], x.shape[2], x.shape[3], 0) == 0:
        raise ValueError("input %s not supported: H and W must be >= 5 (multiples of 16 for the prior network and "
                         "SRNetwork; include/crfr.h, crfr_srnet_io)" % (tuple(x.shape),))


def _out_shapes(section, b, h, w):
    big_h, big_w = 4 * -(-h // 4), 4 * -(-w // 4)
    if section == L.SRNET_NETWORK:
        return [(b, 3, h, w), (b, 3, h, w), (b, 68, h, w), (b, 13, h, w)]
    if section == L.SRNET_PRIOR:
        return [(b, 64, h, w), (b, 68, h, w), (b, 13, h, w)]
    return [(b, 64 if section == L.SRNET_ENCODER else 3, big_h, big_w)]


def _unreached(section, given):
    """Parameter indices no given output gradient reaches (they keep grad None, as under autograd through the layers):
    the heads without their output's gradient; in SRNetwork also the encoder and decoder without the image gradient,
    and the prior trunk when neither the image nor a head has one."""
    if section == L.SRNET_PRIOR:
        return set(([0, 1] if not given[2] else []) + ([2] if not given[1] else []))
    if section != L.SRNET_NETWORK:
        return set()
    dead = set(([52, 53] if not given[3] else []) + ([54] if not given[2] else []))
    if not given[1]:
        dead |= set(range(1006, 1108))
        if not (given[2] or given[3]):
            dead |= set(range(55, 1006))
    return dead


def _table(tensors):
    return (C.c_void_p * len(tensors))(*[None if t is None else t.data_ptr() for t in tensors])


def _flat_grads(params, dev):
    """One zeroed flat fp32 buffer with a 16-byte aligned view per parameter (the native backward accumulates)."""
    offs, tot = [], 0
    for p in params:
        offs.append(tot)
        tot += (p.numel() + 3) // 4 * 4
    flat = torch.zeros(tot, dtype=torch.float32, device=dev)
    return flat, [flat[o:o + p.numel()].view(p.shape) for o, p in zip(offs, params)]


class _SRProgram(torch.autograd.Function):
    """One section as a native program (crfr_srnet_forward) with its own autograd node (crfr_srnet_backward)."""

    @staticmethod
    def forward(ctx, x, engine, section, need_grad, *params):
        x = x.contiguous().float()
        b, _, h, w = x.shape
        outs = [torch.empty(s, dtype=torch.float32, device=x.device) for s in _out_shapes(section, b, h, w)]
        nbytes = L.lib().crfr_srnet_workspace_bytes(section, b, h, w, 1 if need_grad else 0)
        # a private workspace per call when a backward may follow: it holds the saved activations
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device) if need_grad else ops.workspace(nbytes)
        io = L.SrnetIO()
        io.section, io.batch, io.h, io.w = section, b, h, w
        io.x = x.data_ptr()
        for i, o in enumerate(outs):
            io.out[i] = o.data_ptr()
        L.call("crfr_srnet_forward", engine, _table([p.detach() for p in params]), C.byref(io), 1 if need_grad else 0,
               ws.data_ptr(), ws.numel(), ops.stream())
        # only shapes are kept: outputs on ctx would close the cycle output -> grad_fn -> ctx -> output
        ctx.engine, ctx.section, ctx.xshape, ctx.dev = engine, section, tuple(x.shape), x.device
        ctx.ws = ws if need_grad else None
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(*params)
        return tuple(outs)

    @staticmethod
    def backward(ctx, *d_outs):
        params = ctx.saved_tensors
        _, grads = _flat_grads(params, ctx.dev)
        b, _, h, w = ctx.xshape
        io = L.SrnetIO()                       # the backward reads neither x nor the outputs
        io.section, io.batch, io.h, io.w = ctx.section, b, h, w
        keep = [None if d is None else d.contiguous().float() for d in d_outs]
        darr = (C.c_void_p * 4)(*[None if d is None else d.data_ptr() for d in keep] + [None] * (4 - len(keep)))
        dx = torch.empty(ctx.xshape, dtype=torch.float32, device=ctx.dev) if ctx.needs_input_grad[0] else None
        L.call("crfr_srnet_backward", ctx.engine, _table([p.detach() for p in params]), _table(grads), C.byref(io), darr,
               ops.ptr(dx), ctx.ws.data_ptr(), ctx.ws.numel(), ops.stream())
        ctx.ws = None
        dead = _unreached(ctx.section, [d is not None for d in keep] + [False] * (4 - len(keep)))
        return (dx, None, None, None) + tuple(None if i in dead else g for i, g in enumerate(grads))


_TABLES = {}


def check_parameter_table(module, params):
    """The program's channel counts are those of the reference's default constructor arguments: every parameter must
    have the shape the default-constructed module gives it (checked on the host, before any launch)."""
    cls = type(module)
    if cls not in _TABLES:
        ref = cls()
        _TABLES[cls] = [tuple(t.shape) for t in ref.state_dict().values()]
    want = _TABLES[cls]
    got = [tuple(p.shape) for p in params]
    if got != want:
        bad = next(i for i in range(min(len(got), len(want)) + 1) if i >= len(got) or i >= len(want) or got[i] != want[i])
        raise NotImplementedError(
            "%s: the native program runs the reference's default configuration only; parameter %d has shape %s, the "
            "program expects %s (%d parameters, %d expected)" % (cls.__name__, bad, got[bad] if bad < len(got) else None,
                                                                  want[bad] if bad < len(want) else None, len(got),
                                                                  len(want)))


class _Program(nn.Module):
    """forward(x) of a whole section: its parameters in state_dict order are the program's parameter table."""
    _section = None
    _in_channels = 3
    engine = L.ENGINE_AUTO

    def _run(self, x):
        sd = dict(self.named_parameters())
        params = [sd[k] for k in self.state_dict().keys()]
        check_parameter_table(self, params)
        _check(x, self._in_channels, self._section)
        need_grad = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in params))
        return _SRProgram.apply(x, self.engine, self._section, need_grad, *params)


class _Residual_Block(nn.Module):
    """ref: SUPER_RESOLUTION/model/FSRnet.py:12-37: conv -> IN(affine) -> PReLU -> conv -> IN(affine) -> + x (no
    activation after the sum, unlike model/FSRnet.py's block)."""

    def __init__(self, out_channels, in_channels=64):
        super().__init__()
        self.conv1 = nn.Conv2d(in_channels, out_channels, 3, 1, 1, bias=False)
        self.in1 = nn.InstanceNorm2d(out_channels, affine=True)
        self.relu = nn.PReLU(out_channels)
        self.conv2 = nn.Conv2d(out_channels, out_channels, 3, 1, 1, bias=False)
        self.in2 = nn.InstanceNorm2d(out_channels, affine=True)


class Bottleneck(nn.Module):
    """ref: :75-114: pre-activation bottleneck IN -> ReLU -> conv1x1 -> IN -> ReLU -> conv3x3 -> IN -> ReLU -> conv1x1, + x."""
    expansion = 1

    def __init__(self, inplanes, planes, stride=1, downsample=None):
        super().__init__()
        self.bn1 = nn.InstanceNorm2d(inplanes)
        self.conv1 = nn.Conv2d(inplanes, planes, kernel_size=1, bias=True)
        self.bn2 = nn.InstanceNorm2d(planes)
        self.conv2 = nn.Conv2d(planes, planes, kernel_size=3, stride=stride, padding=1, bias=True)
        self.bn3 = nn.InstanceNorm2d(planes)
        self.conv3 = nn.Conv2d(planes, planes, kernel_size=1, bias=True)
        self.relu = nn.ReLU(inplace=True)
        self.downsample = downsample
        self.stride = stride


class Hourglass(nn.Module):
    """ref: :117-156 (same recursion as model/FSRnet.py:176-215)."""

    def __init__(self, block, num_blocks, planes, depth):
        super().__init__()
        self.depth = depth
        self.block = block
        self.hg = nn.ModuleList(
            nn.ModuleList(nn.Sequential(*[block(planes * block.expansion, planes) for _ in range(num_blocks)])
                          for _ in range(4 if d == 0 else 3))
            for d in range(depth))


def _trunk(ngf, n_blocks, stem):
    """The shared body of the coarse network / encoder / decoder: two stride-2 stages, residual blocks, two up stages."""
    m = list(stem)
    m += [nn.ReflectionPad2d(1), nn.Conv2d(ngf, ngf * 2, 3, 2, 0, bias=False),
          nn.ReflectionPad2d(1), nn.Conv2d(ngf * 2, ngf * 2, 3, 1, 0, bias=False), nn.InstanceNorm2d(ngf * 2), nn.ReLU(True),
          nn.ReflectionPad2d(1), nn.Conv2d(ngf * 2, ngf * 4, 3, 2, 0, bias=False),
          nn.ReflectionPad2d(1), nn.Conv2d(ngf * 4, ngf * 4, 3, 1, 0, bias=False), nn.InstanceNorm2d(ngf * 2), nn.ReLU(True)]
    m += [_Residual_Block(out_channels=ngf * 4, in_channels=ngf * 4) for _ in range(n_blocks)]
    m += [nn.ConvTranspose2d(ngf * 4, ngf * 2, 3, 2, 1, 1, bias=False), nn.ReflectionPad2d(1),
          nn.Conv2d(ngf * 2, ngf * 2, 3, 1, 0, bias=False), nn.InstanceNorm2d(ngf * 2), nn.ReLU(True),
          nn.ConvTranspose2d(ngf * 2, ngf, 3, 2, 1, 1, bias=False), nn.ReflectionPad2d(1),
          nn.Conv2d(ngf, ngf, 3, 1, 0, bias=False), nn.InstanceNorm2d(ngf), nn.ReLU(True)]
    return m


class Coarse_SR_Network(_Program):
    """ref: :251-301; forward(x) -> coarse image [B,3,H,W]."""
    _section = L.SRNET_COARSE

    def __init__(self, ngf=64, n_blocks=6):
        super().__init__()
        stem = [nn.ReflectionPad2d(3), nn.Conv2d(3, ngf, 7, 1, 0, bias=False), nn.InstanceNorm2d(ngf), nn.ReLU(True)]
        self.model = nn.Sequential(*_trunk(ngf, n_blocks, stem))
        self.out = nn.Sequential(nn.ReflectionPad2d(1), nn.Conv2d(ngf, 3, 3, 1, 0, bias=False), nn.Tanh())
        self.n_blocks = n_blocks

    def forward(self, x):
        return self._run(x)[0]


class Fine_SR_Encoder(_Program):
    """ref: :304-346; forward(x) -> features [B,ngf,H,W]."""
    _section = L.SRNET_ENCODER

    def __init__(self, ngf=64, n_blocks=6):
        super().__init__()
        stem = [nn.ReflectionPad2d(1), nn.Conv2d(3, ngf, 3, 1, 0, bias=False)]
        self.model = nn.Sequential(*_trunk(ngf, n_blocks, stem))
        self.n_blocks, self.ngf = n_blocks, ngf

    def forward(self, x):
        return self._run(x)[0]


class Prior_Estimation_Network(_Program):
    """ref: :349-376; forward(x) -> (features, landmark_out, parsing_out)."""
    _section = L.SRNET_PRIOR

    def __init__(self, n_hourglass=4, n_blocks=2, ngf=64, parsing_classes=13, num_landmark=68):
        super().__init__()
        self.fc = nn.Conv2d(ngf, parsing_classes, kernel_size=1, bias=True)
        self.fc_landmark = nn.Conv2d(ngf, num_landmark, kernel_size=1, bias=False)
        model = [nn.ReflectionPad2d(3), nn.Conv2d(3, ngf, 7, 1, 0, bias=False), nn.InstanceNorm2d(ngf), nn.ReLU(True)]
        model += [_Residual_Block(ngf) for _ in range(n_blocks)]
        model += [Hourglass(planes=ngf, depth=4, block=Bottleneck, num_blocks=3) for _ in range(n_hourglass)]
        self.model = nn.Sequential(*model)

    def forward(self, x):
        return self._run(x)


class Fine_SR_Decoder(_Program):
    """ref: :379-416; forward(x [B,ngf,H,W]) -> image [B,3,H,W]."""
    _section = L.SRNET_DECODER

    def __init__(self, ngf=128, n_blocks=6):
        super().__init__()
        self.model = nn.Sequential(*_trunk(ngf, n_blocks, []))
        self.out = nn.Sequential(nn.ReflectionPad2d(1), nn.Conv2d(ngf, 3, 3, 1, 0, bias=False), nn.Tanh())
        self.n_blocks, self.ngf = n_blocks, ngf
        self._in_channels = ngf

    def forward(self, x):
        return self._run(x)[0]


class SRNetwork(_Program):
    """The wiring the reference's (unconstructible, :449) ``OverallNetwork`` of this file describes, with the classes that
    exist: coarse image -> encoder and prior network -> cat(prior, encoder) -> decoder;
    forward(x) -> (coarse_out, out, landmark_out, parsing_out).  One native program: the prior and encoder features are
    written straight into the two channel halves of the decoder's 128-channel input."""
    _section = L.SRNET_NETWORK

    def __init__(self):
        super().__init__()
        self._coarse_sr_network = Coarse_SR_Network()
        self._prior_estimation_network = Prior_Estimation_Network()
        self._fine_sr_encoder = Fine_SR_Encoder()
        self._fine_sr_decoder = Fine_SR_Decoder()

    def forward(self, x):
        return self._run(x)
