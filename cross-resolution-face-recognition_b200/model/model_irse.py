"""Drop-in IR / IR-SE teachers backed by the native sm_100a network program (forward, and the gradient w.r.t. the input).

Mirror of the reference's DISTILLATION/model/model_irse.py (face.evoLVe): the six constructors ``IR_50``, ``IR_101``,
``IR_152``, ``IR_SE_50``, ``IR_SE_101`` and ``IR_SE_152`` (distill_main.py:14,201 uses ``IR_50([112, 112])``), with the
same class names (``Backbone``, ``bottleneck_IR``, ``bottleneck_IR_SE``, ``SEModule``, ``Flatten``, ``l2_norm``,
``get_blocks``), constructor arguments, sub-module / parameter / buffer names (identical ``state_dict`` keys, so the
pretrained face.evoLVe checkpoints load) and construction + initialisation order.  The torch layers are parameter
containers only; ``Backbone.forward`` runs ``crfr_irnet_forward`` for the variant (num_layers, mode).  Every variant is
native at 112 x 112; 224 x 224 is not.

The teacher is frozen and evaluated in ``eval()`` mode by the reference (distill_main.py:43, 112-114); only that mode
is native: train-mode Dropout (model_irse.py:144) is stochastic and has no parity definition, so ``forward`` in
training mode raises.

When ``x.requires_grad`` (and grad mode is on), ``forward`` / ``forward_features`` are differentiable with respect to
``x`` through ``crfr_irnet_backward``, so that the teacher can drive an identity or perceptual loss on a super-resolved
face (SUPER_RESOLUTION/train_FHN.py:255-265)::

    sr = fsrnet(x)[1][:, :, 8:120, 8:120]
    f_sr, f_hr = ir50.forward_features(sr), ir50.forward_features(hr)
    loss = pixel_loss + sum(F.mse_loss(a, b) for a, b in zip(f_sr, f_hr))
    loss.backward()          # reaches fsrnet's parameters through IR_50

The teacher's own parameters stay frozen: they never receive a ``.grad``, even with ``requires_grad=True``.
"""
import ctypes as C
from collections import namedtuple

import torch
import torch.nn as nn
from torch.autograd.function import once_differentiable
from torch.nn import (AdaptiveAvgPool2d, BatchNorm1d, BatchNorm2d, Conv2d, Dropout, Linear, MaxPool2d, Module, PReLU, ReLU,
                      Sequential, Sigmoid)

from .. import _lib as L
from .. import ops

__all__ = ["Backbone", "IR_50", "IR_101", "IR_152", "IR_SE_50", "IR_SE_101", "IR_SE_152", "bottleneck_IR",
           "bottleneck_IR_SE", "SEModule", "Flatten", "l2_norm", "get_blocks"]


class Flatten(Module):
    """ref: model_irse.py:10-12."""

    def forward(self, input):
        return input.view(input.size(0), -1)


def l2_norm(input, axis=1):
    """ref: model_irse.py:15-19."""
    norm = torch.norm(input, 2, axis, True)
    return torch.div(input, norm)


class bottleneck_IR(Module):
    """ref: model_irse.py:49-66 (shortcut: MaxPool2d(1, stride) or conv1x1 + BN; residual: BN, conv3x3, PReLU,
    conv3x3(stride), BN)."""

    def __init__(self, in_channel, depth, stride):
        super().__init__()
        if in_channel == depth:
            self.shortcut_layer = MaxPool2d(1, stride)
        else:
            self.shortcut_layer = Sequential(Conv2d(in_channel, depth, (1, 1), stride, bias=False), BatchNorm2d(depth))
        self.res_layer = Sequential(BatchNorm2d(in_channel),
                                    Conv2d(in_channel, depth, (3, 3), (1, 1), 1, bias=False), PReLU(depth),
                                    Conv2d(depth, depth, (3, 3), stride, 1, bias=False), BatchNorm2d(depth))


class SEModule(Module):
    """ref: model_irse.py SEModule: x * sigmoid(fc2(relu(fc1(avg_pool(x))))).  fc1 is xavier-initialised at construction
    (and again by Backbone._initialize_weights), as the reference does: seeded construction draws the same numbers."""

    def __init__(self, channels, reduction):
        super().__init__()
        self.avg_pool = AdaptiveAvgPool2d(1)
        self.fc1 = Conv2d(channels, channels // reduction, kernel_size=1, padding=0, bias=False)
        nn.init.xavier_uniform_(self.fc1.weight.data)
        self.relu = ReLU(inplace=True)
        self.fc2 = Conv2d(channels // reduction, channels, kernel_size=1, padding=0, bias=False)
        self.sigmoid = Sigmoid()


class bottleneck_IR_SE(Module):
    """ref: model_irse.py bottleneck_IR_SE: bottleneck_IR whose residual ends in SEModule(depth, 16)."""

    def __init__(self, in_channel, depth, stride):
        super().__init__()
        if in_channel == depth:
            self.shortcut_layer = MaxPool2d(1, stride)
        else:
            self.shortcut_layer = Sequential(Conv2d(in_channel, depth, (1, 1), stride, bias=False), BatchNorm2d(depth))
        self.res_layer = Sequential(BatchNorm2d(in_channel),
                                    Conv2d(in_channel, depth, (3, 3), (1, 1), 1, bias=False), PReLU(depth),
                                    Conv2d(depth, depth, (3, 3), stride, 1, bias=False), BatchNorm2d(depth),
                                    SEModule(depth, 16))


class Bottleneck(namedtuple("Block", ["in_channel", "depth", "stride"])):
    """A named tuple describing a ResNet block (ref: model_irse.py:92-93)."""


def get_block(in_channel, depth, num_units, stride=2):
    return [Bottleneck(in_channel, depth, stride)] + [Bottleneck(depth, depth, 1) for _ in range(num_units - 1)]


def get_blocks(num_layers):
    """ref: model_irse.py:101-126."""
    table = {50: (3, 4, 14, 3), 100: (3, 13, 30, 3), 152: (3, 8, 36, 3)}
    u = table[num_layers]
    return [get_block(64, 64, u[0]), get_block(64, 128, u[1]), get_block(128, 256, u[2]), get_block(256, 512, u[3])]


class _Table:
    def __init__(self, tensors, n):
        assert len(tensors) == n, (len(tensors), n)
        self.arr = (C.c_void_p * n)(*[t.data_ptr() for t in tensors])
        self.keep = tensors


class Backbone(Module):
    """ref: model_irse.py:129-188; forward(x) -> 512-d embedding."""

    def __init__(self, input_size, num_layers, mode="ir"):
        super().__init__()
        assert input_size[0] in [112, 224], "input_size should be [112, 112] or [224, 224]"
        assert num_layers in [50, 100, 152], "num_layers should be 50, 100 or 152"
        assert mode in ["ir", "ir_se"], "mode should be ir or ir_se"
        blocks = get_blocks(num_layers)
        unit_module = bottleneck_IR if mode == "ir" else bottleneck_IR_SE
        self.input_layer = Sequential(Conv2d(3, 64, (3, 3), 1, 1, bias=False), BatchNorm2d(64), PReLU(64))
        feat = 512 * 7 * 7 if input_size[0] == 112 else 512 * 14 * 14
        self.output_layer = Sequential(BatchNorm2d(512), Dropout(), Flatten(), Linear(feat, 512), BatchNorm1d(512))
        modules = []
        for block in blocks:
            for bottleneck in block:
                modules.append(unit_module(bottleneck.in_channel, bottleneck.depth, bottleneck.stride))
        self.body = Sequential(*modules)
        self._initialize_weights()
        self.engine = L.ENGINE_AUTO
        self._variant = (num_layers, 1 if mode == "ir_se" else 0)   # (num_layers, se) of the crfr_irnet_* calls
        self._native = input_size[0] == 112

    def _initialize_weights(self):
        """ref: model_irse.py:174-188."""
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.xavier_uniform_(m.weight.data)
                if m.bias is not None:
                    m.bias.data.zero_()
            elif isinstance(m, (nn.BatchNorm2d, nn.BatchNorm1d)):
                m.weight.data.fill_(1)
                m.bias.data.zero_()
            elif isinstance(m, nn.Linear):
                nn.init.xavier_uniform_(m.weight.data)
                if m.bias is not None:
                    m.bias.data.zero_()

    def _check(self, x):
        if not self._native:
            raise NotImplementedError("only the 112 x 112 IR / IR_SE backbones have a native network program")
        if self.training:
            raise RuntimeError("the native IR backbone is the frozen teacher: call .eval() first (train-mode Dropout is "
                               "stochastic and has no parity definition)")
        if not x.is_cuda:
            raise RuntimeError("crfr_b200 IR backbone needs a CUDA tensor: the hot path has no CPU fallback")
        if x.dim() != 4 or tuple(x.shape[1:]) != (3, 112, 112):
            raise ValueError("expected [B,3,112,112], got %s" % (tuple(x.shape),))

    def _launch(self, x, want_features, ws=None):
        """crfr_irnet_forward into ``ws`` (default: the shared workspace) -> (emb, feats, tables, io)."""
        b = x.shape[0]
        emb = torch.empty((b, 512), dtype=torch.float32, device=x.device)
        feats = [torch.empty((b, c, s, s), dtype=torch.float32, device=x.device)
                 for c, s in ((64, 56), (128, 28), (256, 14), (512, 7))] if want_features else []
        params = [p.detach() for _, p in self.named_parameters()]
        buffers = [t for _, t in self.named_buffers()]
        n_params, n_bn = L.irnet_sizes(*self._variant)
        ptab, btab = _Table(params, n_params), _Table(buffers, 3 * n_bn)
        io = L.ResnetIO()
        io.batch, io.size, io.x, io.emb = b, 112, x.data_ptr(), emb.data_ptr()
        for i, f in enumerate(feats):
            io.feat[i] = f.data_ptr()
        io.training, io.momentum, io.eps = 0, 0.1, 1e-5
        if ws is None:
            ws = ops.workspace(L.lib().crfr_irnet_workspace_bytes(*self._variant, b, 112))
        L.call("crfr_irnet_forward", self.engine, *self._variant, ptab.arr, btab.arr, C.byref(io), ws.data_ptr(), ws.numel(),
               ops.stream())
        return emb, feats, (ptab, btab), io

    def _run(self, x, want_features):
        self._check(x)
        if torch.is_grad_enabled() and x.requires_grad:
            outs = _IRInputGrad.apply(self, want_features, x)
            return outs[0], list(outs[1:])
        emb, feats, _, _ = self._launch(x.contiguous().float(), want_features)
        return emb, feats

    def forward(self, x):
        """ref: model_irse.py:167-172: the embedding only.  Differentiable with respect to ``x`` when
        ``x.requires_grad``; the parameters never receive a gradient."""
        return self._run(x, False)[0]

    def forward_features(self, x):
        """(embedding, x1, x2, x3, x4): the outputs of the four body stages next to the embedding - the tuple
        distill_main.py:59 unpacks from its teacher, and the 'extracted layers' use of DISTILLATION/model/utils.py:36-52
        (perceptual features, SUPER_RESOLUTION/train_FHN.py:255-265)."""
        emb, feats = self._run(x, True)
        return (emb,) + tuple(feats)


class _IRInputGrad(torch.autograd.Function):
    """IR / IR-SE forward whose backward is the native input gradient (``crfr_irnet_backward``).  The forward runs in a
    private workspace that keeps the saved activations for the backward; the parameters are constants of this function."""

    @staticmethod
    def forward(ctx, net, want_features, x):
        x = x.detach().contiguous().float()
        ws = torch.empty(L.lib().crfr_irnet_grad_workspace_bytes(*net._variant, x.shape[0], 112), dtype=torch.uint8,
                         device=x.device)
        emb, feats, tables, io = net._launch(x, want_features, ws)
        ctx.set_materialize_grads(False)
        ctx.saved = (net.engine, net._variant, tables, io, ws, x)   # x: io.x points at it
        return (emb,) + tuple(feats)

    @staticmethod
    @once_differentiable
    def backward(ctx, d_emb, *d_feats):
        engine, variant, (ptab, btab), io, ws, x = ctx.saved
        keep = []

        def ptr(g):
            if g is None:
                return None
            g = g.contiguous().float()
            keep.append(g)
            return g.data_ptr()
        dfeat = (C.c_void_p * 4)(*([ptr(g) for g in d_feats] + [None] * (4 - len(d_feats))))
        dx = torch.empty_like(x)
        L.call("crfr_irnet_backward", engine, *variant, ptab.arr, btab.arr, C.byref(io), ptr(d_emb), dfeat, dx.data_ptr(),
               ws.data_ptr(), ws.numel(), ops.stream())
        return None, None, dx


def IR_50(input_size):
    """Constructs a ir-50 model (ref: model_irse.py:191-197)."""
    return Backbone(input_size, 50, "ir")


def IR_101(input_size):
    """Constructs a ir-101 model (ref: model_irse.py IR_101)."""
    return Backbone(input_size, 100, "ir")


def IR_152(input_size):
    """Constructs a ir-152 model (ref: model_irse.py IR_152)."""
    return Backbone(input_size, 152, "ir")


def IR_SE_50(input_size):
    """Constructs a ir_se-50 model (ref: model_irse.py IR_SE_50)."""
    return Backbone(input_size, 50, "ir_se")


def IR_SE_101(input_size):
    """Constructs a ir_se-101 model (ref: model_irse.py IR_SE_101)."""
    return Backbone(input_size, 100, "ir_se")


def IR_SE_152(input_size):
    """Constructs a ir_se-152 model (ref: model_irse.py IR_SE_152)."""
    return Backbone(input_size, 152, "ir_se")
