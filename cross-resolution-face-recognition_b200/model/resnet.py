"""Drop-in ResNet face-embedding modules backed by the native sm_100a network program.

Mirror of the reference's operator interface for this path (model/resnet.py of the reference): same class names,
constructor arguments, sub-module / parameter / buffer names (identical ``state_dict`` keys), the same construction
and initialisation order (``torch.manual_seed(s); ResNet_34()`` draws identical weights) and the same
``forward(x) -> (embedding, x1, x2, x3, x4)``.  The torch layer objects are parameter / buffer containers only:
``forward`` runs the whole network in ``crfr_resnet34_forward`` and registers one autograd node whose backward is
``crfr_resnet34_backward``.  ``module.train()`` / ``module.eval()`` select batch statistics (with the running-statistics
update of nn.BatchNorm) or running statistics.  There is no eager / CPU fallback.

Only the configuration the reference can actually construct is native (SURVEY.md section 0.2): ``BasicBlock`` with
layers ``[3, 4, 6, 3]`` at 112x112, i.e. ``ResNet_34()`` - the student and the assistant of distill_main.py:202-203.
"""
import ctypes as C

import torch
import torch.nn as nn
from torch.nn import BatchNorm1d, BatchNorm2d, Conv2d, Dropout, Linear, MaxPool2d, Module, ReLU, Sequential

from .. import _lib as L
from .. import ops

__all__ = ["ResNet", "BasicBlock", "ResNet_34", "kd_train_step"]


def conv3x3(in_planes, out_planes, stride=1):
    """ref: model/resnet.py:9-12."""
    return nn.Conv2d(in_planes, out_planes, kernel_size=3, stride=stride, padding=1, bias=False)


def conv1x1(in_planes, out_planes, stride=1):
    """ref: model/resnet.py:13-16."""
    return Conv2d(in_planes, out_planes, kernel_size=1, stride=stride, bias=False)


class BasicBlock(nn.Module):
    """ref: model/resnet.py:18-47 (conv3x3 -> BN -> ReLU -> conv3x3 -> BN -> (+downsample(x)) -> ReLU)."""
    expansion = 1

    def __init__(self, inplanes, planes, stride=1, downsample=None):
        super().__init__()
        self.conv1 = conv3x3(inplanes, planes, stride)
        self.bn1 = nn.BatchNorm2d(planes)
        self.relu = nn.ReLU(inplace=True)
        self.conv2 = conv3x3(planes, planes)
        self.bn2 = nn.BatchNorm2d(planes)
        self.downsample = downsample
        self.stride = stride


class _TableOfPointers:
    def __init__(self, tensors, n):
        assert len(tensors) == n, (len(tensors), n)
        self.arr = (C.c_void_p * n)(*[None if t is None else t.data_ptr() for t in tensors])
        self.keep = tensors


def _io(x, emb, feats, training, momentum=0.1, eps=1e-5):
    io = L.ResnetIO()
    io.batch, io.size = x.shape[0], x.shape[2]
    io.x, io.emb = x.data_ptr(), emb.data_ptr()
    for i, f in enumerate(feats):
        io.feat[i] = None if f is None else f.data_ptr()
    io.training, io.momentum, io.eps = int(training), momentum, eps
    return io


class _ResNet34Function(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, engine, training, buffers, *params):
        x = x.contiguous().float()
        b, dev = x.shape[0], x.device
        emb = torch.empty((b, 512), dtype=torch.float32, device=dev)
        feats = [torch.empty((b, c, s, s), dtype=torch.float32, device=dev)
                 for c, s in ((64, 56), (128, 28), (256, 14), (512, 7))]
        need_grad = training and any(ctx.needs_input_grad[4:])
        nbytes = L.lib().crfr_resnet34_workspace_bytes(b, 112, 1 if training else 0)
        # a private workspace when a backward may follow: it holds the saved activations
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev) if need_grad else ops.workspace(nbytes)
        ptab = _TableOfPointers([p.detach() for p in params], L.RESNET34_NPARAMS)
        btab = _TableOfPointers(list(buffers), 3 * L.RESNET34_NBN)
        io = _io(x, emb, feats, training)
        L.call("crfr_resnet34_forward", engine, ptab.arr, btab.arr, C.byref(io), ws.data_ptr(), ws.numel(), ops.stream())
        ctx.engine, ctx.ws, ctx.x, ctx.outs = engine, ws, x, (emb, feats)
        ctx.save_for_backward(*params)
        return (emb,) + tuple(feats)

    @staticmethod
    def backward(ctx, d_emb, d1, d2, d3, d4):
        params = ctx.saved_tensors
        sizes = [p.numel() for p in params]
        offs, tot = [], 0
        for n in sizes:
            offs.append(tot)
            tot += (n + 3) // 4 * 4
        flat = torch.zeros(tot, dtype=torch.float32, device=ctx.x.device)
        grads = [flat[o:o + n].view(p.shape) for o, n, p in zip(offs, sizes, params)]
        ptab = _TableOfPointers([p.detach() for p in params], L.RESNET34_NPARAMS)
        gtab = _TableOfPointers(grads, L.RESNET34_NPARAMS)
        emb, feats = ctx.outs
        io = _io(ctx.x, emb, feats, True)

        def g(t):
            return None if t is None else t.contiguous().float()
        de = g(d_emb)
        df = [g(t) for t in (d1, d2, d3, d4)]
        dtab = (C.c_void_p * 4)(*[None if t is None else t.data_ptr() for t in df])
        L.call("crfr_resnet34_backward", ctx.engine, ptab.arr, gtab.arr, C.byref(io), ops.ptr(de), dtab,
               ctx.ws.data_ptr(), ctx.ws.numel(), ops.stream())
        return (None, None, None, None) + tuple(grads)


class ResNet(Module):
    """ref: model/resnet.py:152-225; forward(x) -> (x, x1, x2, x3, x4)."""

    def __init__(self, input_size, block, layers, zero_init_residual=True):
        super().__init__()
        assert input_size[0] in [112, 224], "input_size should be [112, 112] or [224, 224]"
        self.inplanes = 64
        self.conv1 = Conv2d(3, 64, kernel_size=7, stride=2, padding=3, bias=False)
        self.bn1 = BatchNorm2d(64)
        self.relu = ReLU(inplace=True)
        self.maxpool = MaxPool2d(kernel_size=3, stride=2, padding=1)
        self.layer1 = self._make_layer(block, 64, layers[0])
        self.layer2 = self._make_layer(block, 128, layers[1], stride=2)
        self.layer3 = self._make_layer(block, 256, layers[2], stride=2)
        self.layer4 = self._make_layer(block, 512, layers[3], stride=2)
        self.bn_o1 = BatchNorm2d(512)
        self.dropout = Dropout()
        if input_size[0] == 112:
            self.fc = Linear(25088, 512)
        else:
            self.fc = Linear(2048 * 8 * 8, 512)
        self.bn_o2 = BatchNorm1d(512)

        for m in self.modules():
            if isinstance(m, Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
            elif isinstance(m, BatchNorm2d):
                nn.init.constant_(m.weight, 1)
                nn.init.constant_(m.bias, 0)
        if zero_init_residual:
            for m in self.modules():
                if isinstance(m, BasicBlock):
                    nn.init.constant_(m.bn2.weight, 0)
        self.engine = L.ENGINE_AUTO
        self._native = (block is BasicBlock and list(layers) == [3, 4, 6, 3] and input_size[0] == 112)

    def _make_layer(self, block, planes, blocks, stride=1):
        downsample = None
        if stride != 1 or self.inplanes != planes * block.expansion:
            downsample = Sequential(conv1x1(self.inplanes, planes * block.expansion, stride),
                                    BatchNorm2d(planes * block.expansion))
        layers = [block(self.inplanes, planes, stride, downsample)]
        self.inplanes = planes * block.expansion
        for _ in range(1, blocks):
            layers.append(block(self.inplanes, planes))
        return Sequential(*layers)

    def ordered_parameters(self):
        return [p for _, p in self.named_parameters()]

    def ordered_buffers(self):
        return [b for _, b in self.named_buffers()]

    def forward(self, x):
        if not self._native:
            raise NotImplementedError("only ResNet(input_size=[112,112], BasicBlock, [3,4,6,3]) (= ResNet_34) has a "
                                      "native network program; it is also the only variant the reference can construct")
        if not x.is_cuda:
            raise RuntimeError("crfr_b200 ResNet needs a CUDA tensor: the hot path has no CPU fallback")
        if x.dim() != 4 or tuple(x.shape[1:]) != (3, 112, 112):
            raise ValueError("expected [B,3,112,112], got %s" % (tuple(x.shape),))
        params = self.ordered_parameters()
        return _ResNet34Function.apply(x, self.engine, self.training, tuple(self.ordered_buffers()), *params)


def ResNet_34(input_size=[112, 112]):
    """ref: model/resnet.py:231-236."""
    return ResNet(input_size, BasicBlock, [3, 4, 6, 3])


def _flat_grads(net):
    """A zeroed flat fp32 arena with one view per parameter (named_parameters order, 16-byte aligned)."""
    params = net.ordered_parameters()
    offs, tot = [], 0
    for p in params:
        offs.append(tot)
        tot += (p.numel() + 3) // 4 * 4
    flat = torch.zeros(tot, dtype=torch.float32, device=params[0].device)
    return params, [flat[o:o + p.numel()].view(p.shape) for o, p in zip(offs, params)]


def _is_ir50(net):
    """A native IR teacher: any of IR_50 / 101 / 152 and IR_SE_50 / 101 / 152 at 112 x 112."""
    from .model_irse import Backbone
    return isinstance(net, Backbone) and net._native


def _teacher_tables(teacher):
    """(params, buffers) tables of the teacher and its (num_layers, se) variant, or None for ResNet_34."""
    if _is_ir50(teacher):
        params = [p.detach() for _, p in teacher.named_parameters()]
        buffers = [t for _, t in teacher.named_buffers()]
        n_params, n_bn = L.irnet_sizes(*teacher._variant)
        return _TableOfPointers(params, n_params), _TableOfPointers(buffers, 3 * n_bn), teacher._variant
    return (_TableOfPointers([p.detach() for p in teacher.ordered_parameters()], L.RESNET34_NPARAMS),
            _TableOfPointers(teacher.ordered_buffers(), 3 * L.RESNET34_NBN), None)


def kd_workspace_bytes(teacher, batch):
    """Workspace of crfr_kd_train_step with this teacher (a native ResNet_34 or IR / IR-SE backbone)."""
    if _is_ir50(teacher):
        return L.lib().crfr_kd_workspace_bytes_ir(batch, 112, *teacher._variant)
    return L.lib().crfr_kd_workspace_bytes_ex(batch, 112, 0)


def check_kd_nets(teacher, student, assistant):
    if not ((isinstance(teacher, ResNet) and teacher._native) or _is_ir50(teacher)):
        raise NotImplementedError("the KD teacher must be a native ResNet_34 or a 112 x 112 IR / IR_SE backbone")
    for net in (student, assistant):
        if not (isinstance(net, ResNet) and net._native):
            raise NotImplementedError("the KD student and assistant must be native ResNet_34 modules")
    if teacher.training or not (student.training and assistant.training):
        raise RuntimeError("KD step: teacher.eval(), student.train(), assistant.train() expected (distill_main.py:41-43)")


def check_kd_input(x, name="x"):
    if not x.is_cuda or x.dim() != 4 or tuple(x.shape[1:]) != (3, 112, 112):
        raise ValueError("expected a CUDA tensor %s [B,3,112,112], got %s" % (name, tuple(x.shape)))
    return x.contiguous().float()


def kd_native_call(teacher, student, assistant, x_hr, x_lr, stabs, atabs, losses, assistant_grad_to_student=True,
                   events=None, ws=None):
    """crfr_kd_train_step on prepared tables: stabs / atabs = (params, buffers, grads) _TableOfPointers of the student and
    the assistant (gradients are ACCUMULATED into the grads tables)."""
    tp, tb, variant = _teacher_tables(teacher)
    b = x_hr.shape[0]
    io = L.KdIO()
    io.batch, io.size, io.x = b, 112, x_hr.data_ptr()
    io.x_lr = None if x_lr is None else x_lr.data_ptr()
    if variant is not None:
        io.teacher_ir50 = 1
        io.teacher_ir_layers, io.teacher_ir_se = variant
    io.momentum, io.eps, io.assistant_grad_to_student = 0.1, 1e-5, int(bool(assistant_grad_to_student))
    for i, e in enumerate(events or ()):
        io.events[i] = e.cuda_event
    need = kd_workspace_bytes(teacher, b)
    if ws is None or ws.numel() < need:
        ws = ops.workspace(need)
    L.call("crfr_kd_train_step", student.engine, tp.arr, tb.arr, stabs[0].arr, stabs[1].arr, stabs[2].arr, atabs[0].arr,
           atabs[1].arr, atabs[2].arr, C.byref(io), losses.data_ptr(), ws.data_ptr(), ws.numel(), ops.stream())


def kd_train_step(teacher, student, assistant, x, x_lr=None, assistant_grad_to_student=True):
    """The residual knowledge-distillation step of distill_main.py:59-74 as ONE native call (crfr_kd_train_step):
    teacher forward (eval), student and assistant forward (train, BatchNorm buffers updated), the MSE terms of
    distill_main.py:63,68-70 on the bf16 features in place, and both backward passes.

    ``x`` is the HR batch the teacher sees; the student and the assistant see ``x_lr`` when given ("HR teacher / LR
    student"), else ``x`` as well (what distill_main.py:59-61 does).  The teacher is a native ``ResNet_34`` or one of the
    IR / IR-SE backbones at 112 x 112 (``IR_50``, ``IR_SE_50``, ``IR_152``, ...: their four stage outputs are the t_k).

    Sets ``p.grad`` of the student to d(L_s [+ L_a])/dp and of the assistant to dL_a/dp (overwriting), and returns the
    device tensor ``(L_s, L_a)``.  Equivalent to ``(mse(s_emb, t_emb) + sum_k kd(t_k, s_k, a_k)).backward()`` through
    the drop-in modules, without the fp32 NCHW round trip of the five outputs of each network."""
    check_kd_nets(teacher, student, assistant)
    x = check_kd_input(x)
    if x_lr is not None:
        x_lr = check_kd_input(x_lr, "x_lr")
        if x_lr.shape[0] != x.shape[0]:
            raise ValueError("x and x_lr must hold the same number of images")
    sparams, sgrads = _flat_grads(student)
    aparams, agrads = _flat_grads(assistant)
    stabs = (_TableOfPointers([p.detach() for p in sparams], L.RESNET34_NPARAMS),
             _TableOfPointers(student.ordered_buffers(), 3 * L.RESNET34_NBN), _TableOfPointers(sgrads, L.RESNET34_NPARAMS))
    atabs = (_TableOfPointers([p.detach() for p in aparams], L.RESNET34_NPARAMS),
             _TableOfPointers(assistant.ordered_buffers(), 3 * L.RESNET34_NBN), _TableOfPointers(agrads, L.RESNET34_NPARAMS))
    losses = torch.empty((2,), dtype=torch.float32, device=x.device)
    kd_native_call(teacher, student, assistant, x, x_lr, stabs, atabs, losses, assistant_grad_to_student)
    for p, g in zip(sparams, sgrads):
        p.grad = g
    for p, g in zip(aparams, agrads):
        p.grad = g
    return losses
