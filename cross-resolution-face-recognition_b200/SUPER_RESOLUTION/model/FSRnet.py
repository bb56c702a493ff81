"""Drop-in for the reference's SUPER_RESOLUTION/model/FSRnet.py:251-416: the newer face-hallucination network the authors
trained on CelebA-HQ (SURVEY 8f-2) - ReflectionPad convolutions, non-affine InstanceNorm + ReLU, stride-2 encoder /
transposed-conv decoder stages, a prior network of four depth-4 hourglasses of pre-activation Bottleneck blocks, Tanh
image heads.

Same class names, constructor arguments, ``nn.Sequential`` indices and parameter names (identical ``state_dict`` keys;
the parameter-free layers - ReflectionPad2d, InstanceNorm2d, ReLU, Tanh - are kept as containers so the indices match),
same ``forward`` signatures.  ``forward`` never calls the torch layers: every op is a native kernel through
``crfr_b200.functional`` (tcgen05 implicit GEMM for the 3x3 stride-1 convolutions, padding 0 or 1; the lowered tcgen05
recipes for the stride-2, 7x7, 1x1, transposed and 3-channel ones; CUDA cores only for the 13- and 68-channel 1x1 prior heads
and the 3x3 stem's input gradient; fused InstanceNorm + ReLU / PReLU / residual passes, reflection-pad gathers, hourglass
pooling).  Activations are NHWC bf16 between ops; module inputs and outputs are fp32 NCHW.

The reference's ``OverallNetwork`` of this file cannot be constructed (it names a class ``Course_SR_Network`` that the
file does not define, :449; SURVEY Appendix C); ``SRNetwork`` below is that wiring with the classes that do exist
(coarse image -> encoder and prior network -> concatenation -> decoder), the one ``train_FHN.py`` drives by hand.
"""
import torch
import torch.nn as nn

from ... import functional as Fn


def _check(x, channels):
    if not x.is_cuda:
        raise RuntimeError("crfr_b200 SUPER_RESOLUTION networks need CUDA tensors: the hot path has no CPU fallback")
    if x.dim() != 4 or x.shape[1] != channels:
        raise ValueError("expected [B,%d,H,W], got %s" % (channels, tuple(x.shape)))


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

    def run(self, x):
        y = Fn.conv2d(x, self.conv1.weight, None, 1, 1)
        a, _ = Fn.norm_act(y, self.in1.weight, self.in1.bias, alpha=self.relu.weight)
        y = Fn.conv2d(a, self.conv2.weight, None, 1, 1)
        return Fn.norm_act(y, self.in2.weight, self.in2.bias, res=x)[0]


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

    def run(self, x):
        a, _ = Fn.norm_act(x, relu=True)
        y = Fn.conv2d(a, self.conv1.weight, self.conv1.bias, 1, 0)
        a, _ = Fn.norm_act(y, relu=True)
        y = Fn.conv2d(a, self.conv2.weight, self.conv2.bias, self.stride, 1)
        a, _ = Fn.norm_act(y, relu=True)
        y = Fn.conv2d(a, self.conv3.weight, self.conv3.bias, 1, 0)
        return Fn.add(y, x)


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

    @staticmethod
    def _seq(seq, x):
        for blk in seq:
            x = blk.run(x)
        return x

    def _forward(self, n, x):
        up1 = self._seq(self.hg[n - 1][0], x)
        low1 = self._seq(self.hg[n - 1][1], Fn.max_pool2(x))
        low2 = self._forward(n - 1, low1) if n > 1 else self._seq(self.hg[n - 1][3], low1)
        low3 = self._seq(self.hg[n - 1][2], low2)
        return Fn.up2_add(up1, low3)

    def run(self, x):
        return self._forward(self.depth, x)


def _pad_conv(x, conv, pad, stride=1, c=None):
    return Fn.conv2d(Fn.reflect_pad(x, pad, c), conv.weight, None, stride, 0)


def _down_stage(seq, i, x):
    """ReflectionPad(1) conv3x3 s2, ReflectionPad(1) conv3x3 s1, InstanceNorm, ReLU  (six Sequential entries from i)."""
    y = _pad_conv(x, seq[i + 1], 1, 2)
    y = _pad_conv(y, seq[i + 3], 1, 1)
    return Fn.norm_act(y, relu=True)[0]


def _up_stage(seq, i, x):
    """ConvTranspose2d(3, 2, 1, 1), ReflectionPad(1) conv3x3, InstanceNorm, ReLU  (five Sequential entries from i)."""
    y = Fn.conv_transpose2d(x, seq[i].weight, 2, 1, 1)
    y = _pad_conv(y, seq[i + 2], 1, 1)
    return Fn.norm_act(y, relu=True)[0]


def _image_head(seq, x):
    """ReflectionPad(1), conv3x3 -> 3 channels, Tanh; returns fp32 NCHW."""
    y = Fn.conv2d(Fn.reflect_pad(x, 1), seq[1].weight, None, 1, 0)
    return Fn.tanh(Fn.to_nchw(y, 3))


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


def _run_trunk(seq, i, x, n_blocks):
    """Runs the body built by _trunk starting at Sequential index i."""
    x = _down_stage(seq, i, x)
    x = _down_stage(seq, i + 6, x)
    for b in range(n_blocks):
        x = seq[i + 12 + b].run(x)
    j = i + 12 + n_blocks
    x = _up_stage(seq, j, x)
    return _up_stage(seq, j + 5, x)


class Coarse_SR_Network(nn.Module):
    """ref: :251-301; forward(x) -> coarse image [B,3,H,W]."""

    def __init__(self, ngf=64, n_blocks=6):
        super().__init__()
        stem = [nn.ReflectionPad2d(3), nn.Conv2d(3, ngf, 7, 1, 0, bias=False), nn.InstanceNorm2d(ngf), nn.ReLU(True)]
        self.model = nn.Sequential(*_trunk(ngf, n_blocks, stem))
        self.out = nn.Sequential(nn.ReflectionPad2d(1), nn.Conv2d(ngf, 3, 3, 1, 0, bias=False), nn.Tanh())
        self.n_blocks = n_blocks

    def features(self, x4):
        y = _pad_conv(x4, self.model[1], 3, 1, c=3)
        a, _ = Fn.norm_act(y, relu=True)
        return _run_trunk(self.model, 4, a, self.n_blocks)

    def forward(self, x):
        _check(x, 3)
        return _image_head(self.out, self.features(Fn.to_nhwc(x.float())))


class Fine_SR_Encoder(nn.Module):
    """ref: :304-346; forward(x) -> features [B,ngf,H,W]."""

    def __init__(self, ngf=64, n_blocks=6):
        super().__init__()
        stem = [nn.ReflectionPad2d(1), nn.Conv2d(3, ngf, 3, 1, 0, bias=False)]
        self.model = nn.Sequential(*_trunk(ngf, n_blocks, stem))
        self.n_blocks, self.ngf = n_blocks, ngf

    def features(self, x4):
        y = _pad_conv(x4, self.model[1], 1, 1, c=3)          # no norm / activation behind the first conv (:315-316)
        return _run_trunk(self.model, 2, y, self.n_blocks)

    def forward(self, x):
        _check(x, 3)
        return Fn.to_nchw(self.features(Fn.to_nhwc(x.float())))


class Prior_Estimation_Network(nn.Module):
    """ref: :349-376; forward(x) -> (features, landmark_out, parsing_out)."""

    def __init__(self, n_hourglass=4, n_blocks=2, ngf=64, parsing_classes=13, num_landmark=68):
        super().__init__()
        self.fc = nn.Conv2d(ngf, parsing_classes, kernel_size=1, bias=True)
        self.fc_landmark = nn.Conv2d(ngf, num_landmark, kernel_size=1, bias=False)
        model = [nn.ReflectionPad2d(3), nn.Conv2d(3, ngf, 7, 1, 0, bias=False), nn.InstanceNorm2d(ngf), nn.ReLU(True)]
        model += [_Residual_Block(ngf) for _ in range(n_blocks)]
        model += [Hourglass(planes=ngf, depth=4, block=Bottleneck, num_blocks=3) for _ in range(n_hourglass)]
        self.model = nn.Sequential(*model)

    def features(self, x4):
        y = _pad_conv(x4, self.model[1], 3, 1, c=3)
        a, _ = Fn.norm_act(y, relu=True)
        for m in list(self.model)[4:]:
            a = m.run(a)
        return a

    def forward(self, x):
        _check(x, 3)
        f = self.features(Fn.to_nhwc(x.float()))
        parsing = Fn.to_nchw(Fn.conv2d(f, self.fc.weight, self.fc.bias, 1, 0), self.fc.out_channels)
        landmark = Fn.to_nchw(Fn.conv2d(f, self.fc_landmark.weight, None, 1, 0), self.fc_landmark.out_channels)
        return Fn.to_nchw(f), landmark, parsing


class Fine_SR_Decoder(nn.Module):
    """ref: :379-416; forward(x [B,ngf,H,W]) -> image [B,3,H,W]."""

    def __init__(self, ngf=128, n_blocks=6):
        super().__init__()
        self.model = nn.Sequential(*_trunk(ngf, n_blocks, []))
        self.out = nn.Sequential(nn.ReflectionPad2d(1), nn.Conv2d(ngf, 3, 3, 1, 0, bias=False), nn.Tanh())
        self.n_blocks, self.ngf = n_blocks, ngf

    def run(self, x):
        return _image_head(self.out, _run_trunk(self.model, 0, x, self.n_blocks))

    def forward(self, x):
        _check(x, self.ngf)
        return self.run(Fn.to_nhwc(x.float()))


class SRNetwork(nn.Module):
    """The wiring the reference's (unconstructible, :449) ``OverallNetwork`` of this file describes, with the classes that
    exist: coarse image -> encoder and prior network -> cat(prior, encoder) -> decoder;
    forward(x) -> (coarse_out, out, landmark_out, parsing_out).  All activations stay NHWC bf16 between the sub-networks."""

    def __init__(self):
        super().__init__()
        self._coarse_sr_network = Coarse_SR_Network()
        self._prior_estimation_network = Prior_Estimation_Network()
        self._fine_sr_encoder = Fine_SR_Encoder()
        self._fine_sr_decoder = Fine_SR_Decoder()

    def forward(self, x):
        coarse = self._coarse_sr_network(x)
        c4 = Fn.to_nhwc(coarse)
        enc = self._fine_sr_encoder.features(c4)
        p = self._prior_estimation_network
        pe = p.features(c4)
        parsing = Fn.to_nchw(Fn.conv2d(pe, p.fc.weight, p.fc.bias, 1, 0), p.fc.out_channels)
        landmark = Fn.to_nchw(Fn.conv2d(pe, p.fc_landmark.weight, None, 1, 0), p.fc_landmark.out_channels)
        cat = torch.cat((pe, enc), 3)                    # channel concat = last NHWC axis
        out = self._fine_sr_decoder.run(cat)
        return coarse, out, landmark, parsing
