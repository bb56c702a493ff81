"""The SUPER_RESOLUTION FSRNet variant composed op by op from ``crfr_b200.functional``.  TEST AND MEASUREMENT
INFRASTRUCTURE ONLY.

Before the network program (csrc/srnet.cu) the modules of crfr_b200/SUPER_RESOLUTION/model/FSRnet.py ran this
composition: one autograd node per native op (about two thousand for ``SRNetwork``), every op packing its own weights
and allocating its own output.  It stays as the reference the program is compared against (tests/test_srnet_program_gpu.py)
and as the second arm of tools/bench_sr_variant.py.  Every function takes a module of that file and uses its parameters,
so autograd delivers the gradients into the module's ``.grad`` as the module's own forward does.
"""
import torch

from crfr_b200 import functional as Fn


def _res_block(m, x):
    """_Residual_Block :12-37: conv -> IN(affine) -> PReLU -> conv -> IN(affine) -> + x."""
    y = Fn.conv2d(x, m.conv1.weight, None, 1, 1)
    a, _ = Fn.norm_act(y, m.in1.weight, m.in1.bias, alpha=m.relu.weight)
    y = Fn.conv2d(a, m.conv2.weight, None, 1, 1)
    return Fn.norm_act(y, m.in2.weight, m.in2.bias, res=x)[0]


def _bottleneck(m, x):
    """Bottleneck :75-114: IN -> ReLU -> conv1x1 -> IN -> ReLU -> conv3x3 -> IN -> ReLU -> conv1x1, + x."""
    a, _ = Fn.norm_act(x, relu=True)
    y = Fn.conv2d(a, m.conv1.weight, m.conv1.bias, 1, 0)
    a, _ = Fn.norm_act(y, relu=True)
    y = Fn.conv2d(a, m.conv2.weight, m.conv2.bias, m.stride, 1)
    a, _ = Fn.norm_act(y, relu=True)
    y = Fn.conv2d(a, m.conv3.weight, m.conv3.bias, 1, 0)
    return Fn.add(y, x)


def _seq(seq, x):
    for blk in seq:
        x = _bottleneck(blk, x)
    return x


def _hourglass(m, n, x):
    """Hourglass :117-156."""
    up1 = _seq(m.hg[n - 1][0], x)
    low1 = _seq(m.hg[n - 1][1], Fn.max_pool2(x))
    low2 = _hourglass(m, n - 1, low1) if n > 1 else _seq(m.hg[n - 1][3], low1)
    low3 = _seq(m.hg[n - 1][2], low2)
    return Fn.up2_add(up1, low3)


def _pad_conv(x, conv, pad, stride=1, c=None):
    return Fn.conv2d(Fn.reflect_pad(x, pad, c), conv.weight, None, stride, 0)


def _down_stage(seq, i, x):
    y = _pad_conv(x, seq[i + 1], 1, 2)
    y = _pad_conv(y, seq[i + 3], 1, 1)
    return Fn.norm_act(y, relu=True)[0]


def _up_stage(seq, i, x):
    y = Fn.conv_transpose2d(x, seq[i].weight, 2, 1, 1)
    y = _pad_conv(y, seq[i + 2], 1, 1)
    return Fn.norm_act(y, relu=True)[0]


def _image_head(seq, x):
    y = Fn.conv2d(Fn.reflect_pad(x, 1), seq[1].weight, None, 1, 0)
    return Fn.tanh(Fn.to_nchw(y, 3))


def _run_trunk(seq, i, x, n_blocks):
    x = _down_stage(seq, i, x)
    x = _down_stage(seq, i + 6, x)
    for b in range(n_blocks):
        x = _res_block(seq[i + 12 + b], x)
    j = i + 12 + n_blocks
    x = _up_stage(seq, j, x)
    return _up_stage(seq, j + 5, x)


def coarse_features(m, x4):
    y = _pad_conv(x4, m.model[1], 3, 1, c=3)
    a, _ = Fn.norm_act(y, relu=True)
    return _run_trunk(m.model, 4, a, m.n_blocks)


def coarse(m, x):
    """Coarse_SR_Network.forward: fp32 NCHW image -> coarse image."""
    return _image_head(m.out, coarse_features(m, Fn.to_nhwc(x.float())))


def encoder_features(m, x4):
    y = _pad_conv(x4, m.model[1], 1, 1, c=3)
    return _run_trunk(m.model, 2, y, m.n_blocks)


def encoder(m, x):
    return Fn.to_nchw(encoder_features(m, Fn.to_nhwc(x.float())))


def prior_features(m, x4):
    y = _pad_conv(x4, m.model[1], 3, 1, c=3)
    a, _ = Fn.norm_act(y, relu=True)
    for blk in list(m.model)[4:]:
        a = _res_block(blk, a) if hasattr(blk, "conv1") else _hourglass(blk, blk.depth, a)
    return a


def prior_heads(m, f):
    parsing = Fn.to_nchw(Fn.conv2d(f, m.fc.weight, m.fc.bias, 1, 0), m.fc.out_channels)
    landmark = Fn.to_nchw(Fn.conv2d(f, m.fc_landmark.weight, None, 1, 0), m.fc_landmark.out_channels)
    return landmark, parsing


def prior(m, x):
    f = prior_features(m, Fn.to_nhwc(x.float()))
    landmark, parsing = prior_heads(m, f)
    return Fn.to_nchw(f), landmark, parsing


def decoder_run(m, x4):
    return _image_head(m.out, _run_trunk(m.model, 0, x4, m.n_blocks))


def decoder(m, x):
    return decoder_run(m, Fn.to_nhwc(x.float()))


def network(m, x):
    """SRNetwork.forward: coarse -> (encoder, prior) -> cat(prior, encoder) -> decoder."""
    c = coarse(m._coarse_sr_network, x)
    c4 = Fn.to_nhwc(c)
    enc = encoder_features(m._fine_sr_encoder, c4)
    p = m._prior_estimation_network
    pe = prior_features(p, c4)
    landmark, parsing = prior_heads(p, pe)
    out = decoder_run(m._fine_sr_decoder, torch.cat((pe, enc), 3))      # channel concat = last NHWC axis
    return c, out, landmark, parsing


SECTIONS = {"Coarse_SR_Network": coarse, "Fine_SR_Encoder": encoder, "Prior_Estimation_Network": prior,
            "Fine_SR_Decoder": decoder, "SRNetwork": network}


def run(m, x):
    """The composed forward of any module of the file (same outputs as its ``forward``)."""
    return SECTIONS[type(m).__name__](m, x)
