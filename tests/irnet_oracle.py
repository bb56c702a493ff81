"""CPU oracle of the IR / IR-SE teachers (IR_50 / 101 / 152, IR_SE_50 / 101 / 152 of DISTILLATION/model/model_irse.py,
face.evoLVe) in eval mode.  TEST INFRASTRUCTURE ONLY.

It extends ``oracle.resnet_oracle`` (whose ``build_ir50_state_dict`` / ``ir50_forward`` stay the pinned IR_50 oracle) to
every depth and to the squeeze-excitation unit:
  * ``bottleneck_IR_SE`` = ``bottleneck_IR`` whose ``res_layer`` ends in ``SEModule(depth, 16)``:
    x * sigmoid(fc2(relu(fc1(mean_hw(x))))), fc1 / fc2 1x1 convolutions without bias, fc1 xavier-initialised when the
    module is built (so seeded construction consumes those draws too);
  * ``get_blocks``: 50 = (3, 4, 14, 3), 100 = (3, 13, 30, 3), 152 = (3, 8, 36, 3) units per stage.
With ``irnet_forward(..., pr=Precision("bf16"))`` the SE unit works as the native program does: fp32 on the stored
res_layer.3 output, and the unit output (shortcut + e * BN(y)) is rounded once.
"""
from collections import OrderedDict

import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle.fsrnet_oracle import FP32
from oracle.resnet_oracle import BN_EPS, PLANES, _bn, _conv

IR_UNITS = {50: (3, 4, 14, 3), 100: (3, 13, 30, 3), 152: (3, 8, 36, 3)}
SE_REDUCTION = 16


def irnet_block_specs(num_layers):
    """(in_channel, depth, stride) of the bottleneck units, model_irse.py:96-126."""
    specs, in_ch = [], 64
    for units, depth in zip(IR_UNITS[num_layers], PLANES):
        for u in range(units):
            specs.append((in_ch, depth, 2 if u == 0 else 1))
            in_ch = depth
    return specs


def stage_ends(num_layers):
    """Index of the last unit of each stage: (2, 6, 20, 23) for 50 layers, (2, 15, 45, 48) for 100, (2, 10, 46, 49) for 152."""
    ends, n = [], 0
    for u in IR_UNITS[num_layers]:
        n += u
        ends.append(n - 1)
    return tuple(ends)


def build_irnet_state_dict(seed, num_layers, se):
    """state_dict of a freshly constructed ``Backbone([112, 112], num_layers, "ir_se" if se else "ir")`` (reference key
    order, draw-for-draw identical init)."""
    torch.manual_seed(seed)
    mods = OrderedDict()
    mods["input_layer.0"] = nn.Conv2d(3, 64, 3, 1, 1, bias=False)
    mods["input_layer.1"] = nn.BatchNorm2d(64)
    mods["input_layer.2"] = nn.PReLU(64)
    mods["output_layer.0"] = nn.BatchNorm2d(512)
    mods["output_layer.3"] = nn.Linear(512 * 7 * 7, 512)
    mods["output_layer.4"] = nn.BatchNorm1d(512)
    for i, (cin, d, stride) in enumerate(irnet_block_specs(num_layers)):
        p = "body.%d." % i
        if cin != d:
            mods[p + "shortcut_layer.0"] = nn.Conv2d(cin, d, 1, stride, bias=False)
            mods[p + "shortcut_layer.1"] = nn.BatchNorm2d(d)
        mods[p + "res_layer.0"] = nn.BatchNorm2d(cin)
        mods[p + "res_layer.1"] = nn.Conv2d(cin, d, 3, 1, 1, bias=False)
        mods[p + "res_layer.2"] = nn.PReLU(d)
        mods[p + "res_layer.3"] = nn.Conv2d(d, d, 3, stride, 1, bias=False)
        mods[p + "res_layer.4"] = nn.BatchNorm2d(d)
        if se:                                # SEModule(depth, 16).__init__
            mods[p + "res_layer.5.fc1"] = nn.Conv2d(d, d // SE_REDUCTION, 1, padding=0, bias=False)
            nn.init.xavier_uniform_(mods[p + "res_layer.5.fc1"].weight.data)
            mods[p + "res_layer.5.fc2"] = nn.Conv2d(d // SE_REDUCTION, d, 1, padding=0, bias=False)
    for m in mods.values():                   # model_irse.py:174-188
        if isinstance(m, (nn.Conv2d, nn.Linear)):
            nn.init.xavier_uniform_(m.weight.data)
            if m.bias is not None:
                m.bias.data.zero_()
        elif isinstance(m, (nn.BatchNorm2d, nn.BatchNorm1d)):
            m.weight.data.fill_(1)
            m.bias.data.zero_()
    sd = OrderedDict()
    for k, m in mods.items():
        for n, v in m.state_dict().items():
            sd[k + "." + n] = v.detach().clone()
    return sd


def variant_of(sd):
    """(num_layers, se) of an IR / IR-SE state_dict."""
    units = 1 + max(int(k.split(".")[1]) for k in sd if k.startswith("body."))
    num_layers = {sum(u): n for n, u in IR_UNITS.items()}[units]
    return num_layers, int("body.0.res_layer.5.fc1.weight" in sd)


def bn_affine(sd, p):
    """(s, t) of an eval-mode BatchNorm: BN(y) = s * y + t per channel."""
    s = sd[p + "weight"] / torch.sqrt(sd[p + "running_var"] + BN_EPS)
    return s, sd[p + "bias"] - sd[p + "running_mean"] * s


def se_from_pooled(sd, p, pooled):
    """SEModule of unit prefix p on its squeezed input pooled [B, C]: sigmoid(fc2(relu(fc1(pooled)))), fp32."""
    w1 = sd[p + "res_layer.5.fc1.weight"].flatten(1)
    w2 = sd[p + "res_layer.5.fc2.weight"].flatten(1)
    return torch.sigmoid(torch.relu(pooled @ w1.t()) @ w2.t())


def se_excitation(sd, p, y):
    """e [B, C] of unit prefix p from res_layer.3's output y, squeezed as the native program does:
    mean_hw(BN_4(y)) = s * mean_hw(y) + t."""
    s, t = bn_affine(sd, p + "res_layer.4.")
    return se_from_pooled(sd, p, y.mean(dim=(2, 3)) * s + t)


def irnet_forward(sd, x, pr=FP32, want_features=False):
    """Backbone.forward (model_irse.py:167-172) of any IR / IR-SE variant in eval mode -> embedding [B, 512]; with
    ``want_features`` also the outputs of the four body stages.  For an IR_50 state_dict it computes exactly what
    ``oracle.resnet_oracle.ir50_forward`` does."""
    num_layers, se = variant_of(sd)
    ends = stage_ends(num_layers)

    def prelu(y, a):
        a = a.view(1, -1, 1, 1)
        return pr.q(torch.clamp(y, min=0) + a * torch.clamp(y, max=0))

    def bn_prelu(y, p, a):   # BatchNorm (running statistics) + PReLU as one stored pass
        z = (y - sd[p + "running_mean"].view(1, -1, 1, 1)) / torch.sqrt(sd[p + "running_var"].view(1, -1, 1, 1) + BN_EPS)
        z = z * sd[p + "weight"].view(1, -1, 1, 1) + sd[p + "bias"].view(1, -1, 1, 1)
        a = a.view(1, -1, 1, 1)
        return pr.q(torch.clamp(z, min=0) + a * torch.clamp(z, max=0))

    feats = []
    a = _conv(pr, pr.q(x), sd["input_layer.0.weight"], 1, 1)
    a = bn_prelu(a, "input_layer.1.", sd["input_layer.2.weight"])
    for i, (cin, d, stride) in enumerate(irnet_block_specs(num_layers)):
        p = "body.%d." % i
        if cin != d:
            sc = _conv(pr, a, sd[p + "shortcut_layer.0.weight"], stride, 0)
            sc = _bn(pr, sd, p + "shortcut_layer.1.", sc, False, False)
        else:
            sc = a[:, :, ::stride, ::stride]                       # MaxPool2d(1, stride)
        r = _bn(pr, sd, p + "res_layer.0.", a, False, False)
        r = prelu(_conv(pr, r, sd[p + "res_layer.1.weight"], 1, 1), sd[p + "res_layer.2.weight"])
        r = _conv(pr, r, sd[p + "res_layer.3.weight"], stride, 1)
        if se:                                                     # res_layer.4 + SEModule + shortcut, one rounding
            s, t = bn_affine(sd, p + "res_layer.4.")
            z = r * s.view(1, -1, 1, 1) + t.view(1, -1, 1, 1)
            a = pr.st(pr.qg(z * se_from_pooled(sd, p, z.mean(dim=(2, 3)))[:, :, None, None] + sc))
        else:
            a = _bn(pr, sd, p + "res_layer.4.", r, False, False, res=sc)
        if i in ends:
            feats.append(a)
    o = _bn(pr, sd, "output_layer.0.", a, False, False)
    o = o.reshape(o.shape[0], -1)
    y = pr.qb(F.linear(pr.qg(o), pr.q(sd["output_layer.3.weight"]), sd["output_layer.3.bias"]))
    emb = _bn(pr, sd, "output_layer.4.", y, False, False)
    return (emb, feats) if want_features else emb
