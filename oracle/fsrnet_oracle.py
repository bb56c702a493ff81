"""CPU oracle for the FSRNet face-hallucination path.  TEST INFRASTRUCTURE ONLY.

This file is a plain-PyTorch (CPU, fp32) restatement of the reference algorithm.  It is imported only by
``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl reference`` legs of ``bench.py``;
the product package never imports it.

Parity pin: the reference ships no tests or golden vectors (SURVEY.md section 8c), so the pin is live execution of
the reference's own modules.  ``oracle/make_golden.py`` (run in the build container, where ``/root/reference``
exists) checks every function here against the imported reference modules and writes ``tests/golden/*.npz``;
``tests/test_oracle_golden.py`` re-checks this file against those fixtures on any box.

Everything is written against a flat ``state_dict`` (name -> tensor) so the same weights can be loaded into the
reference modules, this oracle and the CUDA drop-in modules.

Reference sites restated (all paths relative to /root/reference):
  _Residual_Block            model/FSRnet.py:75-98
  BasicBlock (hourglass)     model/FSRnet.py:105-135
  Hourglass                  model/FSRnet.py:176-215
  Course_SR_Network          model/FSRnet.py:308-340
  Fine_SR_Encoder            model/FSRnet.py:342-379
  Prior_Estimation_Network   model/FSRnet.py:381-426
  Fine_SR_Decoder            model/FSRnet.py:428-459
  OverallNetwork             model/FSRnet.py:488-508 with the runnable wiring of :538-541 (SURVEY.md 8c-i)
  weights_init               FSR_main.py:38-58
  MSELossFunc                loss/loss.py:7-15
  MSELoss_Landmark           loss/loss.py:17-32
  CrossEntropyLoss2d         loss/loss.py:34-62
  loss composition           FSR_main.py:233-234
"""
import math
from collections import OrderedDict

import torch
import torch.nn.functional as F

EPS = 1e-5  # nn.InstanceNorm2d default


# ----------------------------------------------------------------------------------------------------------------
# parameter inventory (state_dict order of the reference OverallNetwork: 202 keys)
# ----------------------------------------------------------------------------------------------------------------
def _res_block_keys(prefix, c, cin=None):
    cin = c if cin is None else cin
    return [
        (prefix + "conv1.weight", (c, cin, 3, 3)),
        (prefix + "in1.weight", (c,)), (prefix + "in1.bias", (c,)),
        (prefix + "relu.weight", (c,)),
        (prefix + "conv2.weight", (c, c, 3, 3)),
        (prefix + "in2.weight", (c,)), (prefix + "in2.bias", (c,)),
        (prefix + "relu_out.weight", (c,)),
    ]


def fsrnet_param_shapes():
    """Ordered (name, shape) list, identical to ``OverallNetwork().state_dict()`` of the reference."""
    ks = []
    p = "_coarse_sr_network."
    ks += [(p + "conv_input.weight", (64, 3, 3, 3)), (p + "conv_input.bias", (64,)), (p + "relu.weight", (64,))]
    for b in range(3):
        ks += _res_block_keys(p + "residual.%d." % b, 64)
    ks += [(p + "conv_mid.weight", (3, 64, 3, 3)), (p + "conv_mid.bias", (3,)),
           (p + "bn_mid.weight", (64,)), (p + "bn_mid.bias", (64,)),
           (p + "bn_end.weight", (3,)), (p + "bn_end.bias", (3,))]
    p = "_prior_estimation_network."
    ks += [(p + "conv.weight", (128, 3, 7, 7)), (p + "conv.bias", (128,)),
           (p + "bn.weight", (128,)), (p + "bn.bias", (128,)), (p + "relu.weight", (128,))]
    for b in range(3):
        ks += _res_block_keys(p + "residual.%d." % b, 128)
    for b in range(3):
        ks += _res_block_keys(p + "residual_next.%d." % b, 128)
    for d in range(2):
        for s in range(4 if d == 0 else 3):
            for b in range(2):
                q = p + "hg.hg.%d.%d.%d." % (d, s, b)
                ks += [(q + "conv1.weight", (128, 128, 3, 3)), (q + "relu.weight", (128,)),
                       (q + "conv2.weight", (128, 128, 3, 3))]
    ks += [(p + "fc.weight", (11, 128, 1, 1)), (p + "fc.bias", (11,)),
           (p + "fc_landmark.weight", (97, 128, 1, 1)), (p + "fc_landmark.bias", (97,))]
    p = "_fine_sr_encoder."
    ks += [(p + "conv_input.weight", (64, 3, 7, 7)), (p + "conv_input.bias", (64,)), (p + "relu.weight", (64,))]
    for b in range(3):
        ks += _res_block_keys(p + "residual.%d." % b, 64)
    ks += [(p + "conv_mid.weight", (3, 64, 3, 3)), (p + "conv_mid.bias", (3,)),
           (p + "bn_mid.weight", (64,)), (p + "bn_mid.bias", (64,)),
           (p + "bn_end.weight", (3,)), (p + "bn_end.bias", (3,)),
           (p + "conv_end.weight", (64, 64, 3, 3)), (p + "conv_end.bias", (64,))]
    p = "_fine_sr_decoder."
    ks += [(p + "conv_input.weight", (64, 192, 3, 3)), (p + "conv_input.bias", (64,)), (p + "relu.weight", (64,)),
           (p + "bn_mid.weight", (64,)), (p + "bn_mid.bias", (64,)),
           (p + "deconv.weight", (64, 64, 7, 7)), (p + "deconv.bias", (64,))]
    for b in range(3):
        ks += _res_block_keys(p + "residual.%d." % b, 64)
    ks += [(p + "conv_out.weight", (3, 64, 3, 3)), (p + "conv_out.bias", (3,)),
           (p + "instance_norm.weight", (3,)), (p + "instance_norm.bias", (3,))]
    return ks


# Parameters that never influence the oracle-wiring outputs (SURVEY.md Appendix A: 888 789 dead parameters).
def fsrnet_dead_param(name):
    return (".bn_end." in name or ".residual_next." in name or name.startswith("_fine_sr_encoder.conv_mid")
            or ".instance_norm." in name)


# Conv biases that feed straight into an InstanceNorm: the mean subtraction cancels them, so their gradient is
# mathematically zero and the reference only produces rounding noise there (compare with an absolute tolerance).
FSRNET_NULL_GRAD = ("_coarse_sr_network.conv_input.bias", "_prior_estimation_network.conv.bias",
                    "_fine_sr_encoder.conv_input.bias", "_fine_sr_encoder.conv_end.bias",
                    "_fine_sr_decoder.conv_input.bias", "_fine_sr_decoder.deconv.bias")


# ----------------------------------------------------------------------------------------------------------------
# seeded initialisation: reproduces ``torch.manual_seed(s); OverallNetwork(); apply(weights_init)`` draw for draw
# ----------------------------------------------------------------------------------------------------------------
def _default_conv_init(shape, bias):
    """nn.Conv2d / nn.ConvTranspose2d ``reset_parameters`` (torch 2.x): consumes the global RNG identically."""
    w = torch.empty(shape)
    torch.nn.init.kaiming_uniform_(w, a=math.sqrt(5))
    b = None
    if bias:
        fan_in = shape[1] * shape[2] * shape[3]
        bound = 1.0 / math.sqrt(fan_in)
        b = torch.empty(shape[0])
        torch.nn.init.uniform_(b, -bound, bound)
    return w, b


def build_fsrnet_state_dict(seed=1234, xavier=True):
    """Weights as produced by the reference start-up code (FSR_main.py:128,131 with weights_init :38-58).

    Constructor order matters because every Conv2d draws from the global generator when it is built:
    Course_SR_Network (:308-322), Prior_Estimation_Network (:381-392), Fine_SR_Encoder (super().__init__ first,
    then its own members, :342-351), Fine_SR_Decoder (:428-441).  ``weights_init`` afterwards re-draws every
    nn.Conv2d weight with xavier_uniform_ in ``modules()`` order and zeroes conv biases; ConvTranspose2d is not an
    nn.Conv2d instance and keeps its default init.
    """
    torch.manual_seed(seed)
    sd = OrderedDict((k, None) for k, _ in fsrnet_param_shapes())
    shapes = dict(fsrnet_param_shapes())

    def conv(name, bias):
        w, b = _default_conv_init(shapes[name + ".weight"], bias)
        sd[name + ".weight"] = w
        if bias:
            sd[name + ".bias"] = b

    def const(name, v):
        sd[name] = torch.full(shapes[name], v)

    def res_block(prefix):
        conv(prefix + "conv1", False)
        const(prefix + "in1.weight", 1.0); const(prefix + "in1.bias", 0.0); const(prefix + "relu.weight", 0.25)
        conv(prefix + "conv2", False)
        const(prefix + "in2.weight", 1.0); const(prefix + "in2.bias", 0.0); const(prefix + "relu_out.weight", 0.25)

    def coarse_like(p, k_in):
        # members in the order Course_SR_Network.__init__ builds them
        if k_in == 3:
            conv(p + "conv_input", True)
        else:  # encoder: the inherited ctor first builds the 3x3 input conv, later replaced
            _default_conv_init((64, 3, 3, 3), True)
        const(p + "relu.weight", 0.25)
        for b in range(3):
            res_block(p + "residual.%d." % b)
        conv(p + "conv_mid", True)
        const(p + "bn_mid.weight", 1.0); const(p + "bn_mid.bias", 0.0)
        const(p + "bn_end.weight", 1.0); const(p + "bn_end.bias", 0.0)

    # --- OverallNetwork.__init__ (:491-494): coarse, prior, encoder, decoder ---
    coarse_like("_coarse_sr_network.", 3)

    p = "_prior_estimation_network."
    conv(p + "conv", True)
    const(p + "bn.weight", 1.0); const(p + "bn.bias", 0.0); const(p + "relu.weight", 0.25)
    for b in range(3):
        res_block(p + "residual.%d." % b)
    for b in range(3):
        res_block(p + "residual_next.%d." % b)
    for d in range(2):
        for s in range(4 if d == 0 else 3):
            for b in range(2):
                q = p + "hg.hg.%d.%d.%d." % (d, s, b)
                conv(q + "conv1", False); const(q + "relu.weight", 0.25); conv(q + "conv2", False)
    conv(p + "fc", True)
    conv(p + "fc_landmark", True)

    p = "_fine_sr_encoder."
    coarse_like(p, 7)                        # super().__init__()
    conv(p + "conv_input", True)             # 7x7 stride-4 stem replaces the inherited one
    const(p + "relu.weight", 0.25)
    const(p + "bn_mid.weight", 1.0); const(p + "bn_mid.bias", 0.0)
    for b in range(3):
        res_block(p + "residual.%d." % b)    # replaces the inherited residual stack
    conv(p + "conv_end", True)

    p = "_fine_sr_decoder."
    conv(p + "conv_input", True)
    const(p + "relu.weight", 0.25)
    const(p + "bn_mid.weight", 1.0); const(p + "bn_mid.bias", 0.0)
    w, b = _default_conv_init((64, 64, 7, 7), True)    # ConvTranspose2d weight is (in, out, kh, kw)
    sd[p + "deconv.weight"], sd[p + "deconv.bias"] = w, b
    for b_ in range(3):
        res_block(p + "residual.%d." % b_)
    conv(p + "conv_out", True)
    const(p + "instance_norm.weight", 1.0); const(p + "instance_norm.bias", 0.0)

    if xavier:
        # ``model.apply(weights_init)`` (FSR_main.py:131) calls weights_init on every sub-module in post-order, and
        # weights_init itself walks ``m.modules()`` (:45): every Conv2d is therefore re-drawn once per ancestor.
        # The final values come from the root's pass, but every earlier draw advances the generator, so the
        # whole recursion is replayed over the module tree (lists = containers, strings = Conv2d weights).
        def blocks(prefix, names=("residual",)):
            return [[[prefix + "%s.%d.conv1.weight" % (n, b), prefix + "%s.%d.conv2.weight" % (n, b)]
                     for b in range(3)] for n in names]
        pc, pp, pe, pd = ("_coarse_sr_network.", "_prior_estimation_network.", "_fine_sr_encoder.",
                          "_fine_sr_decoder.")
        hg = [[[[pp + "hg.hg.%d.%d.%d.conv1.weight" % (d, s_, b), pp + "hg.hg.%d.%d.%d.conv2.weight" % (d, s_, b)]
                for b in range(2)] for s_ in range(4 if d == 0 else 3)] for d in range(2)]
        tree = [
            [pc + "conv_input.weight"] + blocks(pc) + [pc + "conv_mid.weight"],
            [pp + "conv.weight"] + blocks(pp, ("residual", "residual_next")) + [[hg]]
            + [pp + "fc.weight", pp + "fc_landmark.weight"],
            [pe + "conv_input.weight"] + blocks(pe) + [pe + "conv_mid.weight", pe + "conv_end.weight"],
            [pd + "conv_input.weight"] + blocks(pd) + [pd + "conv_out.weight"],
        ]

        def convs(node):
            if isinstance(node, str):
                return [node]
            return [c for ch in node for c in convs(ch)]

        def draw(k):
            torch.nn.init.xavier_uniform_(sd[k])
            bk = k[:-6] + "bias"
            if bk in sd:
                sd[bk].zero_()

        def apply(node):
            if not isinstance(node, str):
                for ch in node:
                    apply(ch)
            for k in convs(node):
                draw(k)
        apply(tree)
    assert all(v is not None for v in sd.values())
    return sd


# ----------------------------------------------------------------------------------------------------------------
# storage-precision model
# ----------------------------------------------------------------------------------------------------------------
class _RoundFwd(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return x.to(torch.bfloat16).to(torch.float32)

    @staticmethod
    def backward(ctx, g):
        return g


class _RoundBwd(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        return g.to(torch.bfloat16).to(torch.float32)


class Precision:
    """Where the arithmetic is allowed to round.

    ``Precision("fp32")`` is the reference's arithmetic (every hook is the identity).  ``Precision("bf16")`` states
    the storage contract of the CUDA path (DESIGN.md "bf16 contract"): all accumulation, statistics, losses and
    parameters stay fp32, but every tensor that is STORED between two kernels is a bf16 tensor -
      q  : value rounded to bf16 when stored (network input, conv weights, conv outputs, activation outputs);
      qg : gradient rounded to bf16 when stored (gradient w.r.t. a conv input / conv output / pre-activation /
           upsampled branch / a tensor whose consumers' gradients are summed by an add kernel / loss gradients).
    With the hooks at exactly the storage points of the CUDA program, this oracle predicts its results up to
    fp32 summation order, which is what the 1e-2 bf16 tolerance of the parity tests is measured against.
    """

    def __init__(self, mode="fp32"):
        assert mode in ("fp32", "bf16")
        self.on = mode == "bf16"

    def q(self, x):
        return _RoundFwd.apply(x) if self.on else x

    def qg(self, x):
        return _RoundBwd.apply(x) if self.on else x

    def qb(self, x):
        return self.q(self.qg(x)) if self.on else x

    # storage points of ACTIVATIONS (conv outputs, normalise+PReLU outputs, hourglass sums).  Same rounding as q / qb;
    # kept apart from the weight / input roundings so that ``ForcedPrecision`` can substitute them.
    def st(self, x):
        return self.q(x)

    def sb(self, x):
        return self.st(self.qg(x)) if self.on else x


class ForcedPrecision(Precision):
    """Teacher-forced evaluation: the bf16 storage contract, but every stored ACTIVATION takes the value another
    implementation stored at that point (``feed``: the tensors in program order, fp32 NCHW), straight-through for the
    gradient.  Two things follow:
      * ``errors[i]`` = norm-wise relative deviation between the oracle's value computed from the forced inputs and
        the forced value: a per-layer forward check on identical inputs, for every layer of the network in place;
      * the backward pass runs on exactly the forward tensors of the other implementation.  Backward is linear once
        the forward is fixed, so parameter gradients must then agree to rounding noise - the chaotic amplification
        that limits free-running whole-network comparisons (tests/test_fsrnet_gpu.py) is gone, and a sequencing bug
        (a dropped weight-sharing accumulation, a wrong gradient slot) cannot hide behind it.
    """

    def __init__(self, feed):
        super().__init__("bf16")
        self.feed = list(feed)
        self.pos = 0
        self.errors = []        # ||computed - forced|| / ||forced||            (includes the bf16 rounding itself)
        self.errors_q = []      # ||bf16(computed) - forced|| / ||forced||      (0 unless a rounding flips)

    def st(self, x):
        assert self.pos < len(self.feed), "more storage points in the oracle than forced tensors"
        f = self.feed[self.pos]
        self.feed[self.pos] = None          # free as we go: the list holds GBs at 128 x 128
        self.pos += 1
        assert tuple(f.shape) == tuple(x.shape), (self.pos - 1, tuple(f.shape), tuple(x.shape))
        xd = x.detach()
        fn = f.double().norm().clamp_min(1e-30)
        self.errors.append(((xd - f).double().norm() / fn).item())
        self.errors_q.append(((xd.to(torch.bfloat16).to(torch.float32) - f).double().norm() / fn).item())
        return x + (f - xd)


class ForcedExact(ForcedPrecision):
    """Forced forward, NO gradient rounding: the exact (fp32) backward of the stored forward tensors.  The yardstick
    for how much deviation bf16 gradient storage itself causes (about 1e-3 per sqrt(stored gradient) along the chain:
    ~1.1e-2 after the ~180 roundings between the loss and the first coarse layer, profiles/r2_forced_gradient_depth.txt)."""

    def qg(self, x):
        return x


FP32 = Precision("fp32")


# ----------------------------------------------------------------------------------------------------------------
# forward restatement
# ----------------------------------------------------------------------------------------------------------------
def _inorm(x, w=None, b=None):
    # InstanceNorm2d: per-(n,c) biased variance over H*W, eps 1e-5, no running stats (train == eval).
    # F.instance_norm is what nn.InstanceNorm2d.forward calls (model/FSRnet.py:81,87,112,115 ...).
    return F.instance_norm(x, None, None, w, b, True, 0.0, EPS)


def _prelu(x, a):
    return F.prelu(x, a)


def _conv(pr, x, w, b=None, stride=1, pad=0, store=True):
    """Conv2d on a stored activation: bf16 weights, gradient w.r.t. the input stored, output stored (unless fp32)."""
    y = F.conv2d(pr.qg(x), pr.q(w), b, stride, pad)
    return pr.sb(y) if store else y


def _norm_act(pr, y, w=None, b=None, alpha=None, res=None):
    z = _inorm(y, w, b)
    if res is not None:
        z = z + res
    z = pr.qg(z)                       # gradient w.r.t. the pre-activation (== gradient of the residual input)
    return pr.st(_prelu(z, alpha) if alpha is not None else z)


def _res_block(pr, sd, p, x):
    y = _conv(pr, x, sd[p + "conv1.weight"], None, 1, 1)
    y = _norm_act(pr, y, sd[p + "in1.weight"], sd[p + "in1.bias"], sd[p + "relu.weight"])
    y = _conv(pr, y, sd[p + "conv2.weight"], None, 1, 1)
    return _norm_act(pr, y, sd[p + "in2.weight"], sd[p + "in2.bias"], sd[p + "relu_out.weight"], res=x)


def _res_stack(pr, sd, p, x, times):
    for _ in range(times):
        for b in range(3):
            x = _res_block(pr, sd, p + "residual.%d." % b, x)
    return x


def _hg_block(pr, sd, p, x):
    y = _conv(pr, x, sd[p + "conv1.weight"], None, 1, 1)
    y = _norm_act(pr, y, alpha=sd[p + "relu.weight"])
    y = _conv(pr, y, sd[p + "conv2.weight"], None, 1, 1)
    return _norm_act(pr, y, alpha=sd[p + "relu.weight"], res=x)


def _hg_seq(pr, sd, p, d, s, x):
    for b in range(2):
        x = _hg_block(pr, sd, p + "hg.hg.%d.%d.%d." % (d, s, b), x)
    return x


def _hourglass(pr, sd, p, n, x):
    x = pr.qg(x)                       # three consumers (block conv, its skip, the pool): their gradients are summed + stored
    up1 = _hg_seq(pr, sd, p, n - 1, 0, x)
    low1 = _hg_seq(pr, sd, p, n - 1, 1, F.max_pool2d(x, 2, 2))
    low2 = _hourglass(pr, sd, p, n - 1, low1) if n > 1 else _hg_seq(pr, sd, p, 0, 3, low1)
    low3 = _hg_seq(pr, sd, p, n - 1, 2, low2)
    out = up1 + F.interpolate(pr.qg(low3), scale_factor=2)      # default mode: nearest
    return pr.sb(out)


def coarse_forward(sd, x, p="_coarse_sr_network.", pr=FP32):
    y = _conv(pr, pr.q(x), sd[p + "conv_input.weight"], sd[p + "conv_input.bias"], 1, 1)
    y = _norm_act(pr, y, sd[p + "bn_mid.weight"], sd[p + "bn_mid.bias"], sd[p + "relu.weight"])
    y = _res_stack(pr, sd, p, y, 3)
    feat = _norm_act(pr, y, sd[p + "bn_mid.weight"], sd[p + "bn_mid.bias"])
    coarse = _conv(pr, feat, sd[p + "conv_mid.weight"], sd[p + "conv_mid.bias"], 1, 1, store=False)   # fp32 output
    return feat, pr.qg(coarse)         # loss + two stems: summed gradient is stored


def encoder_forward(sd, x, p="_fine_sr_encoder.", pr=FP32):
    y = _conv(pr, pr.q(x), sd[p + "conv_input.weight"], sd[p + "conv_input.bias"], 4, 3)
    y = _norm_act(pr, y, sd[p + "bn_mid.weight"], sd[p + "bn_mid.bias"], sd[p + "relu.weight"])
    y = _res_stack(pr, sd, p, y, 3)
    y = _conv(pr, y, sd[p + "conv_end.weight"], sd[p + "conv_end.bias"], 1, 1)
    return _norm_act(pr, y, sd[p + "bn_mid.weight"], sd[p + "bn_mid.bias"], sd[p + "relu.weight"])


def prior_forward(sd, x, p="_prior_estimation_network.", pr=FP32):
    y = _conv(pr, pr.q(x), sd[p + "conv.weight"], sd[p + "conv.bias"], 4, 3)
    y = _norm_act(pr, y, sd[p + "bn.weight"], sd[p + "bn.bias"], sd[p + "relu.weight"])
    y = _res_stack(pr, sd, p, y, 1)
    y = _hourglass(pr, sd, p, 2, y)
    # the two 1x1 heads (:391-392) evaluated as one 108-channel conv: same arithmetic, one stored input gradient
    w = torch.cat((sd[p + "fc.weight"], sd[p + "fc_landmark.weight"]), 0)
    b = torch.cat((sd[p + "fc.bias"], sd[p + "fc_landmark.bias"]), 0)
    heads = _conv(pr, y, w, b, store=False)
    return y, heads[:, 11:], heads[:, :11]


def decoder_forward(sd, x, p="_fine_sr_decoder.", pr=FP32):
    y = _conv(pr, x, sd[p + "conv_input.weight"], sd[p + "conv_input.bias"], 1, 1)
    y = _norm_act(pr, y, sd[p + "bn_mid.weight"], sd[p + "bn_mid.bias"], sd[p + "relu.weight"])
    y = pr.sb(F.conv_transpose2d(pr.qg(y), pr.q(sd[p + "deconv.weight"]), sd[p + "deconv.bias"], 4, 2, 1))
    y = _norm_act(pr, y, sd[p + "bn_mid.weight"], sd[p + "bn_mid.bias"], sd[p + "relu.weight"])
    y = _res_stack(pr, sd, p, y, 3)
    y = _norm_act(pr, y, sd[p + "bn_mid.weight"], sd[p + "bn_mid.bias"])
    return _conv(pr, y, sd[p + "conv_out.weight"], sd[p + "conv_out.bias"], 1, 1, store=False)


def fsrnet_forward(sd, x, pr=FP32):
    """OverallNetwork.forward with encoder / prior net fed by the 3-channel coarse image (SURVEY.md 8c-i)."""
    _, coarse = coarse_forward(sd, x, pr=pr)
    enc = encoder_forward(sd, coarse, pr=pr)
    pe, landmark, parsing = prior_forward(sd, coarse, pr=pr)
    out = decoder_forward(sd, torch.cat((pe, enc), 1), pr=pr)
    return coarse, out, landmark, parsing


# ----------------------------------------------------------------------------------------------------------------
# losses
# ----------------------------------------------------------------------------------------------------------------
def mse97(x, t):
    return ((x.float() - t.float()) ** 2).mean() * 97.0


def landmark_loss(x, t):
    s = x.sum(dim=1)
    return ((s.float() - t.float()) ** 2).mean() * 97.0


def ce2d(logits, target):
    return F.nll_loss(F.log_softmax(logits, 1), torch.squeeze(target))


def fsrnet_loss(outputs, hr, heatmap, labels, train_batch=None, w_pix=5.0, pr=FP32, out_grad=None):
    """``out_grad`` (optional, fp32 like ``out``): a further gradient at the output image, as another loss term adds it
    (the identity term of crfr_fsrnet_id_train_step): total gains sum(out * out_grad), not counted in ``parts``, and the
    output's gradient is stored once, with the pixel term's."""
    coarse, out, landmark, parsing = outputs
    b = hr.shape[0] if train_batch is None else train_batch
    out = pr.qg(out)
    parts = (mse97(out, hr), mse97(pr.qg(coarse), hr), landmark_loss(pr.qg(landmark), heatmap),
             ce2d(pr.qg(parsing), labels))
    total = (w_pix * parts[0] + w_pix * parts[1] + parts[2] + parts[3]) / (2.0 * b)
    if out_grad is not None:
        total = total + (out * out_grad).sum()
    return total, parts


def synthetic_batch(batch, size=128, seed=4321):
    """SURVEY.md 8d / Appendix E draw order: x, hr, labels, heat-map from one seeded generator."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(batch, 3, size, size, generator=g)
    hr = torch.randn(batch, 3, size, size, generator=g)
    lbl = torch.randint(0, 11, (batch, 1, size // 4, size // 4), generator=g)
    hm = torch.rand(batch, size // 4, size // 4, generator=g)
    return x, hr, lbl, hm


def fsrnet_loss_and_grads(sd, x, hr, hm, lbl, train_batch=None, precision="fp32", out_grad=None):
    """One forward+backward; returns (outputs, total, parts, {name: grad}) - used as the parity oracle.
    ``precision``: "fp32", "bf16" or a ``Precision`` instance (e.g. ``ForcedPrecision``); ``out_grad``: see
    ``fsrnet_loss``."""
    pr = precision if isinstance(precision, Precision) else Precision(precision)
    leaves = OrderedDict((k, v.detach().clone().requires_grad_(True)) for k, v in sd.items())
    outs = fsrnet_forward(leaves, x, pr)
    total, parts = fsrnet_loss(outs, hr, hm, lbl, train_batch, pr=pr, out_grad=out_grad)
    names = [k for k in leaves if not fsrnet_dead_param(k)]
    grads = torch.autograd.grad(total, [leaves[k] for k in names], allow_unused=True)
    gd = OrderedDict((k, None) for k in leaves)
    for k, g in zip(names, grads):
        gd[k] = g
    return [o.detach() for o in outs], total.detach(), [p.detach() for p in parts], gd


# ----------------------------------------------------------------------------------------------------------------
# Discriminator / OverallNetwork_GAN (model/FSRnet.py:461-486, 512-545)
# ----------------------------------------------------------------------------------------------------------------
def discriminator_param_shapes(spatial=56):
    ks = [("conv_input.weight", (64, 192, 3, 3)), ("conv_input.bias", (64,)), ("relu.weight", (64,)),
          ("bn_mid.weight", (64,)), ("bn_mid.bias", (64,))]
    for b in range(3):
        ks += _res_block_keys("residual.%d." % b, 64)
    ks += [("fc.weight", (512, 64 * spatial * spatial)), ("fc.bias", (512,)), ("bn_end.weight", (512,)), ("bn_end.bias", (512,))]
    return ks


def _batch_norm_train(x, w, b, dims, eps=1e-5):
    mu = x.mean(dim=dims, keepdim=True)
    var = ((x - mu) ** 2).mean(dim=dims, keepdim=True)
    shape = [1, -1] + [1] * (x.dim() - 2)
    return (x - mu) / torch.sqrt(var + eps) * w.view(shape) + b.view(shape)


def discriminator_forward(sd, x, p="", pr=FP32):
    """Discriminator.forward (:479-487) in training mode (batch statistics): conv -> BN -> PReLU -> the same BN -> flatten
    (NCHW order) -> Linear -> BatchNorm1d.  The residual stack is never called."""
    y = _conv(pr, pr.q(x), sd[p + "conv_input.weight"], sd[p + "conv_input.bias"], 1, 1)
    a = pr.st(_prelu(pr.qg(_batch_norm_train(y, sd[p + "bn_mid.weight"], sd[p + "bn_mid.bias"], (0, 2, 3))), sd[p + "relu.weight"]))
    a = pr.st(pr.qg(_batch_norm_train(a, sd[p + "bn_mid.weight"], sd[p + "bn_mid.bias"], (0, 2, 3))))
    o = a.reshape(a.shape[0], -1)
    o = pr.sb(F.linear(pr.qg(o), pr.q(sd[p + "fc.weight"]), sd[p + "fc.bias"]))
    return pr.st(pr.qg(_batch_norm_train(o, sd[p + "bn_end.weight"], sd[p + "bn_end.bias"], (0,))))


def gan_forward(sd, lr, hr, pr=FP32):
    """OverallNetwork_GAN.forward (:538-545) on a state dict with the _discriminator.* keys next to the sub-networks."""
    def once(x):
        enc = encoder_forward(sd, x, pr=pr)
        pe, landmark, parsing = prior_forward(sd, x, pr=pr)
        out = torch.cat((pe, enc), 1)
        return out, landmark, parsing, discriminator_forward(sd, out, "_discriminator.", pr)
    _, coarse = coarse_forward(sd, lr, pr=pr)
    out1, lm1, ps1, e1 = once(coarse)
    _, _, _, e2 = once(hr)
    return decoder_forward(sd, out1, pr=pr), coarse, lm1, ps1, e1, e2
