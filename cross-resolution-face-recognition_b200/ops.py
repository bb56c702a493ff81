"""Tensor-level wrappers over the C-ABI (one function per entry point family).

PyTorch is only the owner of device memory and streams here: every function takes CUDA tensors, passes raw
pointers + the current stream to libcrfr.so and returns tensors allocated with torch.empty.  Activations are NHWC
bf16 tensors of shape [N, H, W, ld] (ld >= C, channel padding is explicit).
"""
import ctypes as C

import torch

from . import _lib as L

_WS = {}


def stream():
    return torch.cuda.current_stream().cuda_stream


def ptr(t):
    return None if t is None else t.data_ptr()


def workspace(nbytes, device=None):
    """A cached, growing scratch buffer per device (contents are never assumed to persist across calls)."""
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else device
    key = (device.type, device.index)
    buf = _WS.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _WS[key] = buf
    return buf


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("crfr_b200 ops need CUDA tensors (there is no CPU path)")


# ---------------------------------------------------------------------------------------------- layout
def nchw_to_nhwc(x, ld=None, zero_to=None):
    _need_cuda(x)
    n, c, h, w = x.shape
    ld = c if ld is None else ld
    zero_to = ld if zero_to is None else zero_to
    x = x.contiguous().float()
    out = torch.empty((n, h, w, ld), dtype=torch.bfloat16, device=x.device)
    L.call("crfr_nchw_f32_to_nhwc_bf16", ptr(x), ptr(out), n, c, h, w, ld, zero_to, stream())
    return out


def nhwc_to_nchw(x, c=None):
    _need_cuda(x)
    n, h, w, ld = x.shape
    c = ld if c is None else c
    out = torch.empty((n, c, h, w), dtype=torch.float32, device=x.device)
    L.call("crfr_nhwc_bf16_to_nchw_f32", ptr(x), ptr(out), n, c, h, w, ld, stream())
    return out


def pack_conv_weight(w, for_dgrad=False, transposed=False, s_pad=None):
    """fp32 Conv2d [cout,cin,k,k] (or ConvTranspose2d [cin,cout,k,k]) -> bf16 [k*k][R][s_pad]."""
    _need_cuda(w)
    w = w.contiguous().float()
    if not transposed:
        cout, cin, k, _ = w.shape
    else:
        cin, cout, k, _ = w.shape
    t = k * k
    if not transposed:
        r, s, rs, ss = (cout, cin, cin * t, t) if not for_dgrad else (cin, cout, t, cin * t)
    else:
        r, s, rs, ss = (cout, cin, t, cout * t) if not for_dgrad else (cin, cout, cout * t, t)
    if s_pad is None:
        s_pad = 4 if s < 8 else (s + 7) // 8 * 8
    out = torch.empty((t, r, s_pad), dtype=torch.bfloat16, device=w.device)
    L.call("crfr_pack_weight", ptr(w), ptr(out), t, r, s, s_pad, rs, ss, 1, stream())
    return out


# ---------------------------------------------------------------------------------------------- convolution
def conv_desc(x, cin, cout, k, stride, pad, transposed=False, out_hw=None, out_ld=None):
    n, h, w, ld = x.shape
    if not transposed:
        oh, ow = (h + 2 * pad - k) // stride + 1, (w + 2 * pad - k) // stride + 1
    else:
        oh, ow = out_hw
    out_ld = (cout if cout >= 8 else 4) if out_ld is None else out_ld
    return L.ConvDesc(n, h, w, cin, cout, k, stride, pad, oh, ow, ld, out_ld, 1 if transposed else 0)


def conv_fwd(x, w_packed, cin, cout, k, stride, pad, bias=None, engine=L.ENGINE_AUTO, transposed=False, out_hw=None,
             want_stats=False, nchw_out=False, eps=1e-5, out_ld=None):
    """Returns (y_nhwc_bf16 or None, y_nchw_f32 or None, stats [n,cout,2] or None)."""
    _need_cuda(x, w_packed, bias)
    d = conv_desc(x, cin, cout, k, stride, pad, transposed, out_hw, out_ld)
    y = None if nchw_out else torch.empty((d.n, d.oh, d.ow, d.out_ld), dtype=torch.bfloat16, device=x.device)
    yn = torch.empty((d.n, cout, d.oh, d.ow), dtype=torch.float32, device=x.device) if nchw_out else None
    stats = torch.empty((d.n, cout, 2), dtype=torch.float32, device=x.device) if want_stats else None
    wsb = L.lib().crfr_conv_workspace_bytes(C.byref(d))
    ws = workspace(wsb)
    L.call("crfr_conv_fwd", engine, C.byref(d), ptr(x), ptr(w_packed), w_packed.shape[2], ptr(bias), ptr(y), ptr(yn),
           ptr(stats), eps, ptr(ws), ws.numel(), stream())
    return y, yn, stats


def conv_dgrad(dy, w_packed_t, x_shape, cin, cout, k, stride, pad, engine=L.ENGINE_AUTO, transposed=False):
    """dy: NHWC bf16 [n,oh,ow,out_ld]; x_shape = (n,h,w,in_ld) of the gradient to produce."""
    _need_cuda(dy, w_packed_t)
    n, h, w, in_ld = x_shape
    d = L.ConvDesc(n, h, w, cin, cout, k, stride, pad, dy.shape[1], dy.shape[2], in_ld, dy.shape[3],
                   1 if transposed else 0)
    dx = torch.empty(x_shape, dtype=torch.bfloat16, device=dy.device)
    wsb = L.lib().crfr_conv_workspace_bytes(C.byref(d))
    ws = workspace(wsb)
    L.call("crfr_conv_dgrad", engine, C.byref(d), ptr(dy), ptr(w_packed_t), w_packed_t.shape[2], ptr(dx), ptr(ws),
           ws.numel(), stream())
    return dx


def conv_wgrad(x, dy, cin, cout, k, stride, pad, engine=L.ENGINE_AUTO, transposed=False, want_bias=False):
    """Returns (dw fp32 in the reference layout, dbias or None); fresh (zero-initialised) accumulators."""
    _need_cuda(x, dy)
    n, h, w, in_ld = x.shape
    d = L.ConvDesc(n, h, w, cin, cout, k, stride, pad, dy.shape[1], dy.shape[2], in_ld, dy.shape[3],
                   1 if transposed else 0)
    shape = (cout, cin, k, k) if not transposed else (cin, cout, k, k)
    dw = torch.zeros(shape, dtype=torch.float32, device=x.device)
    db = torch.zeros((cout,), dtype=torch.float32, device=x.device) if want_bias else None
    wsb = L.lib().crfr_conv_workspace_bytes(C.byref(d))
    ws = workspace(wsb)
    L.call("crfr_conv_wgrad", engine, C.byref(d), ptr(x), ptr(dy), ptr(dw), ptr(db), ptr(ws), ws.numel(), stream())
    return dw, db


def set_option(name, value):
    """Implementation switch for tests and profiles (crfr_set_option in include/crfr.h)."""
    L.call("crfr_set_option", name.encode(), int(value))


def engine_supported(engine, op, h, w, cin, cout, k, stride, pad):
    return bool(L.lib().crfr_conv_engine_supported(engine, op, h, w, cin, cout, k, stride, pad))


# ---------------------------------------------------------------------------------------------- norm + act
def _norm_ws(n, hw, c):
    return workspace(L.lib().crfr_norm_workspace_bytes(n, hw, c) + 1024)


def norm_stats(y, c=None, eps=1e-5, groups_as_batch=False):
    _need_cuda(y)
    n, h, w, ld = y.shape
    c = ld if c is None else c
    if groups_as_batch:      # BatchNorm: one statistic per channel over the whole batch
        n, hw = 1, n * h * w
    else:
        hw = h * w
    stats = torch.empty((n, c, 2), dtype=torch.float32, device=y.device)
    ws = _norm_ws(n, hw, c)
    L.call("crfr_norm_stats", ptr(y), n, hw, c, ld, eps, ptr(stats), ptr(ws), ws.numel(), stream())
    return stats


def norm_act_fwd(y, stats, gamma=None, beta=None, alpha=None, relu=False, res=None, c=None, batch_norm=False):
    _need_cuda(y, stats, gamma, beta, alpha, res)
    n, h, w, ld = y.shape
    c = ld if c is None else c
    out = torch.empty((n, h, w, c), dtype=torch.bfloat16, device=y.device)
    nn_, hw = (1, n * h * w) if batch_norm else (n, h * w)
    L.call("crfr_norm_act_fwd", ptr(y), ld, ptr(stats), ptr(gamma), ptr(beta), ptr(alpha), int(relu), ptr(res),
           8 if res is None else res.shape[3], ptr(out), c, nn_, hw, c, stream())
    return out


def norm_act_bwd(dout, y, stats, gamma=None, beta=None, alpha=None, relu=False, res=None, dout_b=None, c=None,
                 batch_norm=False):
    """Returns (dz, dy, dgamma, dbeta, dalpha): dz is the gradient w.r.t. the residual input."""
    _need_cuda(dout, y, stats)
    n, h, w, ld = y.shape
    c = ld if c is None else c
    dev = y.device
    # dz (gradient w.r.t. the residual input) is only produced when somebody can consume it
    dz = torch.empty((n, h, w, c), dtype=torch.bfloat16, device=dev) if (res is not None or dout_b is not None) else None
    dy = torch.empty((n, h, w, c), dtype=torch.bfloat16, device=dev)
    dg = torch.zeros((c,), dtype=torch.float32, device=dev) if gamma is not None else None
    db = torch.zeros((c,), dtype=torch.float32, device=dev) if beta is not None else None
    da = torch.zeros((c,), dtype=torch.float32, device=dev) if alpha is not None else None
    nn_, hw = (1, n * h * w) if batch_norm else (n, h * w)
    ws = _norm_ws(nn_, hw, c)
    L.call("crfr_norm_act_bwd", ptr(dout), dout.shape[3], ptr(dout_b), 8 if dout_b is None else dout_b.shape[3], ptr(y),
           ld, ptr(stats), ptr(gamma), ptr(beta), ptr(alpha), int(relu), ptr(res), 8 if res is None else res.shape[3],
           ptr(dz), c, ptr(dy), c, ptr(dg), ptr(db), ptr(da), nn_, hw, c, ptr(ws), ws.numel(), stream())
    return dz, dy, dg, db, da


def conv_dgrad_norm_bwd(dout, w_packed_t, y, stats, cin, cout, k, stride, pad, gamma=None, beta=None, alpha=None,
                        relu=False, res=None, dx_b=None, engine=L.ENGINE_AUTO):
    """Backward across `conv(act(norm(y) (+ res)))`: dgrad of the convolution + the normalisation backward in one call
    (crfr_conv_dgrad_norm_bwd).  dout: NHWC bf16 gradient of the convolution output; y: the raw map the normalisation
    read.  Returns (dz, dy, dgamma, dbeta, dalpha) as norm_act_bwd does (dz always produced)."""
    _need_cuda(dout, w_packed_t, y, stats)
    n, h, w, ld = y.shape
    c = cin
    d = L.ConvDesc(n, h, w, cin, cout, k, stride, pad, dout.shape[1], dout.shape[2], ld, dout.shape[3], 0)
    dev = y.device
    dz = torch.empty((n, h, w, c), dtype=torch.bfloat16, device=dev)
    dy = torch.empty((n, h, w, c), dtype=torch.bfloat16, device=dev)
    dg = torch.zeros((c,), dtype=torch.float32, device=dev) if gamma is not None else None
    db = torch.zeros((c,), dtype=torch.float32, device=dev) if beta is not None else None
    da = torch.zeros((c,), dtype=torch.float32, device=dev) if alpha is not None else None
    ws = workspace(L.lib().crfr_conv_dgrad_norm_bwd_workspace_bytes(C.byref(d)))
    L.call("crfr_conv_dgrad_norm_bwd", engine, C.byref(d), ptr(dout), ptr(w_packed_t), w_packed_t.shape[2], ptr(dx_b),
           8 if dx_b is None else dx_b.shape[3], ptr(y), ld, ptr(stats), ptr(gamma), ptr(beta), ptr(alpha), int(relu),
           ptr(res), 8 if res is None else res.shape[3], ptr(dz), c, ptr(dy), c, ptr(dg), ptr(db), ptr(da), ptr(ws),
           ws.numel(), stream())
    return dz, dy, dg, db, da


# ---------------------------------------------------------------------------------------------- resampling
def maxpool2_fwd(x):
    n, h, w, c = x.shape
    out = torch.empty((n, h // 2, w // 2, c), dtype=torch.bfloat16, device=x.device)
    L.call("crfr_maxpool2_fwd", ptr(x), c, ptr(out), c, n, h, w, c, stream())
    return out


def maxpool2_bwd(x, dout):
    n, h, w, c = x.shape
    dx = torch.empty_like(x)
    L.call("crfr_maxpool2_bwd", ptr(x), c, ptr(dout), c, ptr(dx), c, n, h, w, c, stream())
    return dx


def upnearest2_add_fwd(up, low):
    n, h, w, c = low.shape
    out = torch.empty_like(up)
    L.call("crfr_upnearest2_add_fwd", ptr(up), c, ptr(low), c, ptr(out), c, n, h, w, c, stream())
    return out


def upnearest2_bwd(dout):
    n, h2, w2, c = dout.shape
    dlow = torch.empty((n, h2 // 2, w2 // 2, c), dtype=torch.bfloat16, device=dout.device)
    L.call("crfr_upnearest2_bwd", ptr(dout), c, ptr(dlow), c, n, h2 // 2, w2 // 2, c, stream())
    return dlow


def add_n(a, b, c3=None):
    n, h, w, c = a.shape
    out = torch.empty_like(a)
    L.call("crfr_add_n", ptr(a), c, ptr(b), c, ptr(c3), c, ptr(out), c, n * h * w, c, stream())
    return out


# ---------------------------------------------------------------------------------------------- losses
def _loss_ws(n, hw):
    return workspace(4 * ((n * hw + 255) // 256) + 4096)


def loss_mse97(x, t, gscale=1.0, want_grad=True):
    _need_cuda(x, t)
    n, c, h, w = x.shape
    loss = torch.empty((1,), dtype=torch.float32, device=x.device)
    dx = torch.empty((n, h, w, 4 if c < 8 else c), dtype=torch.bfloat16, device=x.device) if want_grad else None
    ws = _loss_ws(n, h * w)
    L.call("crfr_loss_mse97", ptr(x.contiguous().float()), ptr(t.contiguous().float()), n, c, h * w, gscale, ptr(loss), ptr(dx),
           0 if dx is None else dx.shape[3], ptr(ws), ws.numel(), stream())
    return loss, dx


def loss_landmark(x, t, gscale=1.0, dx=None, coff=0):
    _need_cuda(x, t)
    n, c, h, w = x.shape
    loss = torch.empty((1,), dtype=torch.float32, device=x.device)
    ws = _loss_ws(n, h * w)
    L.call("crfr_loss_landmark", ptr(x.contiguous().float()), ptr(t.contiguous().float()), n, c, h * w, gscale, ptr(loss),
           ptr(dx), 0 if dx is None else dx.shape[3], coff, ptr(ws), ws.numel(), stream())
    return loss


def loss_ce2d(logits, target, gscale=1.0, dx=None, coff=0):
    _need_cuda(logits, target)
    n, c, h, w = logits.shape
    loss = torch.empty((1,), dtype=torch.float32, device=logits.device)
    ws = _loss_ws(n, h * w)
    L.call("crfr_loss_ce2d", ptr(logits.contiguous().float()), ptr(target.contiguous().long()), n, c, h * w, gscale, ptr(loss),
           ptr(dx), 0 if dx is None else dx.shape[3], coff, ptr(ws), ws.numel(), stream())
    return loss


def loss_kd(t, s, a, gscale=1.0, want=(False, True, True)):
    """mean(((t - s) - a)^2) and optional gradients (dt, ds, da); tensors all fp32 or all bf16, same shape."""
    _need_cuda(t, s, a)
    is_f32 = t.dtype == torch.float32
    loss = torch.empty((1,), dtype=torch.float32, device=t.device)
    outs = [torch.empty_like(t) if w else None for w in want]
    ws = workspace(4 * 148 * 16 + 4096)
    L.call("crfr_loss_kd", ptr(t), ptr(s), ptr(a), t.numel(), int(is_f32), gscale, ptr(loss), ptr(outs[0]),
           ptr(outs[1]), ptr(outs[2]), ptr(ws), ws.numel(), stream())
    return loss, outs


# ---------------------------------------------------------------------------------------------- optimiser
def rmsprop_step(p, g, sq, lr, alpha=0.99, eps=1e-8, weight_decay=0.0, gscale=1.0):
    _need_cuda(p, g, sq)
    L.call("crfr_rmsprop_step", ptr(p), ptr(g), ptr(sq), p.numel(), lr, alpha, eps, weight_decay, gscale, stream())


# ---------------------------------------------------------------------------------------------- bicubic
_TABLES = {}


def bicubic_table_host(in_size, out_size):
    import numpy as np
    n = L.lib().crfr_bicubic_table_size(in_size, out_size)
    tab = np.zeros(n, dtype=np.int32)
    L.call("crfr_bicubic_tables", in_size, out_size, tab.ctypes.data_as(C.c_void_p))
    return tab.reshape(out_size, -1)


def _table(in_size, out_size, device):
    key = (in_size, out_size, device.index)
    if key not in _TABLES:
        _TABLES[key] = torch.from_numpy(bicubic_table_host(in_size, out_size)).to(device)
    return _TABLES[key]


def bicubic_u8(src, out_h, out_w, want_f32=False):
    """src uint8 [N, H, W, C] -> (uint8 [N, out_h, out_w, C], optional fp32 NCHW normalised to [-1, 1])."""
    _need_cuda(src)
    n, ih, iw, c = src.shape
    src = src.contiguous()
    th, tw = _table(ih, out_h, src.device), _table(iw, out_w, src.device)
    tmp = torch.empty((n, ih, out_w, c), dtype=torch.uint8, device=src.device)
    dst = torch.empty((n, out_h, out_w, c), dtype=torch.uint8, device=src.device)
    f32 = torch.empty((n, c, out_h, out_w), dtype=torch.float32, device=src.device) if want_f32 else None
    L.call("crfr_bicubic_u8", ptr(src), n, ih, iw, c, ptr(th), ptr(tw), out_h, out_w, ptr(tmp), ptr(dst), ptr(f32),
           stream())
    return dst, f32


def landmark_heatmap(landmarks, h, w, sigma=1.3):
    """landmarks fp32 [N, K, 2] (x, y) -> heat-map fp32 [N, h, w] (helen_loader.py:118-143, s = 1.3 at :116)."""
    _need_cuda(landmarks)
    lm = landmarks.contiguous().float()
    n, k, _ = lm.shape
    hm = torch.empty((n, h, w), dtype=torch.float32, device=lm.device)
    L.call("crfr_landmark_heatmap", ptr(lm), n, k, float(sigma), h, w, ptr(hm), stream())
    return hm


def rotate_coeffs(h, w, angles):
    """Pillow's 16.16 fixed-point affine coefficients of Image.rotate(angle) for every angle: int32 [N, 6] (host)."""
    out = torch.empty((len(angles), 6), dtype=torch.int32)
    buf = (C.c_int32 * 6)()
    for i, a in enumerate(angles):
        L.call("crfr_rotate_coeffs", h, w, float(a), C.cast(buf, C.c_void_p))
        out[i] = torch.tensor(list(buf), dtype=torch.int32)
    return out


def augment_u8(src, angles, factors=None):
    """helen_loader.py:75-104 on the device: src uint8 [N, H, W, C] rotated by angles[i] degrees (PIL Image.rotate) and
    enhanced with ImageEnhance.Contrast once per column of factors [N, F] (None: rotation only)."""
    _need_cuda(src)
    n, h, w, c = src.shape
    src = src.contiguous()
    coef = rotate_coeffs(h, w, angles).to(src.device)
    fac = None if factors is None else torch.as_tensor(factors, dtype=torch.float32).reshape(n, -1).contiguous().to(src.device)
    dst = torch.empty_like(src)
    L.call("crfr_augment_u8", ptr(src), n, h, w, c, ptr(coef), ptr(fac), 0 if fac is None else fac.shape[1], ptr(dst),
           stream())
    return dst


def crop_u8(src, offsets_yx, out_h, out_w):
    """FHN_loader.py:61-63: per-image windows src[i, y0:y0+out_h, x0:x0+out_w] with (y0, x0) = offsets_yx[i]."""
    _need_cuda(src)
    n, h, w, c = src.shape
    off = torch.as_tensor(offsets_yx, dtype=torch.int32).reshape(n, 2)
    if int(off.min()) < 0 or int(off[:, 0].max()) + out_h > h or int(off[:, 1].max()) + out_w > w:
        raise ValueError("crop_u8: window outside the image")
    dst = torch.empty((n, out_h, out_w, c), dtype=torch.uint8, device=src.device)
    L.call("crfr_crop_u8", ptr(src.contiguous()), n, h, w, c, ptr(off.to(src.device)), out_h, out_w, ptr(dst), stream())
    return dst


# ---------------------------------------------------------------------------------------------- matcher
def l2norm_bf16(x):
    _need_cuda(x)
    x = x.contiguous().float()
    out = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    L.call("crfr_l2norm_bf16", ptr(x), ptr(out), x.shape[0], x.shape[1], stream())
    return out


def cosine_topk(probes, gallery, k, index_base=0, engine=L.ENGINE_AUTO):
    """probes/gallery: unit-norm bf16 [P, D] / [G, D] -> (scores fp32 [P, k], indices int32 [P, k])."""
    _need_cuda(probes, gallery)
    p, d = probes.shape
    g = gallery.shape[0]
    val = torch.empty((p, k), dtype=torch.float32, device=probes.device)
    idx = torch.empty((p, k), dtype=torch.int32, device=probes.device)
    wsb = L.lib().crfr_cosine_topk_workspace_bytes(p, g, d, k)
    ws = workspace(wsb)
    L.call("crfr_cosine_topk", engine, ptr(probes.contiguous()), ptr(gallery.contiguous()), p, g, d, k, index_base,
           ptr(val), ptr(idx), ptr(ws), ws.numel(), stream())
    return val, idx


def topk_merge(vals, idx, k):
    """vals/idx: [parts, P, k] -> merged (vals [P, k], idx [P, k])."""
    parts, p, kk = vals.shape
    assert kk == k
    ov = torch.empty((p, k), dtype=torch.float32, device=vals.device)
    oi = torch.empty((p, k), dtype=torch.int32, device=vals.device)
    L.call("crfr_topk_merge", ptr(vals.contiguous()), ptr(idx.contiguous()), parts, p, k, ptr(ov), ptr(oi), stream())
    return ov, oi


def pair_verify(e1, e2, thr):
    _need_cuda(e1, e2)
    n, d = e1.shape
    dist = torch.empty((n,), dtype=torch.float32, device=e1.device)
    same = torch.empty((n,), dtype=torch.uint8, device=e1.device)
    L.call("crfr_pair_verify", ptr(e1.contiguous().float()), ptr(e2.contiguous().float()), n, d, float(thr), ptr(dist),
           ptr(same), stream())
    return dist, same.bool()


def topk_rows(scores, k):
    """Row-wise top-k (k <= 8) of a materialised fp32 score matrix, ties -> lowest index."""
    _need_cuda(scores)
    scores = scores.contiguous().float()
    p, g = scores.shape
    val = torch.empty((p, k), dtype=torch.float32, device=scores.device)
    idx = torch.empty((p, k), dtype=torch.int32, device=scores.device)
    L.call("crfr_topk_rows", ptr(scores), p, g, k, ptr(val), ptr(idx), stream())
    return val, idx


def verify_sweep(dist, issame, thresholds, subset=None):
    """(tp, fp, tn, fn) of ``dist < t`` for every threshold t over the pairs in ``subset`` (int32 indices; None = all):
    int32 tensor [T, 4] on the device, one launch for the whole sweep (utils/utils.py:70-82)."""
    _need_cuda(dist, issame, thresholds, subset)
    d = dist.contiguous().float()
    s = issame.contiguous().to(torch.uint8)
    t = thresholds.contiguous().float()
    sub = None if subset is None else subset.contiguous().to(torch.int32)
    n = d.numel() if sub is None else sub.numel()
    counts = torch.empty((t.numel(), 4), dtype=torch.int32, device=d.device)
    L.call("crfr_verify_sweep", ptr(d), ptr(s), ptr(sub), n, ptr(t), t.numel(), ptr(counts), stream())
    return counts


def verify_counts(dist, issame, thr):
    """(tp, fp, tn, fn) of ``dist < thr`` against ``issame`` as a device int64 tensor of 4."""
    _need_cuda(dist, issame)
    counts = torch.empty((4,), dtype=torch.int64, device=dist.device)
    L.call("crfr_verify_counts", ptr(dist.contiguous().float()), ptr(issame.contiguous().to(torch.uint8)), dist.numel(),
           float(thr), ptr(counts), stream())
    return counts
