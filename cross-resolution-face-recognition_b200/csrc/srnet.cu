// Native network program for the SUPER_RESOLUTION FSRNet variant (SUPER_RESOLUTION/model/FSRnet.py:251-416): the
// four sub-networks and their SRNetwork wiring (coarse image -> encoder and prior network -> cat(prior, encoder) ->
// decoder) sequenced here in C++ on one stream, over a caller-provided workspace arena.
//
// The same scheme as fsrnet.cu: the forward records a tape of ops (reflection pad, convolution, InstanceNorm +
// ReLU / PReLU / residual, Bottleneck add, max-pool, nearest-up + add, concat-by-view, the combined prior heads, the
// Tanh image heads); the backward replays it in reverse.  A tensor with several consumers gets one gradient slot per
// consumer.  The arena is a deterministic bump allocator, so the backward entry point rebuilds the tape with a dry run
// of the forward and finds every saved activation at the same offset.  Every convolution goes through crfr_conv_fwd /
// crfr_conv_dgrad / crfr_conv_wgrad, so each layer keeps the routing the single-op path gives it.
#include <array>
#include <map>
#include <mutex>
#include <vector>

#include "common.cuh"
#include "crfr.h"
#include "internal.h"

namespace {

constexpr float kEps = 1e-5f;
constexpr int kParsing = 13, kLandmark = 68;   // Prior_Estimation_Network(parsing_classes=13, num_landmark=68)
constexpr int kHeads = kParsing + kLandmark;
constexpr int kHeadsN = 128;                   // the combined head GEMM's output width (rows kHeads.. are zero)
constexpr int kHeadsK = 64;                    // ngf of the prior network

// ---- parameter tables (state_dict order) ----------------------------------------------------------------------------
// _trunk: 4 down convolutions, 6 _Residual_Blocks of 7 tensors, 2 x (ConvTranspose2d, Conv2d)
constexpr int kTrunk = 50, kResBlock = 7, kHgParams = 234;   // Hourglass(depth 4): 13 sequences x 3 Bottlenecks x 6
constexpr int kCoarseN = 52, kEncoderN = 51, kPriorN = 954, kDecoderN = 51;
constexpr int kNetCoarse = 0, kNetPrior = kCoarseN, kNetEncoder = kNetPrior + kPriorN, kNetDecoder = kNetEncoder + kEncoderN;
static_assert(kNetDecoder + kDecoderN == CRFR_SRNET_NPARAMS, "SRNetwork parameter table");

int section_params(int section) {
  switch (section) {
    case CRFR_SRNET_COARSE: return kCoarseN;
    case CRFR_SRNET_ENCODER: return kEncoderN;
    case CRFR_SRNET_PRIOR: return kPriorN;
    case CRFR_SRNET_DECODER: return kDecoderN;
    case CRFR_SRNET_NETWORK: return CRFR_SRNET_NPARAMS;
  }
  return 0;
}

// ---- kernels of the combined prior heads and the Tanh image heads ----------------------------------------------------
// wc [kHeadsN][64] (rows 0..12 fc, 13..80 fc_landmark, rest zero) and bias bc [kHeadsN]; wtd [64][kHeadsN] (the
// transpose, for the input gradient) when not NULL
__global__ void sr_heads_pack_kernel(const float* __restrict__ w_fc, const float* __restrict__ b_fc,
                                     const float* __restrict__ w_lm, bf16* __restrict__ wc, float* __restrict__ bc,
                                     bf16* __restrict__ wtd) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= kHeadsN * kHeadsK) return;
  const int co = i / kHeadsK, ci = i % kHeadsK;
  float v = 0.f;
  if (co < kParsing) v = w_fc[co * kHeadsK + ci];
  else if (co < kHeads) v = w_lm[(co - kParsing) * kHeadsK + ci];
  const bf16 b = __float2bfloat16_rn(v);
  wc[i] = b;
  if (wtd) wtd[ci * kHeadsN + co] = b;
  if (ci == 0) bc[co] = co < kParsing ? b_fc[co] : 0.f;
}

// 32-pixel tiles of one image through shared memory: NHWC rows of kHeadsN <-> the two NCHW maps, both sides coalesced.
// dir 0: y fp32 [npix][kHeadsN] -> parsing [n][13][hw], landmark [n][68][hw];
// dir 1: d_parsing / d_landmark (either NULL = zero) -> g bf16 [npix][kHeadsN] (channels kHeads.. zero)
__global__ void sr_heads_scatter_kernel(int dir, const float* __restrict__ y, float* __restrict__ parsing,
                                        float* __restrict__ landmark, const float* __restrict__ d_parsing,
                                        const float* __restrict__ d_landmark, bf16* __restrict__ g, int hw) {
  __shared__ float tile[kHeadsN][33];
  const int img = blockIdx.y, p0 = blockIdx.x * 32;
  const long long row0 = (long long)img * hw + p0;
  if (dir == 0) {
    for (int i = threadIdx.x; i < 32 * kHeadsN; i += blockDim.x) {
      const int pp = i / kHeadsN, c = i % kHeadsN;
      if (p0 + pp < hw && c < kHeads) tile[c][pp] = y[(row0 + pp) * kHeadsN + c];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 32 * kHeads; i += blockDim.x) {
      const int c = i / 32, pp = i % 32;
      if (p0 + pp >= hw) continue;
      if (c < kParsing) parsing[((long long)img * kParsing + c) * hw + p0 + pp] = tile[c][pp];
      else landmark[((long long)img * kLandmark + c - kParsing) * hw + p0 + pp] = tile[c][pp];
    }
  } else {
    for (int i = threadIdx.x; i < 32 * kHeadsN; i += blockDim.x) {
      const int c = i / 32, pp = i % 32;
      float v = 0.f;
      if (p0 + pp < hw) {
        if (c < kParsing) { if (d_parsing) v = d_parsing[((long long)img * kParsing + c) * hw + p0 + pp]; }
        else if (c < kHeads) { if (d_landmark) v = d_landmark[((long long)img * kLandmark + c - kParsing) * hw + p0 + pp]; }
      }
      tile[c][pp] = v;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 32 * kHeadsN; i += blockDim.x) {
      const int pp = i / kHeadsN, c = i % kHeadsN;
      if (p0 + pp < hw) g[(row0 + pp) * kHeadsN + c] = __float2bfloat16_rn(tile[c][pp]);
    }
  }
}

// dW_fc [13][64] += G[ci][co], dW_fcl [68][64] += G[ci][13 + co]   (G = X^T dY [64][kHeadsN])
__global__ void sr_heads_unpack_kernel(const float* __restrict__ G, float* __restrict__ dw_fc, float* __restrict__ dw_lm) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= kHeads * kHeadsK) return;
  const int co = i / kHeadsK, ci = i % kHeadsK;
  const float g = G[ci * kHeadsN + co];
  if (co < kParsing) {
    if (dw_fc) dw_fc[co * kHeadsK + ci] += g;
  } else if (dw_lm) {
    dw_lm[(co - kParsing) * kHeadsK + ci] += g;
  }
}

// image head: t = tanh(y) for the 3-channel bf16 NHWC4 convolution output y -> fp32 NCHW out, and optionally the bf16
// NHWC4 copy c4 of t (the coarse image the encoder and the prior network read)
__global__ void sr_tanh_fwd_kernel(const bf16* __restrict__ y, float* __restrict__ out, bf16* __restrict__ c4, int hw,
                                   long long npix) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  const long long img = i / hw, p = i % hw;
  for (int c = 0; c < 3; ++c) {
    const float t = tanhf(__bfloat162float(y[i * 4 + c]));
    out[(img * 3 + c) * hw + p] = t;
    if (c4) c4[i * 4 + c] = __float2bfloat16_rn(t);
  }
  if (c4) c4[i * 4 + 3] = __float2bfloat16_rn(0.f);
}

// g = (d (fp32 NCHW) + s1 + s2 (bf16 NHWC slots of the copy's consumers), any of them NULL) * (1 - t^2), t = tanh(y)
// recomputed from the stored y; bf16 NHWC4, channel 3 zero
__global__ void sr_tanh_bwd_kernel(const bf16* __restrict__ y, const float* __restrict__ d, const bf16* __restrict__ s1,
                                   int s1_ld, const bf16* __restrict__ s2, int s2_ld, bf16* __restrict__ g, int hw,
                                   long long npix) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  const long long img = i / hw, p = i % hw;
  for (int c = 0; c < 3; ++c) {
    float v = d ? d[(img * 3 + c) * hw + p] : 0.f;
    if (s1) v += __bfloat162float(s1[i * s1_ld + c]);
    if (s2) v += __bfloat162float(s2[i * s2_ld + c]);
    const float t = tanhf(__bfloat162float(y[i * 4 + c]));
    g[i * 4 + c] = __float2bfloat16_rn(v * (1.f - t * t));
  }
  g[i * 4 + 3] = __float2bfloat16_rn(0.f);
}

// ---- the program ---------------------------------------------------------------------------------------------------
struct Tensor {
  bf16* p = nullptr;
  int n = 0, h = 0, w = 0, c = 0, ld = 0;
  int id = -1;
};

struct Slot {
  bf16* p;
  int ld;
};

// tape kinds (crfr_tape_entry.kind, include/crfr.h)
enum OpKind { OP_CONV = 0, OP_NORM = 1, OP_POOL = 2, OP_UPADD = 3, OP_CAT = 4, OP_HEADS = 5, OP_PAD = 20, OP_ADD = 21,
              OP_TANH = 22 };

struct Op {
  OpKind kind;
  Tensor a, b, out;
  crfr_conv_desc cd;
  int w_idx = -1, b_idx = -1, g_idx = -1, beta_idx = -1, alpha_idx = -1;
  int pad = 0;
  bool relu = false, has_res = false, x_needs_grad = true;
  bool null_bias = false;         // OP_CONV: an InstanceNorm follows, so the exact bias gradient is zero
  float* stats = nullptr;
  int du = -1, du2 = -1;          // OP_TANH: output-gradient index; OP_HEADS: landmark, parsing
  bf16* wtd = nullptr;            // OP_HEADS: transposed combined weight (training)
};

struct Net {
  int engine = CRFR_ENGINE_AUTO;
  const float* const* params = nullptr;
  float* const* grads = nullptr;
  cudaStream_t st = nullptr;
  uint8_t* ws = nullptr;
  size_t ws_bytes = 0, off = 0;
  bool exec = false, training = false;
  int err = CRFR_OK;
  int section = 0, B = 0, H = 0, W = 0;
  bool want_dx = true;
  std::vector<Op> tape;
  std::vector<std::vector<Slot>> slots;
  std::vector<void*> packed_fwd, packed_bwd;
  void* scratch = nullptr;
  size_t scratch_bytes = 0, scratch_need = 0;
  std::vector<crfr_pack_job>* collect = nullptr;
  bool packs_done = false;
  // caller's tensors (fp32 NCHW) and which output gradients are given
  const float* x_user = nullptr;
  float* out_user[4] = {nullptr, nullptr, nullptr, nullptr};
  const float* d_user[4] = {nullptr, nullptr, nullptr, nullptr};
  bool has_du[4] = {false, false, false, false};
  Tensor sec_in, feat;            // the section's bf16 input and (encoder, prior) feature output
  std::vector<crfr_tape_entry>* gtape = nullptr;   // crfr_srnet_grad_tape: the backward's gradient buffers

  void* alloc(size_t bytes) {
    size_t a = (off + 1023) & ~(size_t)1023;
    if (a + bytes > ws_bytes) {
      if (err == CRFR_OK) {
        crfr_set_error("srnet: workspace too small (%zu needed so far, %zu given)", a + bytes, ws_bytes);
        err = CRFR_EWORKSPACE;
      }
      off = a + bytes;
      return ws;
    }
    off = a + bytes;
    return ws + a;
  }
  bool ok() const { return err == CRFR_OK; }
  bool run() const { return exec && err == CRFR_OK; }
  void check(int rc) {
    if (rc != CRFR_OK && err == CRFR_OK) err = rc;
  }
  void check_cuda(cudaError_t e) { check(e == cudaSuccess ? CRFR_OK : CRFR_ECUDA); }
  void need(size_t bytes) {
    if (bytes > scratch_need) scratch_need = bytes;
  }
  static int ldof(int c) { return c < 8 ? 4 : c; }
  Tensor new_tensor(int n, int h, int w, int c) {
    Tensor t;
    t.n = n; t.h = h; t.w = w; t.c = c; t.ld = ldof(c);
    t.p = (bf16*)alloc((size_t)n * h * w * t.ld * sizeof(bf16));
    t.id = (int)slots.size();
    slots.emplace_back();
    return t;
  }
  Tensor view(const Tensor& base, int coff, int c) {
    Tensor t = base;
    t.p = base.p + coff;
    t.c = c;
    t.id = (int)slots.size();
    slots.emplace_back();
    return t;
  }
  float* grad(int idx) const { return (grads && idx >= 0) ? grads[idx] : nullptr; }
  const float* prm(int idx) const { return (params && idx >= 0) ? params[idx] : nullptr; }

  void* pack(int idx, int cout, int cin, int k, int cin_pad, bool transposed_conv, bool for_dgrad) {
    std::vector<void*>& cache = for_dgrad ? packed_bwd : packed_fwd;
    if (cache[idx]) return cache[idx];
    const int T = k * k;
    int R, S;
    long long rs, ss;
    if (!transposed_conv) {
      if (!for_dgrad) { R = cout; S = cin; rs = (long long)cin * T; ss = T; }
      else            { R = cin; S = cout; rs = T; ss = (long long)cin * T; }
    } else {
      if (!for_dgrad) { R = cout; S = cin; rs = T; ss = (long long)cout * T; }
      else            { R = cin; S = cout; rs = (long long)cout * T; ss = T; }
    }
    const int s_pad = for_dgrad ? ldof(S) : cin_pad;
    void* dst = alloc((size_t)T * R * s_pad * sizeof(bf16));
    if (collect && ok()) collect->push_back({params[idx], dst, T, R, S, s_pad, rs, ss, 0, 0});
    else if (run() && !packs_done) check(crfr_pack_weight(params[idx], dst, T, R, S, s_pad, rs, ss, 1, st));
    cache[idx] = dst;
    return dst;
  }

  // ---- forward ops ----
  Tensor reflect(const Tensor& x, int pad, bool x_needs_grad = true) {
    Tensor out = new_tensor(x.n, x.h + 2 * pad, x.w + 2 * pad, x.c);
    if (run()) check(crfr_reflect_pad_fwd(x.p, x.ld, out.p, out.ld, x.n, x.h, x.w, x.c, pad, st));
    Op op;
    op.kind = OP_PAD; op.a = x; op.out = out; op.pad = pad; op.x_needs_grad = x_needs_grad;
    tape.push_back(op);
    return out;
  }

  Tensor conv(const Tensor& x, int w_idx, int b_idx, int cout, int k, int stride, int pad, bool transposed,
              float** stats_out, bool x_needs_grad = true) {
    Op op;
    op.kind = OP_CONV;
    crfr_conv_desc& d = op.cd;
    d.n = x.n; d.h = x.h; d.w = x.w; d.cin = x.c; d.cout = cout; d.k = k; d.stride = stride; d.pad = pad;
    d.transposed = transposed ? 1 : 0;
    d.oh = transposed ? x.h * stride : (x.h + 2 * pad - k) / stride + 1;   // ConvTranspose2d(3, 2, 1, 1): exactly 2x
    d.ow = transposed ? x.w * stride : (x.w + 2 * pad - k) / stride + 1;
    Tensor y = new_tensor(x.n, d.oh, d.ow, cout);
    d.in_ld = x.ld; d.out_ld = y.ld;
    const int cin_pad = ldof(x.c);
    void* wp = pack(w_idx, cout, x.c, k, cin_pad, transposed, false);
    float* stats = nullptr;
    if (stats_out) {
      stats = (float*)alloc((size_t)x.n * cout * 2 * sizeof(float));
      *stats_out = stats;
    }
    need(crfr_conv_workspace_bytes(&d));
    if (stats) need(crfr_norm_ws_bytes(d.n, d.oh * d.ow, cout));
    // The statistics are a pass of their own over the stored output, as the single-op path computes them: with the
    // convolutions' epilogue statistics the program drifted from the single-op composition at batch 32, 128 x 128
    // (DESIGN 6f).
    if (run()) {
      check(crfr_conv_fwd(engine, &d, x.p, wp, cin_pad, prm(b_idx), y.p, nullptr, nullptr, kEps, scratch, scratch_bytes,
                          st));
      if (stats) check(crfr_norm_stats(y.p, y.n, d.oh * d.ow, cout, y.ld, kEps, stats, scratch, scratch_bytes, st));
    }
    op.a = x; op.out = y; op.w_idx = w_idx; op.b_idx = b_idx; op.x_needs_grad = x_needs_grad;
    op.null_bias = stats_out != nullptr;
    tape.push_back(op);
    return y;
  }

  float* stats_of(const Tensor& y) {
    float* stats = (float*)alloc((size_t)y.n * y.c * 2 * sizeof(float));
    need(crfr_norm_ws_bytes(y.n, y.h * y.w, y.c));
    if (run()) check(crfr_norm_stats(y.p, y.n, y.h * y.w, y.c, y.ld, kEps, stats, scratch, scratch_bytes, st));
    return stats;
  }

  Tensor norm(const Tensor& y, float* stats, int g_idx, int beta_idx, int alpha_idx, bool relu, const Tensor* res,
              const Tensor* out_view = nullptr) {
    Tensor out = out_view ? *out_view : new_tensor(y.n, y.h, y.w, y.c);
    need(crfr_norm_ws_bytes(y.n, y.h * y.w, y.c));
    if (run())
      check(crfr_norm_act_fwd(y.p, y.ld, stats, prm(g_idx), prm(beta_idx), prm(alpha_idx), relu ? 1 : 0,
                              res ? res->p : nullptr, res ? res->ld : 8, out.p, out.ld, y.n, y.h * y.w, y.c, st));
    Op op;
    op.kind = OP_NORM;
    op.a = y; op.out = out; op.stats = stats; op.g_idx = g_idx; op.beta_idx = beta_idx; op.alpha_idx = alpha_idx;
    op.relu = relu; op.has_res = res != nullptr;
    if (res) op.b = *res;
    tape.push_back(op);
    return out;
  }

  Tensor add(const Tensor& a, const Tensor& b) {
    Tensor out = new_tensor(a.n, a.h, a.w, a.c);
    if (run()) check(crfr_add_n(a.p, a.ld, b.p, b.ld, nullptr, a.c, out.p, out.ld, (long long)a.n * a.h * a.w, a.c, st));
    Op op;
    op.kind = OP_ADD; op.a = a; op.b = b; op.out = out;
    tape.push_back(op);
    return out;
  }

  Tensor maxpool(const Tensor& x) {
    Tensor out = new_tensor(x.n, x.h / 2, x.w / 2, x.c);
    if (run()) check(crfr_maxpool2_fwd(x.p, x.ld, out.p, out.ld, x.n, x.h, x.w, x.c, st));
    Op op;
    op.kind = OP_POOL; op.a = x; op.out = out;
    tape.push_back(op);
    return out;
  }

  Tensor upadd(const Tensor& up, const Tensor& low, const Tensor* out_view) {
    Tensor out = out_view ? *out_view : new_tensor(up.n, up.h, up.w, up.c);
    if (run()) check(crfr_upnearest2_add_fwd(up.p, up.ld, low.p, low.ld, out.p, out.ld, low.n, low.h, low.w, low.c, st));
    Op op;
    op.kind = OP_UPADD; op.a = up; op.b = low; op.out = out;
    tape.push_back(op);
    return out;
  }

  // ReflectionPad2d(1), Conv2d(cin, 3, 3, 1, 0), Tanh -> fp32 NCHW `out` (+ the bf16 NHWC4 copy c4)
  void image_head(const Tensor& x, int w_idx, float* out, Tensor* c4, int du) {
    Tensor y = conv(reflect(x, 1), w_idx, -1, 3, 3, 1, 0, false, nullptr);
    const long long npix = (long long)y.n * y.h * y.w;
    if (run() && out) {
      sr_tanh_fwd_kernel<<<crfr_cdiv(npix, 256), 256, 0, st>>>(y.p, out, c4 ? c4->p : nullptr, y.h * y.w, npix);
      CRFR_COUNT_LAUNCH();
      check_cuda(cudaGetLastError());
    }
    Op op;
    op.kind = OP_TANH; op.a = y; op.du = du;
    if (c4) op.out = *c4;
    tape.push_back(op);
  }

  // fc (13, bias) and fc_landmark (68, no bias): one 1x1 GEMM 64 -> kHeadsN on the tensor cores (fp32 NHWC rows in the
  // scratch), scattered into the two fp32 NCHW outputs
  void heads(const Tensor& x, int base, float* landmark, float* parsing, int du_lm, int du_ps) {
    const long long npix = (long long)x.n * x.h * x.w;
    bf16* wc = (bf16*)alloc((size_t)kHeadsN * kHeadsK * sizeof(bf16));
    float* bc = (float*)alloc(kHeadsN * sizeof(float));
    bf16* wtd = training ? (bf16*)alloc((size_t)kHeadsK * kHeadsN * sizeof(bf16)) : nullptr;
    need((size_t)npix * kHeadsN * sizeof(float));
    if (run()) {
      sr_heads_pack_kernel<<<crfr_cdiv(kHeadsN * kHeadsK, 256), 256, 0, st>>>(params[base], params[base + 1],
                                                                            params[base + 2], wc, bc, wtd);
      CRFR_COUNT_LAUNCH();
      float* yf = (float*)scratch;
      TcGemm g{x.p, x.n, x.h, x.w, kHeadsK, x.ld, wc, 1, 0, 1, kHeadsN, kHeadsN, yf, kHeadsN, 1, bc};
      check(crfr_tc_gemm(g, st));
      if (landmark && parsing) {
        sr_heads_scatter_kernel<<<dim3(crfr_cdiv(x.h * x.w, 32), x.n), 256, 0, st>>>(0, yf, parsing, landmark, nullptr,
                                                                                   nullptr, nullptr, x.h * x.w);
        CRFR_COUNT_LAUNCH();
      }
      check_cuda(cudaGetLastError());
    }
    Op op;
    op.kind = OP_HEADS; op.a = x; op.w_idx = base; op.du = du_lm; op.du2 = du_ps; op.wtd = wtd;
    tape.push_back(op);
  }

  // ---- network pieces ----
  Tensor res_block(const Tensor& x, int p) {   // _Residual_Block :12-37
    float* s1; float* s2;
    Tensor y = conv(x, p + 0, -1, x.c, 3, 1, 1, false, &s1);
    Tensor a = norm(y, s1, p + 1, p + 2, p + 3, false, nullptr);
    y = conv(a, p + 4, -1, x.c, 3, 1, 1, false, &s2);
    return norm(y, s2, p + 5, p + 6, -1, false, &x);
  }
  Tensor bottleneck(const Tensor& x, int p) {  // Bottleneck :75-114 (pre-activation, IN without affine)
    float* s;
    Tensor a = norm(x, stats_of(x), -1, -1, -1, true, nullptr);
    Tensor y = conv(a, p + 0, p + 1, x.c, 1, 1, 0, false, &s);
    a = norm(y, s, -1, -1, -1, true, nullptr);
    y = conv(a, p + 2, p + 3, x.c, 3, 1, 1, false, &s);
    a = norm(y, s, -1, -1, -1, true, nullptr);
    y = conv(a, p + 4, p + 5, x.c, 1, 1, 0, false, nullptr);
    return add(y, x);
  }
  Tensor hg_seq(Tensor x, int base, int d, int s) {
    const int seq = d == 0 ? s : 4 + 3 * (d - 1) + s;   // hg[d] holds 4 sequences at d == 0, else 3
    for (int b = 0; b < 3; ++b) x = bottleneck(x, base + (seq * 3 + b) * 6);
    return x;
  }
  Tensor hourglass(int n, const Tensor& x, int base, const Tensor* out_view) {   // Hourglass._forward :140-153
    Tensor up1 = hg_seq(x, base, n - 1, 0);
    Tensor low1 = hg_seq(maxpool(x), base, n - 1, 1);
    Tensor low2 = n > 1 ? hourglass(n - 1, low1, base, nullptr) : hg_seq(low1, base, 0, 3);
    Tensor low3 = hg_seq(low2, base, n - 1, 2);
    return upadd(up1, low3, out_view);
  }
  Tensor pad_conv(const Tensor& x, int w_idx, int cout, int k, int pad, int stride, float** stats,
                  bool x_needs_grad = true) {
    return conv(reflect(x, pad, x_needs_grad), w_idx, -1, cout, k, stride, 0, false, stats, x_needs_grad);
  }
  // ReflectionPad2d(pad), Conv2d(k, stride 1), InstanceNorm2d, ReLU
  Tensor pad_conv_in_relu(const Tensor& x, int w_idx, int cout, int k, int pad, bool x_needs_grad = true,
                          const Tensor* out_view = nullptr) {
    float* s = nullptr;
    const Tensor y = pad_conv(x, w_idx, cout, k, pad, 1, &s, x_needs_grad);
    return norm(y, s, -1, -1, -1, true, nullptr, out_view);
  }
  // _trunk: two stride-2 stages, residual blocks, two transposed-convolution stages
  Tensor trunk(Tensor x, int p, int ngf, bool x_needs_grad, const Tensor* out_view = nullptr) {
    x = pad_conv(x, p + 0, ngf * 2, 3, 1, 2, nullptr, x_needs_grad);
    x = pad_conv_in_relu(x, p + 1, ngf * 2, 3, 1);
    x = pad_conv(x, p + 2, ngf * 4, 3, 1, 2, nullptr);
    x = pad_conv_in_relu(x, p + 3, ngf * 4, 3, 1);
    for (int b = 0; b < 6; ++b) x = res_block(x, p + 4 + kResBlock * b);
    x = conv(x, p + 46, -1, ngf * 2, 3, 2, 1, true, nullptr);
    x = pad_conv_in_relu(x, p + 47, ngf * 2, 3, 1);
    x = conv(x, p + 48, -1, ngf, 3, 2, 1, true, nullptr);
    return pad_conv_in_relu(x, p + 49, ngf, 3, 1, true, out_view);
  }

  void coarse_net(const Tensor& x4, int p, float* out, Tensor* c4, int du, bool x_grad) {   // :251-301
    Tensor a = pad_conv_in_relu(x4, p + 0, 64, 7, 3, x_grad);
    image_head(trunk(a, p + 1, 64, true), p + 1 + kTrunk, out, c4, du);
  }
  Tensor encoder_net(const Tensor& x4, int p, const Tensor* out_view, bool x_grad) {   // :304-346
    Tensor y = pad_conv(x4, p + 0, 64, 3, 1, 1, nullptr, x_grad);   // no norm / activation behind the first conv
    return trunk(y, p + 1, 64, true, out_view);
  }
  Tensor prior_net(const Tensor& x4, int p, const Tensor* out_view, float* landmark, float* parsing, int du_lm,
                   int du_ps, bool x_grad) {   // :349-376
    Tensor a = pad_conv_in_relu(x4, p + 3, 64, 7, 3, x_grad);
    a = res_block(a, p + 4);
    a = res_block(a, p + 4 + kResBlock);
    for (int h = 0; h < 4; ++h) a = hourglass(4, a, p + 4 + 2 * kResBlock + kHgParams * h, h == 3 ? out_view : nullptr);
    heads(a, p, landmark, parsing, du_lm, du_ps);
    return a;
  }
  void decoder_net(const Tensor& x, int p, float* out, int du, bool x_grad) {   // :379-416
    image_head(trunk(x, p, 128, x_grad), p + kTrunk, out, nullptr, du);
  }

  Tensor image_in() {
    Tensor t = new_tensor(B, H, W, 3);
    if (run()) check(crfr_nchw_f32_to_nhwc_bf16(x_user, t.p, B, 3, H, W, 4, 4, st));
    return t;
  }

  void prologue() {
    const int n = section_params(section);
    packed_fwd.assign(n, nullptr);
    packed_bwd.assign(n, nullptr);
    need(crfr_tc_wgrad_part_bytes());
    need(1 << 20);
    scratch = alloc(scratch_bytes);
  }

  void forward() {
    prologue();
    switch (section) {
      case CRFR_SRNET_NETWORK: {
        sec_in = image_in();
        Tensor c4 = new_tensor(B, H, W, 3);
        coarse_net(sec_in, kNetCoarse, out_user[0], &c4, 0, want_dx);
        Tensor cat = new_tensor(B, H, W, 128);
        Tensor pe = view(cat, 0, 64), enc = view(cat, 64, 64);   // torch.cat((prior, encoder), 1)
        encoder_net(c4, kNetEncoder, &enc, true);
        prior_net(c4, kNetPrior, &pe, out_user[2], out_user[3], 2, 3, true);
        Op cop;
        cop.kind = OP_CAT; cop.a = pe; cop.b = enc; cop.out = cat;
        tape.push_back(cop);
        decoder_net(cat, kNetDecoder, out_user[1], 1, true);
        break;
      }
      case CRFR_SRNET_COARSE:
        sec_in = image_in();
        coarse_net(sec_in, 0, out_user[0], nullptr, 0, want_dx);
        break;
      case CRFR_SRNET_ENCODER:
        sec_in = image_in();
        feat = encoder_net(sec_in, 0, nullptr, want_dx);
        break;
      case CRFR_SRNET_PRIOR:
        sec_in = image_in();
        feat = prior_net(sec_in, 0, nullptr, out_user[1], out_user[2], 1, 2, want_dx);
        break;
      default:   // CRFR_SRNET_DECODER
        sec_in = new_tensor(B, H, W, 128);
        if (run()) check(crfr_nchw_f32_to_nhwc_bf16(x_user, sec_in.p, B, 128, H, W, 128, 128, st));
        decoder_net(sec_in, 0, out_user[0], 0, want_dx);
        break;
    }
    if (feat.p && run() && out_user[0])
      check(crfr_nhwc_bf16_to_nchw_f32(feat.p, out_user[0], B, feat.c, feat.h, feat.w, feat.ld, st));
  }

  // ---- backward ----
  void add_slot(const Tensor& t, bf16* p, int ld) { slots[t.id].push_back({p, ld}); }
  bool has_grad(const Tensor& t) const { return t.id >= 0 && !slots[t.id].empty(); }
  void squash(const Tensor& t, size_t max_slots) {
    std::vector<Slot>& s = slots[t.id];
    while (s.size() > max_slots) {
      const bool three = s.size() >= 3;
      const int cc = ldof(t.c);
      bf16* out = (bf16*)alloc((size_t)t.n * t.h * t.w * cc * sizeof(bf16));
      const size_t k = s.size();
      Slot a = s[k - 1], b = s[k - 2], c = three ? s[k - 3] : Slot{nullptr, cc};
      if (run()) check(crfr_add_n(a.p, a.ld, b.p, b.ld, c.p, c.ld, out, cc, (long long)t.n * t.h * t.w, cc, st));
      s.resize(k - (three ? 3 : 2));
      s.push_back({out, cc});
    }
  }
  bf16* alloc_grad(const Tensor& x) {   // a dense gradient of x (channels up to ldof(c) zeroed where c < ld)
    const int xc = ldof(x.c);
    const size_t bytes = (size_t)x.n * x.h * x.w * xc * sizeof(bf16);
    bf16* g = (bf16*)alloc(bytes);
    if (xc != x.c && run()) check_cuda(cudaMemsetAsync(g, 0, bytes, st));
    return g;
  }

  // crfr_srnet_grad_tape entries: kind 30 = a gradient slot op i consumes for its output t, kind 31 = a gradient op i
  // produces for its input t (which: 0 first input, 1 second)
  void rec(int kind, int i, const bf16* g, int ld, const Tensor& t, int which) {
    if (!gtape) return;
    crfr_tape_entry e{};
    e.kind = kind;
    e.n = t.n; e.h = t.h; e.w = t.w; e.c = t.c; e.ld = ld;
    e.out_off = g ? (long long)((const uint8_t*)g - (const uint8_t*)nullptr) : -1;
    e.in_off = t.p ? (long long)((const uint8_t*)t.p - (const uint8_t*)nullptr) : -1;
    e.stats_off = -1;
    e.w_idx = i;
    e.has_res = which;
    gtape->push_back(e);
  }
  void rec_out(int i, const Tensor& t) {
    for (const Slot& sl : slots[t.id]) rec(30, i, sl.p, sl.ld, t, 0);
  }

  void backward() {
    for (int i = (int)tape.size() - 1; i >= 0 && ok(); --i) {
      Op& op = tape[i];
      switch (op.kind) {
        case OP_NORM: {
          if (!has_grad(op.out)) break;
          squash(op.out, 2);
          rec_out(i, op.out);
          std::vector<Slot>& s = slots[op.out.id];
          const Tensor& y = op.a;
          const size_t bytes = (size_t)y.n * y.h * y.w * y.c * sizeof(bf16);
          bf16* dz = (op.has_res || s.size() > 1) ? (bf16*)alloc(bytes) : nullptr;
          bf16* dy = (bf16*)alloc(bytes);
          need(crfr_norm_ws_bytes(y.n, y.h * y.w, y.c));
          if (run())
            check(crfr_norm_act_bwd(s[0].p, s[0].ld, s.size() > 1 ? s[1].p : nullptr, s.size() > 1 ? s[1].ld : 8, y.p,
                                    y.ld, op.stats, prm(op.g_idx), prm(op.beta_idx), prm(op.alpha_idx), op.relu ? 1 : 0,
                                    op.has_res ? op.b.p : nullptr, op.has_res ? op.b.ld : 8, dz, y.c, dy, y.c,
                                    grad(op.g_idx), grad(op.beta_idx), grad(op.alpha_idx), y.n, y.h * y.w, y.c, scratch,
                                    scratch_bytes, st));
          add_slot(y, dy, y.c);
          rec(31, i, dy, y.c, y, 0);
          if (op.has_res) {
            add_slot(op.b, dz, y.c);
            rec(31, i, dz, y.c, op.b, 1);
          }
          break;
        }
        case OP_CONV: {
          if (!has_grad(op.out)) break;
          squash(op.out, 1);
          rec_out(i, op.out);
          const Slot dy = slots[op.out.id][0];
          crfr_conv_desc d = op.cd;
          d.out_ld = dy.ld;
          need(crfr_conv_workspace_bytes(&d));
          // the bias of a convolution an InstanceNorm follows cancels in the normalisation: its gradient stays exactly
          // zero (a column sum would return rounding noise only), as in fsrnet.cu
          if (run())
            check(crfr_conv_wgrad(engine, &d, op.a.p, dy.p, grad(op.w_idx), op.null_bias ? nullptr : grad(op.b_idx),
                                  scratch, scratch_bytes, st));
          if (!op.x_needs_grad) break;
          const Tensor& x = op.a;
          bf16* dx = alloc_grad(x);
          crfr_conv_desc dd = d;
          dd.in_ld = ldof(x.c);
          void* wt = pack(op.w_idx, d.cout, d.cin, d.k, 0, d.transposed != 0, true);
          need(crfr_conv_workspace_bytes(&dd));
          if (run()) check(crfr_conv_dgrad(engine, &dd, dy.p, wt, ldof(d.cout), dx, scratch, scratch_bytes, st));
          add_slot(x, dx, ldof(x.c));
          rec(31, i, dx, ldof(x.c), x, 0);
          break;
        }
        case OP_PAD: {
          if (!has_grad(op.out) || !op.x_needs_grad) break;
          squash(op.out, 1);
          const Slot g = slots[op.out.id][0];
          const Tensor& x = op.a;
          bf16* dx = alloc_grad(x);
          rec_out(i, op.out);
          if (run()) check(crfr_reflect_pad_bwd(g.p, g.ld, dx, ldof(x.c), x.n, x.h, x.w, x.c, op.pad, st));
          add_slot(x, dx, ldof(x.c));
          rec(31, i, dx, ldof(x.c), x, 0);
          break;
        }
        case OP_ADD: {
          if (!has_grad(op.out)) break;
          squash(op.out, 1);
          const Slot g = slots[op.out.id][0];
          rec_out(i, op.out);
          add_slot(op.a, g.p, g.ld);
          add_slot(op.b, g.p, g.ld);
          rec(31, i, g.p, g.ld, op.a, 0);
          rec(31, i, g.p, g.ld, op.b, 1);
          break;
        }
        case OP_POOL: {
          if (!has_grad(op.out)) break;
          squash(op.out, 1);
          const Slot g = slots[op.out.id][0];
          const Tensor& x = op.a;
          bf16* dx = (bf16*)alloc((size_t)x.n * x.h * x.w * x.c * sizeof(bf16));
          rec_out(i, op.out);
          if (run()) check(crfr_maxpool2_bwd(x.p, x.ld, g.p, g.ld, dx, x.c, x.n, x.h, x.w, x.c, st));
          add_slot(x, dx, x.c);
          rec(31, i, dx, x.c, x, 0);
          break;
        }
        case OP_UPADD: {
          if (!has_grad(op.out)) break;
          squash(op.out, 1);
          const Slot g = slots[op.out.id][0];
          const Tensor& low = op.b;
          bf16* dlow = (bf16*)alloc((size_t)low.n * low.h * low.w * low.c * sizeof(bf16));
          if (run()) check(crfr_upnearest2_bwd(g.p, g.ld, dlow, low.c, low.n, low.h, low.w, low.c, st));
          rec_out(i, op.out);
          add_slot(op.a, g.p, g.ld);
          add_slot(low, dlow, low.c);
          rec(31, i, g.p, g.ld, op.a, 0);
          rec(31, i, dlow, low.c, low, 1);
          break;
        }
        case OP_CAT: {
          if (!has_grad(op.out)) break;
          squash(op.out, 1);
          const Slot g = slots[op.out.id][0];
          rec_out(i, op.out);
          add_slot(op.a, g.p, g.ld);
          add_slot(op.b, g.p + op.a.c, g.ld);
          rec(31, i, g.p, g.ld, op.a, 0);
          rec(31, i, g.p + op.a.c, g.ld, op.b, 1);
          break;
        }
        case OP_HEADS: {
          if (!has_du[op.du] && !has_du[op.du2]) break;
          const Tensor& x = op.a;
          const long long npix = (long long)x.n * x.h * x.w;
          bf16* dh = (bf16*)alloc((size_t)npix * kHeadsN * sizeof(bf16));
          float* G = (float*)alloc((size_t)kHeadsK * kHeadsN * sizeof(float));
          bf16* dx = (bf16*)alloc((size_t)npix * kHeadsK * sizeof(bf16));
          if (run()) {
            sr_heads_scatter_kernel<<<dim3(crfr_cdiv(x.h * x.w, 32), x.n), 256, 0, st>>>(
                1, nullptr, nullptr, nullptr, d_user[op.du2], d_user[op.du], dh, x.h * x.w);
            CRFR_COUNT_LAUNCH();
            check_cuda(cudaGetLastError());
            TcWgrad wg{x.p, x.n, x.h, x.w, kHeadsK, x.ld, dh, kHeadsN, kHeadsN, 0, G};
            wg.part = (float*)scratch;
            wg.part_bytes = scratch_bytes;
            check(crfr_tc_wgrad_raw(wg, st));
            sr_heads_unpack_kernel<<<crfr_cdiv(kHeads * kHeadsK, 256), 256, 0, st>>>(G, grad(op.w_idx),
                                                                                    grad(op.w_idx + 2));
            CRFR_COUNT_LAUNCH();
            check_cuda(cudaGetLastError());
            if (grad(op.w_idx + 1))
              check(crfr_colsum(dh, kHeadsN, kParsing, npix, grad(op.w_idx + 1), scratch, scratch_bytes, st));
            TcGemm g{dh, x.n, x.h, x.w, kHeadsN, kHeadsN, op.wtd, 1, 0, 1, kHeadsK, kHeadsK, dx, kHeadsK, 0, nullptr};
            check(crfr_tc_gemm(g, st));
          }
          Tensor hd = x;   // the gathered output gradient [pixel][kHeadsN] (no forward tensor of its own)
          hd.p = nullptr;
          hd.c = kHeadsN;
          rec(30, i, dh, kHeadsN, hd, 0);
          add_slot(x, dx, kHeadsK);
          rec(31, i, dx, kHeadsK, x, 0);
          break;
        }
        case OP_TANH: {
          const bool copied = op.out.p != nullptr;
          if (copied) squash(op.out, 2);
          const std::vector<Slot>* s = copied ? &slots[op.out.id] : nullptr;
          const size_t ns = s ? s->size() : 0;
          if (!has_du[op.du] && ns == 0) break;
          if (copied) rec_out(i, op.out);
          const Tensor& y = op.a;
          const long long npix = (long long)y.n * y.h * y.w;
          bf16* g = (bf16*)alloc((size_t)npix * 4 * sizeof(bf16));
          if (run()) {
            sr_tanh_bwd_kernel<<<crfr_cdiv(npix, 256), 256, 0, st>>>(
                y.p, d_user[op.du], ns > 0 ? (*s)[0].p : nullptr, ns > 0 ? (*s)[0].ld : 4, ns > 1 ? (*s)[1].p : nullptr,
                ns > 1 ? (*s)[1].ld : 4, g, y.h * y.w, npix);
            CRFR_COUNT_LAUNCH();
            check_cuda(cudaGetLastError());
          }
          add_slot(y, g, 4);
          rec(31, i, g, 4, y, 0);
          break;
        }
      }
    }
  }
};

// shapes the program takes (include/crfr.h)
bool shape_ok(int section, int batch, int h, int w) {
  if (section < CRFR_SRNET_COARSE || section > CRFR_SRNET_NETWORK || batch <= 0) return false;
  if (section == CRFR_SRNET_PRIOR || section == CRFR_SRNET_NETWORK) {
    if (h < 16 || w < 16 || h % 16 || w % 16) return false;
  } else if (h < 5 || w < 5) {
    return false;
  }
  const long long oh = 4LL * ((h + 3) / 4), ow = 4LL * ((w + 3) / 4);
  return (long long)batch * (oh + 6) * (ow + 6) * 128 < (1LL << 31);
}

void init(Net& net, int section, int batch, int h, int w, int training) {
  net.section = section; net.B = batch; net.H = h; net.W = w; net.training = training != 0;
}

// the scratch every op of the call may use (the largest need of any op, forward and, in training, backward)
size_t scratch_size_uncached(int section, int batch, int h, int w, int training) {
  Net net;
  init(net, section, batch, h, w, training);
  net.ws_bytes = ~(size_t)0 >> 2;
  net.forward();
  if (training) {
    for (bool& b : net.has_du) b = true;
    net.backward();
  }
  return (net.scratch_need + 4095) & ~(size_t)4095;
}
// (a dry run of the whole tape: remembered per shape, since every call's layout needs it)
size_t scratch_size(int section, int batch, int h, int w, int training) {
  static std::mutex mu;
  static std::map<std::array<int, 5>, size_t> cache;
  const std::array<int, 5> key = {section, batch, h, w, training != 0};
  {
    std::lock_guard<std::mutex> lock(mu);
    auto it = cache.find(key);
    if (it != cache.end()) return it->second;
  }
  const size_t bytes = scratch_size_uncached(section, batch, h, w, training);
  std::lock_guard<std::mutex> lock(mu);
  cache[key] = bytes;
  return bytes;
}

// the layout of a call: forward (exec false) over ws; with `grads`, the output-gradient flags of the backward
void layout(Net& net, int section, int batch, int h, int w, int training, void* ws, size_t ws_bytes) {
  init(net, section, batch, h, w, training);
  net.ws = (uint8_t*)ws;
  net.ws_bytes = ws_bytes;
  net.scratch_bytes = scratch_size(section, batch, h, w, training);
}

int noutputs(int section) {
  return section == CRFR_SRNET_NETWORK ? 4 : (section == CRFR_SRNET_PRIOR ? 3 : 1);
}

int check_call(int engine, const float* const* params, const crfr_srnet_io* io, const void* ws, const char* who,
               bool need_tensors) {
  CRFR_CHECK_ARG(io && params && ws, "%s: null pointer", who);
  CRFR_CHECK_ARG(engine == CRFR_ENGINE_AUTO || engine == CRFR_ENGINE_DIRECT || engine == CRFR_ENGINE_TCGEN05,
                 "%s: unknown engine %d", who, engine);
  CRFR_CHECK_ARG(shape_ok(io->section, io->batch, io->h, io->w),
                 "%s: section %d, batch %d, %d x %d not supported (include/crfr.h: crfr_srnet_io)", who, io->section,
                 io->batch, io->h, io->w);
  const int np = section_params(io->section);
  for (int i = 0; i < np; ++i) CRFR_CHECK_ARG(params[i], "%s: parameter %d is NULL", who, i);
  if (need_tensors) {
    CRFR_CHECK_ARG(io->x, "%s: null input", who);
    for (int i = 0; i < noutputs(io->section); ++i) CRFR_CHECK_ARG(io->out[i], "%s: null output %d", who, i);
  }
  return CRFR_OK;
}

void set_grads(Net& net, const float* const* d_out) {
  for (int i = 0; i < 4; ++i) {
    net.d_user[i] = (d_out && i < noutputs(net.section)) ? d_out[i] : nullptr;
    net.has_du[i] = net.d_user[i] != nullptr;
  }
}

// backward after the forward dry run: the feature output's gradient, the replay, the input gradient (dx, when
// input_grad; a dry run writes nothing)
void run_backward(Net& net, bool input_grad, float* dx) {
  if (net.feat.p && net.has_du[0]) {
    const Tensor& f = net.feat;
    bf16* g = (bf16*)net.alloc((size_t)f.n * f.h * f.w * f.c * sizeof(bf16));
    if (net.run()) net.check(crfr_nchw_f32_to_nhwc_bf16(net.d_user[0], g, f.n, f.c, f.h, f.w, f.c, f.c, net.st));
    net.add_slot(f, g, f.c);
  }
  net.backward();
  if (!input_grad || !net.ok()) return;
  const Tensor& x = net.sec_in;
  if (!net.has_grad(x)) {   // no output gradient given: the input gradient is zero
    if (net.run())
      net.check_cuda(cudaMemsetAsync(dx, 0, (size_t)x.n * x.c * x.h * x.w * sizeof(float), net.st));
    return;
  }
  net.squash(x, 1);
  const Slot g = net.slots[x.id][0];
  if (net.run()) net.check(crfr_nhwc_bf16_to_nchw_f32(g.p, dx, x.n, x.c, x.h, x.w, g.ld, net.st));
}

}  // namespace

extern "C" size_t crfr_srnet_workspace_bytes(int section, int batch, int h, int w, int training) {
  if (!shape_ok(section, batch, h, w)) return 0;
  Net net;
  layout(net, section, batch, h, w, training, nullptr, ~(size_t)0 >> 2);
  net.forward();
  if (training) {
    for (bool& b : net.has_du) b = true;
    run_backward(net, true, nullptr);
  }
  return net.off + 65536;
}

extern "C" int crfr_srnet_tape(int section, int batch, int h, int w, int training, crfr_tape_entry* entries,
                               int max_entries) {
  if (!shape_ok(section, batch, h, w)) return -1;
  Net net;
  layout(net, section, batch, h, w, training, nullptr, ~(size_t)0 >> 2);
  net.forward();
  const int count = (int)net.tape.size();
  auto off = [](const void* p) { return p ? (long long)((const uint8_t*)p - (const uint8_t*)nullptr) : -1LL; };
  for (int i = 0; i < count && i < max_entries && entries; ++i) {
    const Op& op = net.tape[i];
    crfr_tape_entry& e = entries[i];
    const Tensor& t = op.out.p ? op.out : op.a;
    e.kind = (int)op.kind;
    e.n = t.n; e.h = t.h; e.w = t.w; e.c = t.c; e.ld = t.ld;
    if (op.kind == OP_HEADS) e.c = kHeads;
    e.out_off = off(op.out.p);
    e.in_off = off(op.a.p);
    e.stats_off = op.kind == OP_NORM ? off(op.stats) : off(op.b.p);
    e.w_idx = op.kind == OP_PAD ? op.pad : op.w_idx;
    e.has_res = op.has_res ? 1 : 0;
  }
  return count;
}

extern "C" int crfr_srnet_grad_tape(int section, int batch, int h, int w, int grad_mask, int input_grad,
                                    crfr_tape_entry* entries, int max_entries) {
  if (!shape_ok(section, batch, h, w) || grad_mask <= 0 || grad_mask >= (1 << noutputs(section))) return -1;
  Net net;
  layout(net, section, batch, h, w, 1, nullptr, ~(size_t)0 >> 2);
  net.want_dx = input_grad != 0;
  net.forward();
  for (int i = 0; i < 4; ++i) net.has_du[i] = (grad_mask >> i) & 1;
  std::vector<crfr_tape_entry> g;
  net.gtape = &g;
  run_backward(net, input_grad != 0, nullptr);
  if (!net.ok()) return -1;
  const int count = (int)g.size();
  for (int i = 0; i < count && i < max_entries && entries; ++i) entries[i] = g[i];
  return count;
}

extern "C" int crfr_srnet_forward(int engine, const float* const* host_params, const crfr_srnet_io* io, int training,
                                  void* ws, size_t ws_bytes, void* stream) {
  CRFR_TRY(check_call(engine, host_params, io, ws, "srnet_forward", true));
  cudaStream_t st = (cudaStream_t)stream;
  {   // dry run over the given arena: every weight pack in one batch, nothing launched if the arena is too small
    std::vector<crfr_pack_job> jobs;
    Net dry;
    layout(dry, io->section, io->batch, io->h, io->w, training, ws, ws_bytes);
    dry.params = host_params;
    dry.collect = &jobs;
    dry.forward();
    if (!dry.ok()) return dry.err;
    CRFR_TRY(crfr_pack_weight_batch(jobs.data(), (int)jobs.size(), st));
  }
  Net net;
  layout(net, io->section, io->batch, io->h, io->w, training, ws, ws_bytes);
  net.engine = engine; net.params = host_params; net.st = st; net.exec = true; net.packs_done = true;
  net.x_user = io->x;
  for (int i = 0; i < 4; ++i) net.out_user[i] = i < noutputs(io->section) ? io->out[i] : nullptr;
  net.forward();
  return net.err;
}

extern "C" int crfr_srnet_backward(int engine, const float* const* host_params, float* const* host_grads,
                                   const crfr_srnet_io* io, const float* const* d_out, float* dx, void* ws,
                                   size_t ws_bytes, void* stream) {
  CRFR_TRY(check_call(engine, host_params, io, ws, "srnet_backward", false));
  CRFR_CHECK_ARG(host_grads, "srnet_backward: null gradient table");
  cudaStream_t st = (cudaStream_t)stream;
  {   // dry run of the whole call: the backward's weight packs in one batch; nothing launched if the arena is too small
    std::vector<crfr_pack_job> jobs;
    Net dry;
    layout(dry, io->section, io->batch, io->h, io->w, 1, ws, ws_bytes);
    dry.params = host_params;
    dry.want_dx = dx != nullptr;
    dry.forward();
    set_grads(dry, d_out);
    dry.collect = &jobs;
    run_backward(dry, dx != nullptr, dx);
    if (!dry.ok()) return dry.err;
    CRFR_TRY(crfr_pack_weight_batch(jobs.data(), (int)jobs.size(), st));
  }
  Net net;
  layout(net, io->section, io->batch, io->h, io->w, 1, ws, ws_bytes);
  net.engine = engine; net.params = host_params; net.grads = host_grads; net.st = st; net.packs_done = true;
  net.want_dx = dx != nullptr;
  net.forward();   // dry: rebuilds the tape and the saved offsets
  if (!net.ok()) return net.err;
  net.exec = true;
  set_grads(net, d_out);
  run_backward(net, dx != nullptr, dx);
  return net.err;
}
