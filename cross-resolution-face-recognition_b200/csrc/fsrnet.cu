// Native FSRNet network program: the whole OverallNetwork forward / backward / train step is sequenced here in C++
// (no per-layer Python), on one stream, over a caller-provided workspace arena.
//
// The forward pass records a tape of fused ops (conv [+ InstanceNorm statistics], normalise+PReLU(+residual),
// max-pool, nearest-up+add, concat-by-view); the backward pass replays the tape in reverse.  A tensor that feeds
// several consumers gets one gradient "slot" per consumer; the producer's backward sums them on the fly
// (norm_act_bwd reads two) or with one add_n launch.  Because the arena is a deterministic bump allocator, the
// backward entry point rebuilds the tape with a dry run of the forward (no launches) and finds every saved
// activation at the same offset.
//
// ref: model/FSRnet.py:75-98 (_Residual_Block), :105-135 (BasicBlock), :176-215 (Hourglass), :308-340 (coarse),
//      :342-379 (encoder), :381-426 (prior), :428-459 (decoder), :488-508 + :538-541 (OverallNetwork wiring),
//      FSR_main.py:233-234 (loss composition).
#include <stdlib.h>

#include <vector>

#include "common.cuh"
#include "crfr.h"
#include "internal.h"

// dst[ci][coff + r] = w[r][ci]  (transposed 1x1 weights into a column range of a wider matrix)
int crfr_pack_weight_cols(const float* w, void* dst, int cin, int rows, int ld, int coff, cudaStream_t st);

namespace {

constexpr float kEps = 1e-5f;
constexpr int kHeadsPad = 128;   // fc (11) + fc_landmark (97) output channels padded to one UMMA-friendly width

// ---- parameter table (state_dict order, 202 entries) ---------------------------------------------
enum { RB_CONV1 = 0, RB_IN1_W, RB_IN1_B, RB_RELU, RB_CONV2, RB_IN2_W, RB_IN2_B, RB_RELU_OUT };
enum {
  C_CONV_IN_W = 0, C_CONV_IN_B = 1, C_RELU = 2, C_RES = 3, C_CONV_MID_W = 27, C_CONV_MID_B = 28, C_BN_MID_W = 29,
  C_BN_MID_B = 30,
  P_CONV_W = 33, P_CONV_B = 34, P_BN_W = 35, P_BN_B = 36, P_RELU = 37, P_RES = 38, P_HG = 86, P_FC_W = 128,
  P_FC_B = 129, P_FCL_W = 130, P_FCL_B = 131,
  E_CONV_IN_W = 132, E_CONV_IN_B = 133, E_RELU = 134, E_RES = 135, E_BN_MID_W = 161, E_BN_MID_B = 162,
  E_CONV_END_W = 165, E_CONV_END_B = 166,
  D_CONV_IN_W = 167, D_CONV_IN_B = 168, D_RELU = 169, D_BN_MID_W = 170, D_BN_MID_B = 171, D_DECONV_W = 172,
  D_DECONV_B = 173, D_RES = 174, D_CONV_OUT_W = 198, D_CONV_OUT_B = 199
};
inline int hg_param(int d, int s, int b, int which) { return P_HG + (d == 0 ? 0 : 24) + ((s * 2 + b) * 3) + which; }

// combined head weight [co = 128][ci = 128] (rows 0..10 fc, 11..107 fc_landmark, rest zero) and bias [128]
__global__ void heads_pack_kernel(const float* __restrict__ w_fc, const float* __restrict__ b_fc,
                                  const float* __restrict__ w_lm, const float* __restrict__ b_lm, bf16* __restrict__ wc,
                                  float* __restrict__ bc) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= kHeadsPad * 128) return;
  const int co = i >> 7, ci = i & 127;
  float v = 0.f;
  if (co < 11) v = w_fc[co * 128 + ci];
  else if (co < 108) v = w_lm[(co - 11) * 128 + ci];
  wc[i] = __float2bfloat16_rn(v);
  if (ci == 0) bc[co] = co < 11 ? b_fc[co] : (co < 108 ? b_lm[co - 11] : 0.f);
}

// fp32 NHWC [npix][128] -> parsing [n][11][hw] and landmark [n][97][hw] (fp32 NCHW); one thread per output element,
// consecutive threads walk consecutive pixels of one channel (coalesced writes, 512-byte-strided L2-resident reads)
__global__ void heads_split_kernel(const float* __restrict__ y, float* __restrict__ parsing, float* __restrict__ landmark,
                                   int n, int hw) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)n * 108 * hw;
  if (i >= total) return;
  const int p = (int)(i % hw);
  const long long q = i / hw;
  const int c = (int)(q % 108);
  const long long img = q / 108;
  const float v = y[(img * hw + p) * kHeadsPad + c];
  if (c < 11) parsing[(img * 11 + c) * hw + p] = v;
  else landmark[(img * 97 + (c - 11)) * hw + p] = v;
}

// dW_fc [11][128] += G[ci][co], dW_fcl [97][128] += G[ci][11 + co]
__global__ void heads_unpack_kernel(const float* __restrict__ G, float* __restrict__ dw_fc, float* __restrict__ dw_lm) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 108 * 128) return;
  const int co = i >> 7, ci = i & 127;
  const float g = G[ci * kHeadsPad + co];
  if (co < 11) {
    if (dw_fc) dw_fc[co * 128 + ci] += g;
  } else if (dw_lm) {
    dw_lm[(co - 11) * 128 + ci] += g;
  }
}

struct Tensor {
  bf16* p = nullptr;
  int n = 0, h = 0, w = 0, c = 0, ld = 0;
  int id = -1;
};

struct Slot {
  bf16* p;
  int ld;
};

enum OpKind { OP_CONV, OP_NORM, OP_POOL, OP_UPADD, OP_CAT, OP_HEADS, OP_IMGCONV };

// Helper stream for the weight-gradient GEMMs of the backward pass.  A conv's wgrad (tensor-bound) has no consumer
// until the optimiser step, while the InstanceNorm backward of the layer below (HBM-bound) is on the critical path:
// the wgrad is forked onto this stream behind the layer's dgrad so that the two run concurrently, and joined back
// before a gradient bucket is published / before the call returns its work to the caller's stream.  From the
// caller's point of view everything is still ordered on the stream it passed.
struct SideStream {
  cudaStream_t st = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
};
SideStream* side_stream() {
  static thread_local SideStream per_dev[16];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) return nullptr;
  SideStream& s = per_dev[dev];
  if (!s.st) {
    if (cudaStreamCreateWithFlags(&s.st, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&s.join, cudaEventDisableTiming) != cudaSuccess) {
      cudaGetLastError();
      s.st = nullptr;
      return nullptr;
    }
  }
  return &s;
}
int side_enabled() { return crfr_opt(CRFR_OPT_WGRAD_STREAM); }

struct Op {
  OpKind kind;
  Tensor a, b, out;        // inputs / output
  crfr_conv_desc cd;       // OP_CONV / OP_IMGCONV
  int w_idx = -1, b_idx = -1, g_idx = -1, beta_idx = -1, alpha_idx = -1;
  int cin_pad = 0;
  float* stats = nullptr;  // OP_NORM
  bool has_res = false;
  bool x_needs_grad = true;
  bool bwd_done = false;   // OP_NORM: its backward already ran, fused into the backward of the convolution it feeds
};

struct Net {
  int engine;
  const float* const* params;
  float* const* grads;
  const crfr_fsrnet_io* io;
  cudaStream_t st;
  uint8_t* ws;
  size_t ws_bytes, off = 0;
  bool exec;        // false: dry run (allocate + record only)
  bool training;
  int err = CRFR_OK;
  std::vector<Op> tape;
  std::vector<std::vector<Slot>> slots;
  void* packed_fwd[CRFR_FSRNET_NPARAMS];
  void* packed_bwd[CRFR_FSRNET_NPARAMS];
  void* scratch = nullptr;
  size_t scratch_bytes = 0;
  void* scratch2 = nullptr;          // private scratch of the wgrad helper stream
  size_t scratch2_bytes = 0;
  SideStream* side = nullptr;
  bool side_dirty = false;
  // weight packing: a dry run of the program (exec = false) collects every pack job here, the entry point issues them
  // as one batch, and the real run (packs_done) only re-derives the same arena offsets
  std::vector<crfr_pack_job>* collect = nullptr;
  bool packs_done = false;
  // fixed buffers
  Tensor x4, coarse4, cat;
  int tape_enc_start = 0, tape_dec_start = 0;   // first tape index of the encoder / decoder sections
  // output gradients (bf16): NHWC4 images and the combined 128-wide heads buffer
  bf16* d_coarse4 = nullptr;
  bf16* d_out4 = nullptr;
  bf16* d_heads = nullptr;
  // sub-network mode (crfr_fsrnet_section_*): one of the four sub-networks on its own, fp32 NCHW in and out
  int section = -1;
  const crfr_fsrnet_section_io* sio = nullptr;
  bool want_dx = false;       // backward: the gradient w.r.t. the section input is requested
  int fuse_bwd = -1;          // -1: option fuse_norm_bwd; 0 / 1: forced (the workspace sizing runs take the larger layout)
  Tensor sec_in, sec_feat;    // the section's bf16 input (NHWC) and its bf16 feature output

  void* alloc(size_t bytes) {
    size_t a = (off + 1023) & ~(size_t)1023;
    if (a + bytes > ws_bytes) {
      if (err == CRFR_OK) {
        crfr_set_error("fsrnet: workspace too small (%zu needed so far, %zu given)", a + bytes, ws_bytes);
        err = CRFR_EWORKSPACE;
      }
      off = a + bytes;  // keep counting so the dry run reports the total
      return ws;        // harmless pointer, nothing executes after an error
    }
    off = a + bytes;
    return ws + a;
  }
  bool ok() const { return err == CRFR_OK; }
  bool run() const { return exec && err == CRFR_OK; }
  void check(int rc) {
    if (rc != CRFR_OK && err == CRFR_OK) err = rc;
  }
  Tensor new_tensor(int n, int h, int w, int c) {
    Tensor t;
    t.n = n; t.h = h; t.w = w; t.c = c; t.ld = c;
    t.p = (bf16*)alloc((size_t)n * h * w * c * sizeof(bf16));
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

  // ---- weight packing (once per call and per direction) ----
  void* pack(int idx, int cout, int cin, int k, int cin_pad, bool transposed_conv, bool for_dgrad) {
    void** cache = for_dgrad ? packed_bwd : packed_fwd;
    if (cache[idx]) return cache[idx];
    const int T = k * k;
    int R, S, s_pad;
    long long rs, ss;
    if (!transposed_conv) {           // Conv2d weight [cout][cin][k][k]
      if (!for_dgrad) { R = cout; S = cin; rs = (long long)cin * T; ss = T; }
      else            { R = cin; S = cout; rs = T; ss = (long long)cin * T; }
    } else {                          // ConvTranspose2d weight [cin][cout][k][k]
      if (!for_dgrad) { R = cout; S = cin; rs = T; ss = (long long)cout * T; }
      else            { R = cin; S = cout; rs = (long long)cout * T; ss = T; }
    }
    s_pad = for_dgrad ? ((S + 7) / 8) * 8 : cin_pad;
    if (for_dgrad && S < 8) s_pad = 4;
    void* dst = alloc((size_t)T * R * s_pad * sizeof(bf16));
    if (collect && ok()) collect->push_back({params[idx], dst, T, R, S, s_pad, rs, ss, 0, 0});
    else if (run() && !packs_done) check(crfr_pack_weight(params[idx], dst, T, R, S, s_pad, rs, ss, 1, st));
    cache[idx] = dst;
    return dst;
  }

  // ---- forward ops ----
  Tensor conv(const Tensor& x, int w_idx, int b_idx, int cout, int k, int stride, int pad, bool transposed,
              float** stats_out, const Tensor* out_view = nullptr, bool x_needs_grad = true) {
    Op op;
    op.kind = OP_CONV;
    crfr_conv_desc& d = op.cd;
    d.n = x.n; d.h = x.h; d.w = x.w; d.cin = x.c; d.cout = cout; d.k = k; d.stride = stride; d.pad = pad;
    d.transposed = transposed ? 1 : 0;
    if (!transposed) {
      d.oh = (x.h + 2 * pad - k) / stride + 1;
      d.ow = (x.w + 2 * pad - k) / stride + 1;
    } else {
      d.oh = x.h * stride;  // k=7, s=4, p=2, output_padding=1 -> exactly 4x
      d.ow = x.w * stride;
    }
    Tensor y = out_view ? *out_view : new_tensor(x.n, d.oh, d.ow, cout);
    d.in_ld = x.ld; d.out_ld = y.ld;
    op.cin_pad = x.c < 8 ? 4 : x.c;
    void* wp = pack(w_idx, cout, x.c, k, op.cin_pad, transposed, false);
    float* stats = nullptr;
    if (stats_out) {
      stats = (float*)alloc((size_t)x.n * cout * 2 * sizeof(float));
      *stats_out = stats;
    }
    if (run()) {
      // (Finalising the statistics inside the normalisation pass that follows instead of by stats_finalize_kernel was
      // measured and dropped: every CTA of that pass then sums the partial slots of its image before its first pixel,
      // 66 us against 49 us + a 4.7 us finalize launch per layer.)
      check(crfr_conv_fwd(engine, &d, x.p, wp, op.cin_pad, b_idx >= 0 ? params[b_idx] : nullptr, y.p, nullptr, stats,
                          kEps, scratch, scratch_bytes, st));
    }
    op.a = x; op.out = y; op.w_idx = w_idx; op.b_idx = b_idx; op.x_needs_grad = x_needs_grad;
    tape.push_back(op);
    return y;
  }

  float* stats_of(const Tensor& y) {
    float* stats = (float*)alloc((size_t)y.n * y.c * 2 * sizeof(float));
    if (run()) check(crfr_norm_stats(y.p, y.n, y.h * y.w, y.c, y.ld, kEps, stats, scratch, scratch_bytes, st));
    return stats;
  }

  Tensor norm_act(const Tensor& y, float* stats, int g_idx, int beta_idx, int alpha_idx, const Tensor* res,
                  const Tensor* out_view = nullptr) {
    Tensor out = out_view ? *out_view : new_tensor(y.n, y.h, y.w, y.c);
    if (run())
      check(crfr_norm_act_fwd(y.p, y.ld, stats, g_idx >= 0 ? params[g_idx] : nullptr,
                              beta_idx >= 0 ? params[beta_idx] : nullptr, alpha_idx >= 0 ? params[alpha_idx] : nullptr,
                              0, res ? res->p : nullptr, res ? res->ld : 8, out.p, out.ld, y.n, y.h * y.w, y.c, st));
    Op op;
    op.kind = OP_NORM;
    op.a = y; op.out = out; op.stats = stats; op.g_idx = g_idx; op.beta_idx = beta_idx; op.alpha_idx = alpha_idx;
    op.has_res = res != nullptr;
    if (res) op.b = *res;
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

  Tensor upadd(const Tensor& up, const Tensor& low, const Tensor* out_view = nullptr) {
    Tensor out = out_view ? *out_view : new_tensor(up.n, up.h, up.w, up.c);
    if (run()) check(crfr_upnearest2_add_fwd(up.p, up.ld, low.p, low.ld, out.p, out.ld, low.n, low.h, low.w, low.c, st));
    Op op;
    op.kind = OP_UPADD; op.a = up; op.b = low; op.out = out;
    tape.push_back(op);
    return out;
  }

  // ---- network pieces ----
  Tensor res_block(const Tensor& x, int base) {   // _Residual_Block, FSRnet.py:75-98
    float* s1; float* s2;
    Tensor y1 = conv(x, base + RB_CONV1, -1, x.c, 3, 1, 1, false, &s1);
    Tensor a1 = norm_act(y1, s1, base + RB_IN1_W, base + RB_IN1_B, base + RB_RELU, nullptr);
    Tensor y2 = conv(a1, base + RB_CONV2, -1, x.c, 3, 1, 1, false, &s2);
    return norm_act(y2, s2, base + RB_IN2_W, base + RB_IN2_B, base + RB_RELU_OUT, &x);
  }
  Tensor res_stack(Tensor x, int base, int times) {
    for (int t = 0; t < times; ++t)
      for (int b = 0; b < 3; ++b) x = res_block(x, base + 8 * b);
    return x;
  }
  Tensor hg_block(const Tensor& x, int d, int s, int b) {  // BasicBlock :105-135
    float* s1; float* s2;
    Tensor y1 = conv(x, hg_param(d, s, b, 0), -1, 128, 3, 1, 1, false, &s1);
    Tensor a1 = norm_act(y1, s1, -1, -1, hg_param(d, s, b, 1), nullptr);
    Tensor y2 = conv(a1, hg_param(d, s, b, 2), -1, 128, 3, 1, 1, false, &s2);
    return norm_act(y2, s2, -1, -1, hg_param(d, s, b, 1), &x);
  }
  Tensor hg_seq(const Tensor& x, int d, int s) { return hg_block(hg_block(x, d, s, 0), d, s, 1); }
  Tensor hourglass(int n, const Tensor& x, const Tensor* out_view) {  // Hourglass._hour_glass_forward :200-212
    Tensor up1 = hg_seq(x, n - 1, 0);
    Tensor low1 = hg_seq(maxpool(x), n - 1, 1);
    Tensor low2 = n > 1 ? hourglass(n - 1, low1, nullptr) : hg_seq(low1, 0, 3);
    Tensor low3 = hg_seq(low2, n - 1, 2);
    return upadd(up1, low3, out_view);
  }

  // 64 -> 3 output convolution: fp32 NCHW result for the caller (+ optional bf16 NHWC4 copy for the stems)
  void img_conv(const Tensor& x, int w_idx, int b_idx, float* y_nchw, Tensor* y4) {
    Op op;
    op.kind = OP_IMGCONV;
    crfr_conv_desc& d = op.cd;
    d.n = x.n; d.h = x.h; d.w = x.w; d.cin = x.c; d.cout = 3; d.k = 3; d.stride = 1; d.pad = 1; d.oh = x.h; d.ow = x.w;
    d.in_ld = x.ld; d.out_ld = 4; d.transposed = 0;
    op.cin_pad = x.c;
    void* wp = pack(w_idx, 3, x.c, 3, x.c, false, false);
    if (run()) {
      if (y4) check(cudaMemsetAsync(y4->p, 0, (size_t)x.n * x.h * x.w * 4 * sizeof(bf16), st) == cudaSuccess ? CRFR_OK : CRFR_ECUDA);
      check(crfr_conv_fwd(engine, &d, x.p, wp, x.c, params[b_idx], y4 ? y4->p : nullptr, y_nchw, nullptr, kEps, scratch,
                          scratch_bytes, st));
    }
    op.a = x; op.w_idx = w_idx; op.b_idx = b_idx;
    if (y4) op.out = *y4;
    tape.push_back(op);
  }

  // fc (11) and fc_landmark (97), model/FSRnet.py:391-392: both 1x1 heads as ONE tcgen05 GEMM over the combined
  // [128 = 11 | 97 | zero pad][128] weight (fp32 NHWC result), then split + transposed into the two fp32 NCHW outputs
  void heads(const Tensor& x, float* landmark, float* parsing) {
    const long long npix = (long long)x.n * x.h * x.w;
    bf16* wc = (bf16*)alloc((size_t)kHeadsPad * 128 * sizeof(bf16));       // [co][ci]
    float* bc = (float*)alloc(kHeadsPad * sizeof(float));
    float* yf = (float*)alloc((size_t)npix * kHeadsPad * sizeof(float));   // fp32 NHWC
    if (run()) {
      heads_pack_kernel<<<crfr_cdiv(kHeadsPad * 128, 256), 256, 0, st>>>(params[P_FC_W], params[P_FC_B], params[P_FCL_W],
                                                                         params[P_FCL_B], wc, bc);
      CRFR_COUNT_LAUNCH();
      TcGemm g{x.p, x.n, x.h, x.w, 128, x.ld, wc, 1, 0, 1, kHeadsPad, kHeadsPad, yf, kHeadsPad, 1, bc};
      check(crfr_tc_gemm(g, st));
      const long long total = npix * 108;
      heads_split_kernel<<<crfr_cdiv(total, 256), 256, 0, st>>>(yf, parsing, landmark, x.n, x.h * x.w);
      CRFR_COUNT_LAUNCH();
      check(cudaGetLastError() == cudaSuccess ? CRFR_OK : CRFR_ECUDA);
    }
    Op op;
    op.kind = OP_HEADS; op.a = x;
    tape.push_back(op);
  }

  void prologue(int B, int S) {
    for (int i = 0; i < CRFR_FSRNET_NPARAMS; ++i) packed_fwd[i] = packed_bwd[i] = nullptr;
    // shared scratch: norm partials / wgrad accumulators of the largest layer
    scratch_bytes = crfr_norm_ws_bytes(B, S * S, 128) + sizeof(float) * 9 * 192 * 128 + 4096 + crfr_tc_wgrad_part_bytes();
    {  // the lowered edge layers (lowered_conv.cu) stage their im2col / partial-product buffers here
      const crfr_conv_desc shapes[5] = {
          {B, S, S, 64, 64, 3, 1, 1, S, S, 64, 64, 0},          // residual stacks (row-streaming kernels' scratch)
          {B, S, S, 3, 64, 3, 1, 1, S, S, 4, 64, 0},            // coarse conv_input
          {B, S, S, 64, 3, 3, 1, 1, S, S, 64, 4, 0},            // conv_mid / conv_out
          {B, S, S, 3, 128, 7, 4, 3, S / 4, S / 4, 4, 128, 0},  // stems
          {B, S / 4, S / 4, 64, 64, 7, 4, 2, S, S, 64, 64, 1}}; // deconv
      for (const crfr_conv_desc& sd : shapes) {
        size_t b = crfr_conv_workspace_bytes(&sd);
        if (b > scratch_bytes) scratch_bytes = b;
      }
      const size_t fb = crfr_conv_dgrad_norm_bwd_workspace_bytes(&shapes[0]);
      if (fb > scratch_bytes) scratch_bytes = fb;
    }
    scratch = alloc(scratch_bytes);
    if (training) {
      const crfr_conv_desc big = {B, S, S, 64, 64, 3, 1, 1, S, S, 64, 64, 0};
      scratch2_bytes = crfr_tc_workspace_bytes(&big) + sizeof(float) * 9 * 192 * 128 + 4096;
      scratch2 = alloc(scratch2_bytes);
    }
  }

  // fp32 NCHW 3-channel image -> bf16 NHWC4
  Tensor image_in(const float* src, int B, int S) {
    Tensor t = new_tensor(B, S, S, 4);
    t.c = 3;
    if (run()) check(crfr_nchw_f32_to_nhwc_bf16(src, t.p, B, 3, S, S, 4, 4, st));
    return t;
  }

  // ---- coarse SR network (:328-340): returns the 64-channel feature; coarse image -> y_nchw (+ bf16 copy y4) ----
  Tensor coarse_net(const Tensor& xin, float* coarse_nchw, Tensor* c4, bool x_grad) {
    float* s0;
    Tensor y = conv(xin, C_CONV_IN_W, C_CONV_IN_B, 64, 3, 1, 1, false, &s0, nullptr, x_grad);
    Tensor a = norm_act(y, s0, C_BN_MID_W, C_BN_MID_B, C_RELU, nullptr);
    a = res_stack(a, C_RES, 3);
    Tensor feat = norm_act(a, stats_of(a), C_BN_MID_W, C_BN_MID_B, -1, nullptr);
    img_conv(feat, C_CONV_MID_W, C_CONV_MID_B, coarse_nchw, c4);
    return feat;
  }

  // ---- fine SR encoder (:359-379) ----
  Tensor encoder_net(const Tensor& img4, const Tensor* out_view, bool x_grad) {
    float* se;
    Tensor ye = conv(img4, E_CONV_IN_W, E_CONV_IN_B, 64, 7, 4, 3, false, &se, nullptr, x_grad);
    Tensor ae = norm_act(ye, se, E_BN_MID_W, E_BN_MID_B, E_RELU, nullptr);
    ae = res_stack(ae, E_RES, 3);
    float* se2;
    Tensor ye2 = conv(ae, E_CONV_END_W, E_CONV_END_B, 64, 3, 1, 1, false, &se2);
    return norm_act(ye2, se2, E_BN_MID_W, E_BN_MID_B, E_RELU, nullptr, out_view);
  }

  // ---- prior estimation network (:408-426): 128-channel feature; heads -> landmark / parsing (fp32 NCHW) ----
  Tensor prior_net(const Tensor& img4, const Tensor* out_view, float* landmark, float* parsing, bool x_grad) {
    float* sp;
    Tensor yp = conv(img4, P_CONV_W, P_CONV_B, 128, 7, 4, 3, false, &sp, nullptr, x_grad);
    Tensor ap = norm_act(yp, sp, P_BN_W, P_BN_B, P_RELU, nullptr);
    ap = res_stack(ap, P_RES, 1);
    Tensor pe = hourglass(2, ap, out_view);
    heads(pe, landmark, parsing);
    return pe;
  }

  // ---- fine SR decoder (:448-459) ----
  void decoder_net(const Tensor& in192, float* out_nchw) {
    float* sd;
    Tensor yd = conv(in192, D_CONV_IN_W, D_CONV_IN_B, 64, 3, 1, 1, false, &sd);
    Tensor ad = norm_act(yd, sd, D_BN_MID_W, D_BN_MID_B, D_RELU, nullptr);
    float* sd2;
    Tensor yd2 = conv(ad, D_DECONV_W, D_DECONV_B, 64, 7, 4, 2, true, &sd2);
    Tensor ad2 = norm_act(yd2, sd2, D_BN_MID_W, D_BN_MID_B, D_RELU, nullptr);
    ad2 = res_stack(ad2, D_RES, 3);
    Tensor fd = norm_act(ad2, stats_of(ad2), D_BN_MID_W, D_BN_MID_B, -1, nullptr);
    img_conv(fd, D_CONV_OUT_W, D_CONV_OUT_B, out_nchw, nullptr);
  }

  void forward() {
    if (section >= 0) {
      forward_section();
      return;
    }
    const int B = io->batch, S = io->size;
    prologue(B, S);
    x4 = image_in(io->x, B, S);
    coarse4 = new_tensor(B, S, S, 4);
    coarse4.c = 3;
    coarse_net(x4, io->coarse, &coarse4, false);

    const int Q = S / 4;
    cat = new_tensor(B, Q, Q, 192);
    Tensor pe_view = view(cat, 0, 128), enc_view = view(cat, 128, 64);
    tape_enc_start = (int)tape.size();
    encoder_net(coarse4, &enc_view, true);
    prior_net(coarse4, &pe_view, io->landmark, io->parsing, true);

    // ---- decoder on cat(prior, encoder) (:505) ----
    tape_dec_start = (int)tape.size();
    Op cop;
    cop.kind = OP_CAT; cop.a = pe_view; cop.b = enc_view; cop.out = cat;
    tape.push_back(cop);
    decoder_net(cat, io->out);
  }

  // One sub-network on its own (Course_SR_Network / Fine_SR_Encoder / Prior_Estimation_Network / Fine_SR_Decoder
  // .forward of the reference, model/FSRnet.py:328-340, 359-379, 408-426, 448-459): fp32 NCHW in and out.
  void forward_section() {
    const int B = sio->batch, S = sio->size, Q = S / 4;
    prologue(B, S);
    tape_enc_start = tape_dec_start = -1;
    switch (section) {
      case CRFR_FSRNET_COARSE: {
        sec_in = image_in(sio->x, B, S);
        sec_feat = coarse_net(sec_in, sio->out[1], nullptr, want_dx);
        if (run()) check(crfr_nhwc_bf16_to_nchw_f32(sec_feat.p, sio->out[0], B, 64, S, S, sec_feat.ld, st));
        break;
      }
      case CRFR_FSRNET_ENCODER: {
        sec_in = image_in(sio->x, B, S);
        sec_feat = encoder_net(sec_in, nullptr, want_dx);
        if (run()) check(crfr_nhwc_bf16_to_nchw_f32(sec_feat.p, sio->out[0], B, 64, Q, Q, sec_feat.ld, st));
        break;
      }
      case CRFR_FSRNET_PRIOR: {
        sec_in = image_in(sio->x, B, S);
        sec_feat = prior_net(sec_in, nullptr, sio->out[1], sio->out[2], want_dx);
        if (run()) check(crfr_nhwc_bf16_to_nchw_f32(sec_feat.p, sio->out[0], B, 128, Q, Q, sec_feat.ld, st));
        break;
      }
      default: {   // CRFR_FSRNET_DECODER: [B,192,Q,Q] -> [B,3,S,S]
        sec_in = new_tensor(B, Q, Q, 192);
        if (run()) check(crfr_nchw_f32_to_nhwc_bf16(sio->x, sec_in.p, B, 192, Q, Q, 192, 192, st));
        decoder_net(sec_in, sio->out[0]);
        break;
      }
    }
  }

  // ---- backward helpers ----
  float* grad(int idx) { return (grads && idx >= 0) ? grads[idx] : nullptr; }
  void add_slot(const Tensor& t, bf16* p, int ld) { slots[t.id].push_back({p, ld}); }
  // reduce the slots of t to at most `max_slots`
  void squash(const Tensor& t, size_t max_slots) {
    std::vector<Slot>& s = slots[t.id];
    while (s.size() > max_slots) {
      const bool three = s.size() >= 3;
      const int cc = t.c < 8 ? 4 : t.c;
      bf16* out = (bf16*)alloc((size_t)t.n * t.h * t.w * cc * sizeof(bf16));
      size_t k = s.size();
      Slot a = s[k - 1], b = s[k - 2], c = three ? s[k - 3] : Slot{nullptr, cc};
      if (run()) check(crfr_add_n(a.p, a.ld, b.p, b.ld, c.p, c.ld, out, cc, (long long)t.n * t.h * t.w, cc, st));
      s.resize(k - (three ? 3 : 2));
      s.push_back({out, cc});
    }
  }
  bool has_grad(const Tensor& t) const { return t.id >= 0 && !slots[t.id].empty(); }

  void join_side() {   // the caller's stream waits for every forked weight gradient
    if (side_dirty && run()) {
      check(cudaEventRecord(side->join, side->st) == cudaSuccess ? CRFR_OK : CRFR_ECUDA);
      check(cudaStreamWaitEvent(st, side->join, 0) == cudaSuccess ? CRFR_OK : CRFR_ECUDA);
    }
    side_dirty = false;
  }

  void record_bucket(int k) {
    join_side();
    if (run() && io && io->bucket_events[k])
      check(cudaEventRecord((cudaEvent_t)io->bucket_events[k], st) == cudaSuccess ? CRFR_OK : CRFR_ECUDA);
  }

  void backward() {
    side = (exec && side_enabled()) ? side_stream() : nullptr;
    for (int i = (int)tape.size() - 1; i >= 0 && ok(); --i) {
      if (i == tape_dec_start - 1) record_bucket(0);   // every decoder op has run: its gradients are final
      if (i == tape_enc_start - 1) record_bucket(1);   // prior + encoder done
      Op& op = tape[i];
      switch (op.kind) {
        case OP_NORM: {
          if (op.bwd_done || !has_grad(op.out)) break;
          squash(op.out, 2);
          std::vector<Slot>& s = slots[op.out.id];
          const Tensor& y = op.a;
          const size_t bytes = (size_t)y.n * y.h * y.w * y.c * sizeof(bf16);
          // dz is only materialised when somebody consumes it (the residual branch) or a second gradient is summed in
          bf16* dz = (op.has_res || s.size() > 1) ? (bf16*)alloc(bytes) : nullptr;
          bf16* dy = (bf16*)alloc(bytes);
          if (run()) check(crfr_norm_act_bwd(s[0].p, s[0].ld, s.size() > 1 ? s[1].p : nullptr, s.size() > 1 ? s[1].ld : 8, y.p, y.ld,
                                  op.stats, op.g_idx >= 0 ? params[op.g_idx] : nullptr,
                                  op.beta_idx >= 0 ? params[op.beta_idx] : nullptr,
                                  op.alpha_idx >= 0 ? params[op.alpha_idx] : nullptr, 0,
                                  op.has_res ? op.b.p : nullptr, op.has_res ? op.b.ld : 8, dz, y.c, dy, y.c,
                                  grad(op.g_idx), grad(op.beta_idx), grad(op.alpha_idx), y.n, y.h * y.w, y.c, scratch,
                                  scratch_bytes, st));
          add_slot(y, dy, y.c);
          if (op.has_res) add_slot(op.b, dz, y.c);
          break;
        }
        case OP_CONV: {
          if (!has_grad(op.out)) break;
          squash(op.out, 1);
          Slot dy = slots[op.out.id][0];
          crfr_conv_desc d = op.cd;
          d.out_ld = dy.ld;
          // The bias of a convolution whose output is instance-normalised cancels in the normalisation: its gradient is
          // identically zero (the reference's autograd returns float noise of ~1e-9 relative for it).  The column sum over
          // the bf16 gradient map (42 us per 128-image layer at 128 x 128, and the one float-atomic kernel of the step) is
          // skipped for these layers: their bias gradient stays exactly zero.
          const bool null_bias = op.b_idx >= 0 && i + 1 < (int)tape.size() && tape[i + 1].kind == OP_NORM &&
                                 tape[i + 1].a.id == op.out.id && tape[i + 1].stats != nullptr;
          float* dbias = null_bias ? nullptr : grad(op.b_idx);
          // plain tcgen05 weight gradients go to the helper stream, behind this layer's dgrad (see SideStream)
          const bool forked = side && scratch2 && engine != CRFR_ENGINE_DIRECT && crfr_lowered_recipe(&d) == 0 &&
                              !d.transposed && crfr_tc_supported(2, d.h, d.w, d.cin, d.cout, d.k, d.stride, d.pad);
          if (!forked && run())
            check(crfr_conv_wgrad(engine, &d, op.a.p, dy.p, grad(op.w_idx), dbias, scratch, scratch_bytes, st));
          // The convolution's input is the output of the normalisation recorded just before it (every other consumer of
          // that tensor comes later in the tape, so its remaining gradient slots are complete): dgrad + the whole
          // normalisation backward as one operation - for the row-streaming shapes the first pass of the normalisation
          // backward runs inside the dgrad epilogue and the dgrad output never reaches memory.
          Op* nop = (i > 0 && tape[i - 1].kind == OP_NORM && tape[i - 1].out.id == op.a.id) ? &tape[i - 1] : nullptr;
          if (op.x_needs_grad && nop && !d.transposed && engine != CRFR_ENGINE_DIRECT &&
              (fuse_bwd < 0 ? crfr_opt(CRFR_OPT_FUSE_NORM_BWD) : fuse_bwd) &&
              crfr_lowered_recipe(&d) == 0 && crfr_rowconv_supported(d.h, d.w, d.cin, d.cout, d.k, d.stride, d.pad) &&
              crfr_rowconv_pair_supported(d.n, d.h) && op.a.c == nop->a.c) {
            const Tensor& x = op.a;
            const Tensor& yn = nop->a;
            squash(x, 1);
            std::vector<Slot>& xs = slots[x.id];
            const size_t bytes = (size_t)x.n * x.h * x.w * x.c * sizeof(bf16);
            bf16* dz = (bf16*)alloc(bytes);
            bf16* dyn = (bf16*)alloc(bytes);
            crfr_conv_desc dd = d;
            dd.in_ld = x.c;
            void* wt = pack(op.w_idx, d.cout, d.cin, d.k, 0, false, true);
            if (run())
              check(crfr_conv_dgrad_norm_bwd(engine, &dd, dy.p, wt, d.cout, xs.empty() ? nullptr : xs[0].p,
                                             xs.empty() ? 8 : xs[0].ld, yn.p, yn.ld, nop->stats,
                                             nop->g_idx >= 0 ? params[nop->g_idx] : nullptr,
                                             nop->beta_idx >= 0 ? params[nop->beta_idx] : nullptr,
                                             nop->alpha_idx >= 0 ? params[nop->alpha_idx] : nullptr, 0,
                                             nop->has_res ? nop->b.p : nullptr, nop->has_res ? nop->b.ld : 8, dz, x.c, dyn,
                                             x.c, grad(nop->g_idx), grad(nop->beta_idx), grad(nop->alpha_idx), scratch,
                                             scratch_bytes, st));
            xs.clear();
            add_slot(yn, dyn, x.c);
            if (nop->has_res) add_slot(nop->b, dz, x.c);
            nop->bwd_done = true;
          } else if (op.x_needs_grad) {
            const Tensor& x = op.a;
            const int xc = x.c < 8 ? 4 : x.c;
            bf16* dx = (bf16*)alloc((size_t)x.n * x.h * x.w * xc * sizeof(bf16));
            crfr_conv_desc dd = d;
            dd.in_ld = xc;
            void* wt = pack(op.w_idx, d.cout, d.cin, d.k, 0, d.transposed != 0, true);
            const int cout_pad = d.cout;
            if (run()) check(crfr_conv_dgrad(engine, &dd, dy.p, wt, cout_pad, dx, scratch, scratch_bytes, st));
            add_slot(x, dx, xc);
          }
          if (forked && run()) {
            check(cudaEventRecord(side->fork, st) == cudaSuccess ? CRFR_OK : CRFR_ECUDA);
            check(cudaStreamWaitEvent(side->st, side->fork, 0) == cudaSuccess ? CRFR_OK : CRFR_ECUDA);
            check(crfr_conv_wgrad(engine, &d, op.a.p, dy.p, grad(op.w_idx), dbias, scratch2, scratch2_bytes,
                                  side->st));
            side_dirty = true;
          }
          break;
        }
        case OP_POOL: {
          if (!has_grad(op.out)) break;
          squash(op.out, 1);
          Slot g = slots[op.out.id][0];
          const Tensor& x = op.a;
          bf16* dx = (bf16*)alloc((size_t)x.n * x.h * x.w * x.c * sizeof(bf16));
          if (run()) check(crfr_maxpool2_bwd(x.p, x.ld, g.p, g.ld, dx, x.c, x.n, x.h, x.w, x.c, st));
          add_slot(x, dx, x.c);
          break;
        }
        case OP_UPADD: {
          if (!has_grad(op.out)) break;
          squash(op.out, 1);
          Slot g = slots[op.out.id][0];
          const Tensor& low = op.b;
          bf16* dlow = (bf16*)alloc((size_t)low.n * low.h * low.w * low.c * sizeof(bf16));
          if (run()) check(crfr_upnearest2_bwd(g.p, g.ld, dlow, low.c, low.n, low.h, low.w, low.c, st));
          add_slot(op.a, g.p, g.ld);
          add_slot(low, dlow, low.c);
          break;
        }
        case OP_CAT: {
          if (!has_grad(op.out)) break;
          squash(op.out, 1);
          Slot g = slots[op.out.id][0];
          add_slot(op.a, g.p, g.ld);
          add_slot(op.b, g.p + op.a.c, g.ld);
          break;
        }
        case OP_HEADS: {
          if (!d_heads) break;
          const Tensor& x = op.a;
          const long long npix = (long long)x.n * x.h * x.w;
          // combined [.., 128] gradient buffer: parsing channels 0..10, landmark 11..107, zero padding 108..127
          float* G = (float*)scratch;                       // [ci = 128][co = 128] fp32
          bf16* wt = (bf16*)alloc((size_t)128 * kHeadsPad * sizeof(bf16));   // [ci][co]: rows of fc, fc_landmark, zeros
          bf16* dx = (bf16*)alloc((size_t)npix * x.c * sizeof(bf16));
          if (run()) {
            check(cudaMemsetAsync(G, 0, sizeof(float) * 128 * kHeadsPad, st) == cudaSuccess ? CRFR_OK : CRFR_ECUDA);
            TcWgrad wg{x.p, x.n, x.h, x.w, 128, x.ld, d_heads, kHeadsPad, kHeadsPad, 0, G};
            const size_t part_off = (sizeof(float) * 128 * kHeadsPad + 255) & ~(size_t)255;
            wg.part = (float*)((uint8_t*)scratch + part_off);
            wg.part_bytes = scratch_bytes - part_off;
            check(crfr_tc_wgrad_raw(wg, st));
            heads_unpack_kernel<<<crfr_cdiv(108 * 128, 256), 256, 0, st>>>(G, grad(P_FC_W), grad(P_FCL_W));
            CRFR_COUNT_LAUNCH();
            if (grad(P_FC_B)) check(crfr_colsum(d_heads, kHeadsPad, 11, npix, grad(P_FC_B), scratch, scratch_bytes, st));
            if (grad(P_FCL_B)) check(crfr_colsum(d_heads + 11, kHeadsPad, 97, npix, grad(P_FCL_B), scratch, scratch_bytes, st));
            check(cudaMemsetAsync(wt, 0, (size_t)128 * kHeadsPad * sizeof(bf16), st) == cudaSuccess ? CRFR_OK : CRFR_ECUDA);
            check(crfr_pack_weight_cols(params[P_FC_W], wt, 128, 11, kHeadsPad, 0, st));
            check(crfr_pack_weight_cols(params[P_FCL_W], wt, 128, 97, kHeadsPad, 11, st));
            TcGemm g{d_heads, x.n, x.h, x.w, kHeadsPad, kHeadsPad, wt, 1, 0, 1, 128, 128, dx, x.c, 0, nullptr};
            check(crfr_tc_gemm(g, st));
          }
          add_slot(x, dx, x.c);
          break;
        }
        case OP_IMGCONV: {
          // gradient of the 3-channel image: explicit (loss / caller) + consumers' slots if it fed the stems
          // The 3-element bias gradient is a sum with heavy cancellation (|sum| ~ 1e-3 of sum|.|): the explicit part is
          // summed in fp32 from the fp32 loss gradient by the caller (mse97 / nchw_chansum), the stems' contributions
          // are summed slot by slot here - never from the bf16-rounded total.
          const bool is_coarse = op.out.p != nullptr;
          bf16* g = is_coarse ? d_coarse4 : d_out4;
          if (is_coarse && has_grad(op.out)) {
            if (run() && grad(op.b_idx))
              for (const Slot& sl : slots[op.out.id])
                check(crfr_colsum(sl.p, sl.ld, 3, (long long)op.cd.n * op.cd.h * op.cd.w, grad(op.b_idx), scratch, scratch_bytes,
                                 st));
            if (g) add_slot(op.out, g, 4);
            squash(op.out, 1);
            g = slots[op.out.id][0].p;
          }
          if (!g) break;
          crfr_conv_desc d = op.cd;
          d.out_ld = 4;
          if (run() && grad(op.w_idx))
            check(crfr_conv_wgrad(engine, &d, op.a.p, g, grad(op.w_idx), nullptr, scratch, scratch_bytes, st));
          const Tensor& x = op.a;
          bf16* dx = (bf16*)alloc((size_t)x.n * x.h * x.w * x.c * sizeof(bf16));
          void* wt = pack(op.w_idx, 3, x.c, 3, 0, false, true);
          crfr_conv_desc dd = d;
          dd.in_ld = x.c;
          if (run()) check(crfr_conv_dgrad(engine, &dd, g, wt, 4, dx, scratch, scratch_bytes, st));
          add_slot(x, dx, x.c);
          break;
        }
      }
    }
    record_bucket(2);
  }
};

__global__ void pack_cols_kernel(const float* __restrict__ w, bf16* __restrict__ dst, int cin, int rows, int ld,
                                 int coff) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;  // over rows*cin; w is [rows][cin]
  if (i >= rows * cin) return;
  int r = i / cin, ci = i - r * cin;
  dst[(long long)ci * ld + coff + r] = __float2bfloat16_rn(w[i]);
}

__global__ void total_loss_kernel(float* losses, float w_pix, float inv_div) {
  losses[0] = (w_pix * losses[1] + w_pix * losses[2] + losses[3] + losses[4]) * inv_div;
}

void init_net(Net& net, int engine, const float* const* params, float* const* grads, const crfr_fsrnet_io* io,
              void* ws, size_t ws_bytes, cudaStream_t st, bool exec, bool training) {
  net.engine = engine; net.params = params; net.grads = grads; net.io = io; net.st = st;
  net.ws = (uint8_t*)ws; net.ws_bytes = ws_bytes; net.exec = exec; net.training = training;
}

int check_io(const crfr_fsrnet_io* io, const char* who, bool need_tensors = true) {
  CRFR_CHECK_ARG(io && io->batch > 0 && io->size >= 32 && io->size % 16 == 0, "%s: batch/size invalid (size must be a multiple of 16, >= 32)", who);
  // the backward pass reads neither the input nor the outputs (everything it needs was saved in the workspace)
  CRFR_CHECK_ARG(!need_tensors || (io->x && io->coarse && io->out && io->landmark && io->parsing), "%s: null tensor pointer", who);
  return CRFR_OK;
}

}  // namespace

int crfr_pack_weight_cols(const float* w, void* dst, int cin, int rows, int ld, int coff, cudaStream_t st) {
  pack_cols_kernel<<<crfr_cdiv(rows * cin, 256), 256, 0, st>>>(w, (bf16*)dst, cin, rows, ld, coff);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

namespace {

// allocate the output-gradient buffers right after the forward region (same order in sizing and execution)
void alloc_out_grads(Net& net, bool coarse, bool out, bool heads) {
  const int B = net.io ? net.io->batch : net.sio->batch, S = net.io ? net.io->size : net.sio->size, Q = S / 4;
  net.d_coarse4 = coarse ? (bf16*)net.alloc((size_t)B * S * S * 4 * sizeof(bf16)) : nullptr;
  net.d_out4 = out ? (bf16*)net.alloc((size_t)B * S * S * 4 * sizeof(bf16)) : nullptr;
  net.d_heads = heads ? (bf16*)net.alloc((size_t)B * Q * Q * kHeadsPad * sizeof(bf16)) : nullptr;
}

// Dry run of the program over the real arena: collects the weight-pack jobs of the forward (and backward) pass and
// issues them as one batch.  The arena is a deterministic bump allocator, so the real run finds every packed weight at
// the offset the dry run gave it.
int collect_packs(std::vector<crfr_pack_job>& jobs, int engine, const float* const* params, const crfr_fsrnet_io* io,
                  void* ws, size_t ws_bytes, cudaStream_t st, bool training, bool backward, bool og_coarse, bool og_out,
                  bool og_heads) {
  Net dry;
  init_net(dry, engine, params, nullptr, io, ws, ws_bytes, st, false, training);
  dry.collect = &jobs;
  dry.forward();
  if (backward && dry.ok()) {
    alloc_out_grads(dry, og_coarse, og_out, og_heads);
    dry.backward();
  }
  return dry.err;
}
int pack_all(int engine, const float* const* params, const crfr_fsrnet_io* io, void* ws, size_t ws_bytes, cudaStream_t st,
             bool training, bool backward, bool og_coarse, bool og_out, bool og_heads) {
  std::vector<crfr_pack_job> jobs;
  CRFR_TRY(collect_packs(jobs, engine, params, io, ws, ws_bytes, st, training, backward, og_coarse, og_out, og_heads));
  return crfr_pack_weight_batch(jobs.data(), (int)jobs.size(), st);
}

}  // namespace

extern "C" size_t crfr_fsrnet_workspace_bytes(int batch, int size, int training) {
  if (batch <= 0 || size < 32 || size % 16) return 0;
  crfr_fsrnet_io io = {};
  io.batch = batch; io.size = size;
  size_t need = 0;
  for (int fuse = 0; fuse < 2; ++fuse) {   // the backward's arena layout depends on the fused / unfused boundary operation:
    Net net;                               // a workspace of this size serves either setting of the option
    init_net(net, CRFR_ENGINE_AUTO, nullptr, nullptr, &io, nullptr, ~(size_t)0 >> 2, nullptr, false, training != 0);
    net.fuse_bwd = fuse;
    net.forward();
    if (training) {
      alloc_out_grads(net, true, true, true);
      net.backward();
    }
    if (net.off > need) need = net.off;
    if (!training) break;
  }
  return need + 65536;
}

namespace {
// the stored forward tensors of a program run (dry or not) whose workspace base is the null pointer
int fill_tape(const Net& net, crfr_tape_entry* entries, int max_entries) {
  const int count = (int)net.tape.size();
  for (int i = 0; i < count && i < max_entries && entries; ++i) {
    const Op& op = net.tape[i];
    crfr_tape_entry& e = entries[i];
    const Tensor& t = op.out;
    e.kind = (int)op.kind;
    e.n = t.n; e.h = t.h; e.w = t.w; e.c = t.c; e.ld = t.ld;
    e.out_off = t.p ? (long long)((uint8_t*)t.p - (uint8_t*)nullptr) : -1;
    e.in_off = op.a.p ? (long long)((uint8_t*)op.a.p - (uint8_t*)nullptr) : -1;
    e.stats_off = op.stats ? (long long)((uint8_t*)op.stats - (uint8_t*)nullptr) : -1;
    e.w_idx = op.w_idx;
    e.has_res = op.has_res ? 1 : 0;
  }
  return count;
}
}  // namespace

// Layout of the saved forward tensors in the workspace (a dry run: nothing is launched).  Parity tests read the stored
// bf16 activations through this table and replay them into the CPU oracle (teacher-forced forward / backward checks).
extern "C" int crfr_fsrnet_tape(int batch, int size, int training, crfr_tape_entry* entries, int max_entries) {
  if (batch <= 0 || size < 32 || size % 16) return -1;
  crfr_fsrnet_io io = {};
  io.batch = batch; io.size = size;
  Net net;
  init_net(net, CRFR_ENGINE_AUTO, nullptr, nullptr, &io, nullptr, ~(size_t)0 >> 2, nullptr, false, training != 0);
  net.forward();
  return fill_tape(net, entries, max_entries);
}

extern "C" int crfr_fsrnet_forward(int engine, const float* const* host_params, const crfr_fsrnet_io* io,
                                   int training, void* ws, size_t ws_bytes, void* stream) {
  CRFR_TRY(check_io(io, "fsrnet_forward"));
  CRFR_CHECK_ARG(host_params && ws, "fsrnet_forward: null pointer");
  CRFR_TRY(pack_all(engine, host_params, io, ws, ws_bytes, (cudaStream_t)stream, training != 0, false, false, false, false));
  Net net;
  init_net(net, engine, host_params, nullptr, io, ws, ws_bytes, (cudaStream_t)stream, true, training != 0);
  net.packs_done = true;
  net.forward();
  return net.err;
}

extern "C" int crfr_fsrnet_backward(int engine, const float* const* host_params, float* const* host_grads,
                                    const crfr_fsrnet_io* io, const float* d_coarse, const float* d_out,
                                    const float* d_landmark, const float* d_parsing, void* ws, size_t ws_bytes,
                                    void* stream) {
  CRFR_TRY(check_io(io, "fsrnet_backward", false));
  CRFR_CHECK_ARG(host_params && host_grads && ws, "fsrnet_backward: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  Net net;
  init_net(net, engine, host_params, host_grads, io, ws, ws_bytes, st, false, true);
  net.forward();  // dry run: rebuild the tape and the saved-activation offsets
  if (!net.ok()) return net.err;
  net.exec = true;
  const int B = io->batch, S = io->size, Q = S / 4;
  alloc_out_grads(net, d_coarse != nullptr, d_out != nullptr, d_landmark || d_parsing);
  if (!net.ok()) return net.err;
  if (d_coarse) {
    CRFR_TRY(crfr_nchw_f32_to_nhwc_bf16(d_coarse, net.d_coarse4, B, 3, S, S, 4, 4, stream));
    if (host_grads[C_CONV_MID_B])
      CRFR_TRY(crfr_nchw_chansum(d_coarse, B, 3, S * S, host_grads[C_CONV_MID_B], net.scratch, net.scratch_bytes, st));
  }
  if (d_out) {
    CRFR_TRY(crfr_nchw_f32_to_nhwc_bf16(d_out, net.d_out4, B, 3, S, S, 4, 4, stream));
    if (host_grads[D_CONV_OUT_B])
      CRFR_TRY(crfr_nchw_chansum(d_out, B, 3, S * S, host_grads[D_CONV_OUT_B], net.scratch, net.scratch_bytes, st));
  }
  if (net.d_heads) {
    CRFR_CUDA(cudaMemsetAsync(net.d_heads, 0, (size_t)B * Q * Q * kHeadsPad * sizeof(bf16), st));
    if (d_parsing) CRFR_TRY(crfr_nchw_f32_to_nhwc_bf16(d_parsing, net.d_heads, B, 11, Q, Q, kHeadsPad, 11, stream));
    if (d_landmark) CRFR_TRY(crfr_nchw_f32_to_nhwc_bf16(d_landmark, net.d_heads + 11, B, 97, Q, Q, kHeadsPad, 97, stream));
  }
  net.backward();
  return net.err;
}

// ---- sub-networks on their own -----------------------------------------------------------------------------------
namespace {

int check_section(const crfr_fsrnet_section_io* io, const char* who) {
  CRFR_CHECK_ARG(io && io->section >= 0 && io->section <= 3 && io->batch > 0 && io->size >= 32 && io->size % 16 == 0,
                 "%s: section/batch/size invalid (size must be a multiple of 16, >= 32)", who);
  const int nout = io->section == CRFR_FSRNET_COARSE ? 2 : (io->section == CRFR_FSRNET_PRIOR ? 3 : 1);
  CRFR_CHECK_ARG(io->x, "%s: null input", who);
  for (int i = 0; i < nout; ++i) CRFR_CHECK_ARG(io->out[i], "%s: null output %d", who, i);
  return CRFR_OK;
}

void init_section(Net& net, int engine, const float* const* params, float* const* grads, const crfr_fsrnet_section_io* sio,
                  void* ws, size_t ws_bytes, cudaStream_t st, bool exec, bool training) {
  init_net(net, engine, params, grads, nullptr, ws, ws_bytes, st, exec, training);
  net.section = sio->section;
  net.sio = sio;
}

}  // namespace

extern "C" size_t crfr_fsrnet_section_workspace_bytes(int section, int batch, int size, int training) {
  if (section < 0 || section > 3 || batch <= 0 || size < 32 || size % 16) return 0;
  crfr_fsrnet_section_io sio = {};
  sio.section = section; sio.batch = batch; sio.size = size;
  size_t need = 0;
  for (int fuse = 0; fuse < 2; ++fuse) {   // either setting of option fuse_norm_bwd (see crfr_fsrnet_workspace_bytes)
    Net net;
    init_section(net, CRFR_ENGINE_AUTO, nullptr, nullptr, &sio, nullptr, ~(size_t)0 >> 2, nullptr, false, training != 0);
    net.want_dx = true;
    net.fuse_bwd = fuse;
    net.forward();
    if (training) {
      alloc_out_grads(net, false, section == CRFR_FSRNET_COARSE || section == CRFR_FSRNET_DECODER,
                      section == CRFR_FSRNET_PRIOR);
      if (section != CRFR_FSRNET_DECODER) {   // gradient of the feature output, converted to bf16 NHWC
        net.add_slot(net.sec_feat, (bf16*)net.alloc((size_t)batch * net.sec_feat.h * net.sec_feat.w * net.sec_feat.c * sizeof(bf16)),
                     net.sec_feat.c);
      }
      net.backward();
      if (net.has_grad(net.sec_in)) net.squash(net.sec_in, 1);
    }
    if (net.off > need) need = net.off;
    if (!training) break;
  }
  return need + 65536;
}

extern "C" int crfr_fsrnet_section_forward(int engine, const float* const* host_params, const crfr_fsrnet_section_io* io,
                                           int training, void* ws, size_t ws_bytes, void* stream) {
  CRFR_TRY(check_section(io, "fsrnet_section_forward"));
  CRFR_CHECK_ARG(host_params && ws, "fsrnet_section_forward: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  {   // batched weight packing (dry run collects the jobs)
    std::vector<crfr_pack_job> jobs;
    Net dry;
    init_section(dry, engine, host_params, nullptr, io, ws, ws_bytes, st, false, training != 0);
    dry.want_dx = true;
    dry.collect = &jobs;
    dry.forward();
    if (!dry.ok()) return dry.err;
    CRFR_TRY(crfr_pack_weight_batch(jobs.data(), (int)jobs.size(), st));
  }
  Net net;
  init_section(net, engine, host_params, nullptr, io, ws, ws_bytes, st, true, training != 0);
  net.want_dx = true;
  net.packs_done = true;
  net.forward();
  return net.err;
}

extern "C" int crfr_fsrnet_section_backward(int engine, const float* const* host_params, float* const* host_grads,
                                            const crfr_fsrnet_section_io* io, const float* const* d_out, float* dx,
                                            void* ws, size_t ws_bytes, void* stream) {
  CRFR_TRY(check_section(io, "fsrnet_section_backward"));
  CRFR_CHECK_ARG(host_params && host_grads && ws && d_out, "fsrnet_section_backward: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int B = io->batch, S = io->size, Q = S / 4, sec = io->section;
  Net net;
  init_section(net, engine, host_params, host_grads, io, ws, ws_bytes, st, false, true);
  net.want_dx = dx != nullptr;   // (only decides whether the first layer's input gradient is computed; the forward
  net.forward();                 //  layout does not depend on it)  dry run: rebuild the tape and the saved offsets
  if (!net.ok()) return net.err;
  net.exec = true;
  const float* d_img = sec == CRFR_FSRNET_COARSE ? d_out[1] : (sec == CRFR_FSRNET_DECODER ? d_out[0] : nullptr);
  const float* d_feat = sec == CRFR_FSRNET_DECODER ? nullptr : d_out[0];
  const float* d_lm = sec == CRFR_FSRNET_PRIOR ? d_out[1] : nullptr;
  const float* d_ps = sec == CRFR_FSRNET_PRIOR ? d_out[2] : nullptr;
  alloc_out_grads(net, false, sec == CRFR_FSRNET_COARSE || sec == CRFR_FSRNET_DECODER, sec == CRFR_FSRNET_PRIOR);
  bf16* gfeat = nullptr;
  if (sec != CRFR_FSRNET_DECODER)
    gfeat = (bf16*)net.alloc((size_t)B * net.sec_feat.h * net.sec_feat.w * net.sec_feat.c * sizeof(bf16));
  if (!net.ok()) return net.err;
  if (net.d_out4) {
    if (d_img) {
      CRFR_TRY(crfr_nchw_f32_to_nhwc_bf16(d_img, net.d_out4, B, 3, S, S, 4, 4, stream));
      float* db = host_grads[sec == CRFR_FSRNET_COARSE ? C_CONV_MID_B : D_CONV_OUT_B];
      if (db) CRFR_TRY(crfr_nchw_chansum(d_img, B, 3, S * S, db, net.scratch, net.scratch_bytes, st));
    } else {
      net.d_out4 = nullptr;   // no gradient for the image output: the image conv is skipped
    }
  }
  if (net.d_heads) {
    if (d_lm || d_ps) {
      CRFR_CUDA(cudaMemsetAsync(net.d_heads, 0, (size_t)B * Q * Q * kHeadsPad * sizeof(bf16), st));
      if (d_ps) CRFR_TRY(crfr_nchw_f32_to_nhwc_bf16(d_ps, net.d_heads, B, 11, Q, Q, kHeadsPad, 11, stream));
      if (d_lm) CRFR_TRY(crfr_nchw_f32_to_nhwc_bf16(d_lm, net.d_heads + 11, B, 97, Q, Q, kHeadsPad, 97, stream));
    } else {
      net.d_heads = nullptr;
    }
  }
  if (gfeat && d_feat) {
    const Tensor& f = net.sec_feat;
    CRFR_TRY(crfr_nchw_f32_to_nhwc_bf16(d_feat, gfeat, B, f.c, f.h, f.w, f.c, f.c, stream));
    net.add_slot(f, gfeat, f.c);
  }
  net.backward();
  if (!net.ok()) return net.err;
  if (dx) {
    const Tensor& x = net.sec_in;
    if (!net.has_grad(x)) {
      crfr_set_error("fsrnet_section_backward: no gradient reached the section input");
      return CRFR_EINVAL;
    }
    net.squash(x, 1);
    if (!net.ok()) return net.err;
    const Slot g = net.slots[x.id][0];
    CRFR_TRY(crfr_nhwc_bf16_to_nchw_f32(g.p, dx, B, x.c, x.h, x.w, g.ld, stream));
  }
  return net.err;
}

namespace {

constexpr int kIdCrop = 8;   // crop(t) = t[:, :, 8:120, 8:120] of the 128 x 128 output

size_t fsr_arena_bytes(int batch, int size) {
  return (crfr_fsrnet_workspace_bytes(batch, size, 1) + 4095) & ~(size_t)4095;
}

crfr_ir_identity_args id_args(int engine, const crfr_fsrnet_io* io, const crfr_fsrnet_id_io* id, float* losses,
                              void* ws, size_t ws_bytes, cudaStream_t st) {
  crfr_ir_identity_args a;
  a.engine = engine; a.layers = id->teacher_layers; a.se = id->teacher_se; a.batch = io->batch;
  a.params = id->teacher_params; a.buffers = id->teacher_buffers;
  a.hr = io->hr; a.sr = io->out; a.src_size = io->size; a.crop = kIdCrop; a.terms = id->terms;
  a.gscale = id->w_id * id->id_scale; a.w_id = id->w_id; a.id_scale = id->id_scale;
  a.losses = losses; a.ws = ws; a.ws_bytes = ws_bytes; a.st = st;
  return a;
}

// forward + losses + backward of crfr_fsrnet_train_step; id != NULL adds the identity term of crfr_fsrnet_id_train_step,
// whose teacher programs use the workspace after the FSRNet arena
int train_step(int engine, const float* const* host_params, float* const* host_grads, const crfr_fsrnet_io* io,
               const crfr_fsrnet_id_io* id, float* losses, void* ws, size_t ws_bytes, cudaStream_t st) {
  const size_t fsr_bytes = id ? fsr_arena_bytes(io->batch, io->size) : ws_bytes;
  if (fsr_bytes > ws_bytes) {
    crfr_set_error("fsrnet_id_train_step: workspace too small (%zu given, crfr_fsrnet_id_workspace_bytes)", ws_bytes);
    return CRFR_EWORKSPACE;
  }
  crfr_ir_identity_args ia{};
  if (id) ia = id_args(engine, io, id, losses, (uint8_t*)ws + fsr_bytes, ws_bytes - fsr_bytes, st);
  {   // every weight pack of the step - FSRNet both directions, the teacher's two forwards - in one batched launch
    std::vector<crfr_pack_job> jobs;
    CRFR_TRY(collect_packs(jobs, engine, host_params, io, ws, fsr_bytes, st, true, true, true, true, true));
    if (id) CRFR_TRY(crfr_ir_identity(ia, false, &jobs, nullptr, nullptr));
    CRFR_TRY(crfr_pack_weight_batch(jobs.data(), (int)jobs.size(), st));
  }
  Net net;
  init_net(net, engine, host_params, host_grads, io, ws, fsr_bytes, st, true, true);
  net.packs_done = true;
  net.forward();
  if (!net.ok()) return net.err;
  const int B = io->batch, S = io->size, Q = S / 4;
  alloc_out_grads(net, true, true, true);
  if (!net.ok()) return net.err;
  // FSR_main.py:233-234: (w*mse(sr,hr) + w*mse(coarse,hr) + landmark + ce) / (2*train_batch)
  const float inv = 1.f / io->loss_div;
  CRFR_TRY(crfr_loss_mse97_chan(io->out, io->hr, B, 3, S * S, io->w_pix * inv, losses + 1, net.d_out4, 4,
                                host_grads[D_CONV_OUT_B], net.scratch, net.scratch_bytes, st));
  CRFR_TRY(crfr_loss_mse97_chan(io->coarse, io->hr, B, 3, S * S, io->w_pix * inv, losses + 2, net.d_coarse4, 4,
                                host_grads[C_CONV_MID_B], net.scratch, net.scratch_bytes, st));
  CRFR_CUDA(cudaMemsetAsync(net.d_heads, 0, (size_t)B * Q * Q * kHeadsPad * sizeof(bf16), st));
  CRFR_TRY(crfr_loss_landmark(io->landmark, io->heatmap, B, 97, Q * Q, inv, losses + 3, net.d_heads, kHeadsPad, 11,
                              net.scratch, net.scratch_bytes, st));
  CRFR_TRY(crfr_loss_ce2d(io->parsing, io->labels, B, 11, Q * Q, inv, losses + 4, net.d_heads, kHeadsPad, 0, net.scratch,
                          net.scratch_bytes, st));
  total_loss_kernel<<<1, 1, 0, st>>>(losses, io->w_pix, inv);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  if (id) {
    // the teacher's forwards on crop(hr) and crop(sr), the feature terms and its input gradient, which joins the pixel
    // loss's gradient at the output image (and the output convolution's bias gradient) before the FSRNet backward
    const void* dx4 = nullptr;
    CRFR_TRY(crfr_ir_identity(ia, true, nullptr, nullptr, &dx4));
    CRFR_TRY(crfr_mse97_add_window_grad(io->out, io->hr, B, 3, S, S, io->w_pix * inv, dx4, kIdSize, kIdSize, 4, kIdCrop,
                                        kIdCrop, net.d_out4, 4, host_grads[D_CONV_OUT_B], net.scratch, net.scratch_bytes,
                                        st));
  }
  net.backward();
  return net.err;
}

}  // namespace

extern "C" int crfr_fsrnet_train_step(int engine, const float* const* host_params, float* const* host_grads,
                                      const crfr_fsrnet_io* io, float* losses, void* ws, size_t ws_bytes,
                                      void* stream) {
  CRFR_TRY(check_io(io, "fsrnet_train_step"));
  CRFR_CHECK_ARG(host_params && host_grads && ws && losses, "fsrnet_train_step: null pointer");
  CRFR_CHECK_ARG(io->hr && io->heatmap && io->labels && io->loss_div > 0.f, "fsrnet_train_step: missing targets");
  return train_step(engine, host_params, host_grads, io, nullptr, losses, ws, ws_bytes, (cudaStream_t)stream);
}

extern "C" size_t crfr_fsrnet_id_workspace_bytes(int teacher_layers, int teacher_se, int batch, int size) {
  if (batch <= 0 || size != kIdSize + 2 * kIdCrop) return 0;
  crfr_fsrnet_io io = {};
  io.batch = batch; io.size = size;
  crfr_fsrnet_id_io id = {};
  id.teacher_layers = teacher_layers; id.teacher_se = teacher_se; id.terms = 31;
  crfr_ir_identity_args a = id_args(CRFR_ENGINE_AUTO, &io, &id, nullptr, nullptr, ~(size_t)0 >> 2, nullptr);
  size_t ir_bytes = 0;
  if (crfr_ir_identity(a, false, nullptr, &ir_bytes, nullptr) != CRFR_OK) return 0;
  return fsr_arena_bytes(batch, size) + ir_bytes;
}

// Where crfr_fsrnet_id_train_step leaves its tensors (include/crfr.h): the dry runs of train_step's two halves over the
// step's own layout - the FSRNet forward and its output gradients in the arena at 0, then crfr_ir_identity recording from
// inside, with its arena at fsr_arena_bytes
extern "C" int crfr_fsrnet_id_tape(int teacher_layers, int teacher_se, int batch, int size, int terms,
                                   crfr_tape_entry* entries, int max_entries) {
  if (crfr_fsrnet_id_workspace_bytes(teacher_layers, teacher_se, batch, size) == 0 || terms < 1 || terms > 31) return -1;
  crfr_fsrnet_io io = {};
  io.batch = batch; io.size = size;
  crfr_fsrnet_id_io id = {};
  id.teacher_layers = teacher_layers; id.teacher_se = teacher_se; id.terms = terms;
  const size_t fsr_bytes = fsr_arena_bytes(batch, size);
  Net net;
  init_net(net, CRFR_ENGINE_AUTO, nullptr, nullptr, &io, nullptr, fsr_bytes, nullptr, false, true);
  net.forward();
  alloc_out_grads(net, true, true, true);
  if (!net.ok()) return -1;
  std::vector<crfr_tape_entry> tape(net.tape.size());
  fill_tape(net, tape.data(), (int)tape.size());
  crfr_tape_entry d{};
  d.kind = 19;
  d.n = batch; d.h = size; d.w = size; d.c = 3; d.ld = 4;
  d.out_off = (long long)((uint8_t*)net.d_out4 - (uint8_t*)nullptr);
  d.in_off = d.stats_off = -1;
  d.w_idx = -1;
  tape.push_back(d);
  const crfr_ir_identity_args a = id_args(CRFR_ENGINE_AUTO, &io, &id, nullptr, (uint8_t*)nullptr + fsr_bytes,
                                          ~(size_t)0 >> 2, nullptr);
  if (crfr_ir_identity(a, false, nullptr, nullptr, nullptr, &tape) != CRFR_OK) return -1;
  const int count = (int)tape.size();
  for (int i = 0; i < count && i < max_entries && entries; ++i) entries[i] = tape[i];
  return count;
}

extern "C" int crfr_fsrnet_id_train_step(int engine, const float* const* host_params, float* const* host_grads,
                                         const crfr_fsrnet_io* io, const crfr_fsrnet_id_io* id, float* losses, void* ws,
                                         size_t ws_bytes, void* stream) {
  CRFR_TRY(check_io(io, "fsrnet_id_train_step"));
  CRFR_CHECK_ARG(io->size == kIdSize + 2 * kIdCrop,
                 "fsrnet_id_train_step: size %d unsupported (the identity term takes the 112 x 112 centre of a 128 x 128 "
                 "output)", io->size);
  CRFR_CHECK_ARG(host_params && host_grads && ws && losses && id && id->teacher_params && id->teacher_buffers,
                 "fsrnet_id_train_step: null pointer");
  CRFR_CHECK_ARG(io->hr && io->heatmap && io->labels && io->loss_div > 0.f, "fsrnet_id_train_step: missing targets");
  CRFR_CHECK_ARG(id->terms > 0 && id->terms < 32, "fsrnet_id_train_step: terms 0x%x must select 1 to 5 of the outputs "
                 "(embedding, x1, x2, x3, x4)", id->terms);
  CRFR_CHECK_ARG(id->id_scale > 0.f && id->id_scale <= 1.f, "fsrnet_id_train_step: id_scale %g not in (0, 1]",
                 (double)id->id_scale);
  CRFR_TRY(crfr_irnet_sizes(id->teacher_layers, id->teacher_se, nullptr, nullptr));   // the variant is supported
  const size_t need = crfr_fsrnet_id_workspace_bytes(id->teacher_layers, id->teacher_se, io->batch, io->size);
  if (ws_bytes < need) {
    crfr_set_error("fsrnet_id_train_step: workspace %zu < %zu (crfr_fsrnet_id_workspace_bytes)", ws_bytes, need);
    return CRFR_EWORKSPACE;
  }
  return train_step(engine, host_params, host_grads, io, id, losses, ws, ws_bytes, (cudaStream_t)stream);
}
