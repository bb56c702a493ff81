// Native ResNet_34 face-embedding network program (student / assistant / teacher of the residual knowledge
// distillation step): the whole forward and backward are sequenced here in C++ on one stream over a caller-provided
// workspace arena, exactly like fsrnet.cu - a tape of fused ops recorded by the forward and replayed in reverse.
//
// Layers: 7x7 s2 stem (lowered im2col + tcgen05 GEMM), 16 BasicBlocks of 3x3 convolutions on the tcgen05 implicit-GEMM
// engine (stage transitions: 3x3 s2 and 1x1 s2 through the lowered recipe 5), train-mode BatchNorm (+ReLU, +residual)
// as the n = 1 grouping of the fused normalise kernels with the running-statistics update, the 25088 -> 512 linear
// head as a tcgen05 GEMM over the NHWC-flattened feature (weights re-ordered from the reference's NCHW flatten), and
// BatchNorm1d on the embedding.
//
// The frozen IR teachers (DISTILLATION/model/model_irse.py: IR_50 / 101 / 152 and IR_SE_50 / 101 / 152) are a second
// program over the same ops: BN -> conv3x3 -> PReLU -> conv3x3(stride) -> BN [-> SEModule], plus a MaxPool2d(1, stride) /
// conv1x1+BN shortcut, 24 / 49 / 50 blocks.  Its backward (backward_ir) is the gradient with respect to the input image
// only: eval-mode BatchNorm couples no images, so it is a per-sample linear map of dgrads, per-channel scales, PReLU masks
// and, with SE, the per-image excitation and its squeeze path.
//
// ref: model/resnet.py:18-47 (BasicBlock), :152-225 (ResNet.__init__/_make_layer/forward), :231-236 (ResNet_34);
//      DISTILLATION/model/model_irse.py:49-66 (bottleneck_IR), SEModule and bottleneck_IR_SE, :101-126 (get_blocks),
//      :129-172 (Backbone).
#include <vector>

#include "common.cuh"
#include "crfr.h"
#include "internal.h"

namespace {

struct Tensor {
  bf16* p = nullptr;
  int n = 0, h = 0, w = 0, c = 0, ld = 0;
  int id = -1;
  float* bn_stats = nullptr;   // train-mode BatchNorm statistics of a convolution output, computed by its epilogue
};
struct Slot {
  bf16* p;
  int ld;
};
enum OpKind { OP_CONV, OP_BN, OP_LINEAR, OP_PRELU, OP_SUB2, OP_SE };
struct Op {
  OpKind kind;
  Tensor a, b, out;
  crfr_conv_desc cd;
  int w_idx = -1, b_idx = -1, g_idx = -1, beta_idx = -1, alpha_idx = -1;
  int cin_pad = 0;
  float* stats = nullptr;   // OP_SE: the excitation e [n][c]
  float* bn_stats = nullptr, *squeeze = nullptr;   // OP_SE: res_layer.4's (mean, rstd) [c][2], mean_hw(y) [n][c][2]
  bool relu = false, has_res = false, x_needs_grad = true;
};

// IR / IR-SE variants (DISTILLATION/model/model_irse.py:101-126): units per stage
bool ir_units_of(int num_layers, int units[4]) {
  static const int t50[4] = {3, 4, 14, 3}, t100[4] = {3, 13, 30, 3}, t152[4] = {3, 8, 36, 3};
  const int* t = num_layers == 50 ? t50 : num_layers == 100 ? t100 : num_layers == 152 ? t152 : nullptr;
  if (!t) return false;
  for (int l = 0; l < 4; ++l) units[l] = t[l];
  return true;
}
constexpr int kSeReduction = 16;   // SEModule(depth, 16): hidden widths 4, 8, 16, 32

constexpr int kFeat = 512, kEmb = 512;

// W [o][c*HW + hw] (fp32, reference flatten order) -> Wp [o][hw*C + c] and WpT [hw*C + c][o] (bf16); the optional fp32
// scales o_scale[o] and c_scale[c] multiply the weight before its rounding (BatchNorm scales folded into the input gradient)
__global__ void linear_pack_kernel(const float* __restrict__ w, bf16* __restrict__ wp, bf16* __restrict__ wpt, int O,
                                   int C, int HW, const float* __restrict__ o_scale = nullptr,
                                   const float* __restrict__ c_scale = nullptr) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long K = (long long)C * HW;
  if (i >= (long long)O * K) return;
  const int o = (int)(i / K);
  const long long k = i - (long long)o * K;       // hw*C + c
  const int hw = (int)(k / C), c = (int)(k - (long long)hw * C);
  float f = w[(long long)o * K + (long long)c * HW + hw];
  if (o_scale) f *= o_scale[o];
  if (c_scale) f *= c_scale[c];
  const bf16 v = __float2bfloat16_rn(f);
  if (wp) wp[i] = v;
  if (wpt) wpt[k * O + o] = v;
}

// dW [o][c*HW + hw] += G[hw*C + c][o]
__global__ void linear_unpack_kernel(const float* __restrict__ G, float* __restrict__ dw, int O, int C, int HW) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long K = (long long)C * HW;
  if (i >= (long long)O * K) return;
  const int o = (int)(i / K);
  const long long r = i - (long long)o * K;       // c*HW + hw
  const int c = (int)(r / HW), hw = (int)(r - (long long)c * HW);
  dw[i] += G[((long long)hw * C + c) * O + o];
}

// MaxPool2d(kernel 1, stride 2) = pixel subsampling (model_irse.py:53): out[n][y][x][:] = x[n][2y][2x][:]
__global__ void subsample2_kernel(const bf16* __restrict__ x, int x_ld, bf16* __restrict__ out, int out_ld, int oh,
                                  int ow, int groups, long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int g = (int)(i % groups);
  long long p = i / groups;
  const int ox = (int)(p % ow);
  long long q = p / ow;
  const int oy = (int)(q % oh);
  const long long n = q / oh;
  const long long src = ((n * (2 * oh) + 2 * oy) * (2LL * ow) + 2 * ox) * x_ld + g * 8;
  *reinterpret_cast<uint4*>(out + p * out_ld + g * 8) = *reinterpret_cast<const uint4*>(x + src);
}

// stats[c] = (mean 0, rstd 1): turns the fused normalise kernel into a plain PReLU pass
__global__ void identity_stats_kernel(float* __restrict__ stats, int c) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < c) {
    stats[2 * i] = 0.f;
    stats[2 * i + 1] = 1.f;
  }
}

// s[c] = gamma[c] * rstd[c]: the scale of an eval-mode BatchNorm (stats [c][2] = (mean, rstd))
__global__ void bn_scale_kernel(const float* __restrict__ stats, const float* __restrict__ gamma, int c,
                                float* __restrict__ s) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < c) s[i] = gamma[i] * stats[2 * i + 1];
}

// 8 consecutive fp32 values (32-byte aligned) as two 16-byte loads
__device__ __forceinline__ void load8f(const float* __restrict__ p, float* v) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// Element-wise input-gradient pass of the IR_50 backward (eval-mode BatchNorm and / or PReLU, plus a second gradient):
//   out[p][c] = s[c] * act'(s[c] * y[p][c] + t[c]) * g[p][c] (+ add)
// with s = gamma * rstd, t = beta - mean * s computed as the forward's normalise kernel does (no stats: s = 1, t = 0),
// act' = 1 where z > 0 and alpha[c] elsewhere (no alpha: identity; no y: act' = 1, the pass is a plain sum).
// add_mode 1 adds add[p][c]; 2 adds the gradient of a stride-2 pixel subsampling (MaxPool2d(1, 2)), i.e. add at the
// half-resolution pixel for the even pixels and nothing elsewhere - a gather, so no atomics.  With nscale (the SE unit's
// residual branch) the first factor is per (image, channel) instead: v = nscale[n][c] * g + nshift[n][c].  One thread per
// 8 channels of a pixel (16-byte loads and store), fp32 arithmetic, one rounding.  out may alias g (each element is read,
// then written, by the same thread).
__global__ void __launch_bounds__(256)
ir50_bwd_ew_kernel(const bf16* g, int g_ld, const bf16* __restrict__ y, int y_ld, const float* __restrict__ stats,
                   const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ alpha,
                   const bf16* __restrict__ add, int add_ld, int add_mode, bf16* out, int out_ld, int h, int w, int groups,
                   long long total, const float* __restrict__ nscale = nullptr, const float* __restrict__ nshift = nullptr) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int cg = (int)(i % groups);
  const long long p = i / groups;
  float v[8];
  unpack8(*reinterpret_cast<const bf16x8*>(g + p * g_ld + cg * 8), v);
  if (nscale) {
    const long long nc = (p / ((long long)h * w)) * groups * 8 + cg * 8;
    float a[8], b[8];
    load8f(nscale + nc, a);
    load8f(nshift + nc, b);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = fmaf(a[j], v[j], b[j]);
  }
  if (y) {
    float f[8];
    unpack8(*reinterpret_cast<const bf16x8*>(y + p * y_ld + cg * 8), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int ch = cg * 8 + j;
      float sc = 1.f, sh = 0.f;
      if (stats) {
        sc = gamma[ch] * stats[2 * ch + 1];
        sh = beta[ch] - stats[2 * ch] * sc;
      }
      const float z = fmaf(f[j], sc, sh);
      v[j] *= (alpha && !(z > 0.f)) ? sc * alpha[ch] : sc;
    }
  }
  if (add_mode == 1) {
    float a[8];
    unpack8(*reinterpret_cast<const bf16x8*>(add + p * add_ld + cg * 8), a);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] += a[j];
  } else if (add_mode == 2) {
    const int x = (int)(p % w);
    const long long q = p / w;
    const int yy = (int)(q % h);
    const long long n = q / h;
    if (((x | yy) & 1) == 0) {
      const long long ps = (n * (h / 2) + yy / 2) * (w / 2) + x / 2;
      float a[8];
      unpack8(*reinterpret_cast<const bf16x8*>(add + ps * add_ld + cg * 8), a);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] += a[j];
    }
  }
  *reinterpret_cast<bf16x8*>(out + p * out_ld + cg * 8) = pack8(v);
}

// ---- squeeze-excitation unit (SEModule(depth, 16), model_irse.py: x * sigmoid(fc2(relu(fc1(mean_hw(x)))))) ----
// The SE input is r = s * y + t, res_layer.4's eval-mode BatchNorm of the res_layer.3 output y (s = gamma * rstd,
// t = beta - mean * s), so its squeeze is s * mean_hw(y) + t: it comes from the InstanceNorm statistics of the stored y.

// pooled[c] = s_c * mean_hw(y)[n][c] + t_c into shared memory, then the hidden pre-activation pre[j] = W1[j][:] . pooled
// (one warp per hidden unit, lanes over channels, shuffle reduction: a fixed order, shared by the forward and backward
// so both see the same ReLU mask)
__device__ __forceinline__ void se_hidden(const float* __restrict__ sq, const float* __restrict__ bnst,
                                          const float* __restrict__ gamma, const float* __restrict__ beta,
                                          const float* __restrict__ w1, int n, int C, int Hd, float* pooled, float* pre) {
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float s = gamma[c] * bnst[2 * c + 1];
    pooled[c] = fmaf(sq[2 * ((long long)n * C + c)], s, beta[c] - bnst[2 * c] * s);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  for (int j = warp; j < Hd; j += nwarps) {
    float acc = 0.f;
    for (int c = lane; c < C; c += 32) acc = fmaf(w1[(long long)j * C + c], pooled[c], acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) pre[j] = acc;
  }
  __syncthreads();
}

// Excitation, one CTA per image: e[n][c] = sigmoid(W2[c][:] . relu(pre)), fp32 (W1 [Hd][C], W2 [C][Hd]: the reference's
// [out][in][1][1] layouts); also the unit output's per-(image, channel) affine map e * BN_4: ea = e * s_c, eb = e * t_c
__global__ void __launch_bounds__(256)
se_excite_kernel(const float* __restrict__ sq, const float* __restrict__ bnst, const float* __restrict__ gamma,
                 const float* __restrict__ beta, const float* __restrict__ w1, const float* __restrict__ w2, int C, int Hd,
                 float* __restrict__ e, float* __restrict__ ea, float* __restrict__ eb) {
  __shared__ float pooled[512], pre[32];
  const int n = blockIdx.x;
  se_hidden(sq, bnst, gamma, beta, w1, n, C, Hd, pooled, pre);
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float acc = 0.f;
    for (int j = 0; j < Hd; ++j) acc = fmaf(w2[(long long)c * Hd + j], fmaxf(pre[j], 0.f), acc);
    const float ex = 1.f / (1.f + expf(-acc)), s = gamma[c] * bnst[2 * c + 1];
    e[(long long)n * C + c] = ex;
    ea[(long long)n * C + c] = ex * s;
    eb[(long long)n * C + c] = ex * (beta[c] - bnst[2 * c] * s);
  }
}

// Unit output with SE: out = res + ea[n][c] * y + eb[n][c] (= res + e * (s_c * y + t_c)), fp32, one rounding (replaces the
// BatchNorm + residual pass; same traffic).  One thread per 8 channels of a pixel, 16-byte loads throughout.
__global__ void __launch_bounds__(256)
se_apply_kernel(const bf16* __restrict__ y, int y_ld, const float* __restrict__ ea, const float* __restrict__ eb,
                const bf16* __restrict__ res, int res_ld, bf16* __restrict__ out, int out_ld, int hw, int groups,
                long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int cg = (int)(i % groups);
  const long long p = i / groups;
  const long long nc = (p / hw) * groups * 8 + cg * 8;
  float f[8], r[8], a[8], b[8];
  unpack8(*reinterpret_cast<const bf16x8*>(y + p * y_ld + cg * 8), f);
  unpack8(*reinterpret_cast<const bf16x8*>(res + p * res_ld + cg * 8), r);
  load8f(ea + nc, a);
  load8f(eb + nc, b);
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] += fmaf(a[j], f[j], b[j]);
  *reinterpret_cast<bf16x8*>(out + p * out_ld + cg * 8) = pack8(r);
}

// Pixel chunks of the SE backward reduction: a function of the image size only, so that the order of the fp32 sums (and
// the bits) do not depend on the batch
__host__ __device__ inline int se_chunks(int hw) { return (hw + 255) / 256; }

// First pass of the SE backward: per (image, pixel chunk) the sums (sum g * y, sum g) over the chunk's pixels of every
// channel -> part[n][chunk][2][C].  Thread = (channel group of 8, pixel lane); the lanes are combined in shared memory in
// a fixed order (no atomics).
__global__ void __launch_bounds__(256)
se_bwd_reduce_kernel(const bf16* __restrict__ g, int g_ld, const bf16* __restrict__ y, int y_ld, int hw, int C,
                     float* __restrict__ part) {
  __shared__ float red[2 * 2048];
  const int n = blockIdx.y, chunk = blockIdx.x, chunks = gridDim.x;
  const int groups = C / 8, lanes = blockDim.x / groups;
  const int cg = threadIdx.x % groups, lane = threadIdx.x / groups;
  const int p0 = (int)((long long)hw * chunk / chunks), p1 = (int)((long long)hw * (chunk + 1) / chunks);
  float sgy[8], sg[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) sgy[j] = sg[j] = 0.f;
  if (lane < lanes) {
    for (int p = p0 + lane; p < p1; p += lanes) {
      const long long pix = (long long)n * hw + p;
      float a[8], b[8];
      unpack8(*reinterpret_cast<const bf16x8*>(g + pix * g_ld + cg * 8), a);
      unpack8(*reinterpret_cast<const bf16x8*>(y + pix * y_ld + cg * 8), b);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        sgy[j] = fmaf(a[j], b[j], sgy[j]);
        sg[j] += a[j];
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      red[(lane * 2 + 0) * C + cg * 8 + j] = sgy[j];
      red[(lane * 2 + 1) * C + cg * 8 + j] = sg[j];
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < 2 * C; k += blockDim.x) {
    const int which = k / C, c = k - which * C;
    float acc = 0.f;
    for (int l = 0; l < lanes; ++l) acc += red[(l * 2 + which) * C + c];
    part[(((long long)n * chunks + chunk) * 2 + which) * C + c] = acc;
  }
}

// Tail of the SE backward, one CTA per image: de[c] = s_c * sum(g*y) + t_c * sum(g) (= sum_hw g * r), u = de * e (1 - e),
// dh = W2^T u masked by relu', dpool = W1^T dh; shift[n][c] = dpool[c] / hw, the part of dr that every pixel shares
// (dr = e * g + shift, see ir50_bwd_ew_kernel).
__global__ void __launch_bounds__(256)
se_bwd_tail_kernel(const float* __restrict__ part, int chunks, const float* __restrict__ sq, const float* __restrict__ bnst,
                   const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ w1,
                   const float* __restrict__ w2, const float* __restrict__ e, int C, int Hd, int hw,
                   float* __restrict__ shift) {
  __shared__ float pooled[512], u[512], pre[32], dh[32];
  const int n = blockIdx.x;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float sgy = 0.f, sg = 0.f;
    for (int k = 0; k < chunks; ++k) {
      sgy += part[(((long long)n * chunks + k) * 2 + 0) * C + c];
      sg += part[(((long long)n * chunks + k) * 2 + 1) * C + c];
    }
    const float s = gamma[c] * bnst[2 * c + 1];
    const float de = fmaf(s, sgy, (beta[c] - bnst[2 * c] * s) * sg);
    const float ec = e[(long long)n * C + c];
    u[c] = de * ec * (1.f - ec);
  }
  se_hidden(sq, bnst, gamma, beta, w1, n, C, Hd, pooled, pre);   // (its first __syncthreads also publishes u)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  for (int j = warp; j < Hd; j += nwarps) {
    float acc = 0.f;
    for (int c = lane; c < C; c += 32) acc = fmaf(w2[(long long)c * Hd + j], u[c], acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) dh[j] = pre[j] > 0.f ? acc : 0.f;
  }
  __syncthreads();
  const float inv = 1.f / (float)hw;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float acc = 0.f;
    for (int j = 0; j < Hd; ++j) acc = fmaf(w1[(long long)j * C + c], dh[j], acc);
    shift[(long long)n * C + c] = acc * inv;
  }
}

// tape indices of one bottleneck_IR / bottleneck_IR_SE unit of the IR program (-1: absent); bn4 is the SE apply op
// (OP_SE) in an SE unit
struct IrUnit {
  int sc_conv = -1, sc_bn = -1, sub = -1, bn0, conv1, prelu, conv2, bn4;
  int fc1 = -1;   // SE units: parameter index of res_layer.5.fc1 (fc2 follows)
};

struct Net {
  int engine;
  const float* const* params;
  float* const* grads;
  void* const* buffers;
  const crfr_resnet_io* io;
  cudaStream_t st;
  uint8_t* ws;
  size_t ws_bytes, off = 0;
  bool exec;
  int err = CRFR_OK;
  std::vector<Op> tape;
  std::vector<std::vector<Slot>> slots;
  void* scratch = nullptr;
  size_t scratch_bytes = 0;
  Tensor feat[4], emb;
  // weight packing: a dry run of the program (exec = false) collects every pack job here, the entry point issues them as
  // one batch, and the real run (packs_done) only re-derives the same arena offsets (as in fsrnet.cu)
  std::vector<crfr_pack_job>* collect = nullptr;
  bool packs_done = false;
  bf16* wp = nullptr;    // packed linear weights (forward)
  bf16* wpt = nullptr;   // transposed (backward)
  int pcur = 0, bncur = 0;
  std::vector<IrUnit> ir_units;               // IR program: the units, and the stem / head ops, as tape indices
  int ir_stem_conv = -1, ir_stem_bn = -1, ir_head_bn0 = -1, ir_head_lin = -1, ir_head_bn1 = -1;
  int ir_layers = 50, ir_se = 0;              // IR program variant: 50 / 100 / 152 layers, bottleneck_IR(_SE)
  std::vector<crfr_tape_entry>* grad_tape = nullptr;   // set: backward_ir lists its stored gradients here (kinds 11-16)

  void* alloc(size_t bytes) {
    size_t a = (off + 1023) & ~(size_t)1023;
    if (a + bytes > ws_bytes) {
      if (err == CRFR_OK) {
        crfr_set_error("resnet34: workspace too small (%zu needed so far, %zu given)", a + bytes, ws_bytes);
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
  void check_cuda(cudaError_t e) {
    if (e != cudaSuccess && err == CRFR_OK) {
      crfr_set_error("resnet34: %s", cudaGetErrorString(e));
      err = CRFR_ECUDA;
    }
  }
  Tensor new_tensor(int n, int h, int w, int c) {
    Tensor t;
    t.n = n; t.h = h; t.w = w; t.c = c; t.ld = c < 8 ? 4 : c;
    t.p = (bf16*)alloc((size_t)n * h * w * t.ld * sizeof(bf16));
    t.id = (int)slots.size();
    slots.emplace_back();
    return t;
  }
  float* grad(int idx) { return (grads && idx >= 0) ? grads[idx] : nullptr; }

  // ---- forward ops ----
  // inst_stats: also the per-(image, channel) (mean, rstd) [n][cout][2] of the stored output (the SE unit's squeeze)
  Tensor conv(const Tensor& x, int w_idx, int cout, int k, int stride, int pad, bool x_needs_grad,
              float* inst_stats = nullptr) {
    Op op;
    op.kind = OP_CONV;
    crfr_conv_desc& d = op.cd;
    d.n = x.n; d.h = x.h; d.w = x.w; d.cin = x.c; d.cout = cout; d.k = k; d.stride = stride; d.pad = pad;
    d.transposed = 0;
    d.oh = (x.h + 2 * pad - k) / stride + 1;
    d.ow = (x.w + 2 * pad - k) / stride + 1;
    Tensor y = new_tensor(x.n, d.oh, d.ow, cout);
    d.in_ld = x.ld; d.out_ld = y.ld;
    op.cin_pad = x.c < 8 ? 4 : x.c;
    const int T = k * k;
    void* wpk = alloc((size_t)T * cout * op.cin_pad * sizeof(bf16));
    if (collect && ok()) collect->push_back({params[w_idx], wpk, T, cout, x.c, op.cin_pad, (long long)x.c * T, T, 0, 0});
    // every convolution of this network feeds a BatchNorm: in training its batch statistics come out of the epilogue
    float* bn_stats = io->training ? (float*)alloc((size_t)cout * 2 * sizeof(float)) : nullptr;
    y.bn_stats = bn_stats;
    if (run()) {
      if (!packs_done) check(crfr_pack_weight(params[w_idx], wpk, T, cout, x.c, op.cin_pad, (long long)x.c * T, T, 1, st));
      if (bn_stats)
        check(crfr_conv_fwd_bnstats(engine, &d, x.p, wpk, op.cin_pad, y.p, bn_stats, io->eps, scratch, scratch_bytes, st));
      else
        check(crfr_conv_fwd(engine, &d, x.p, wpk, op.cin_pad, nullptr, y.p, nullptr, inst_stats, io->eps, scratch,
                            scratch_bytes, st));
    }
    op.a = x; op.out = y; op.w_idx = w_idx; op.x_needs_grad = x_needs_grad;
    tape.push_back(op);
    return y;
  }

  // BatchNorm (batch statistics over n*h*w in training, running statistics otherwise) + optional residual + ReLU
  Tensor bn(const Tensor& y, int g_idx, int relu, const Tensor* res, int alpha_idx = -1, int bn_index = -1) {
    const int bi = bn_index >= 0 ? bn_index : bncur++;
    const long long count = (long long)y.n * y.h * y.w;
    Tensor out = new_tensor(y.n, y.h, y.w, y.c);
    const bool have_stats = io->training && y.bn_stats;   // computed by the producing convolution's epilogue
    float* stats = have_stats ? y.bn_stats : (float*)alloc((size_t)y.c * 2 * sizeof(float));
    float* rmean = buffers ? (float*)buffers[3 * bi] : nullptr;
    float* rvar = buffers ? (float*)buffers[3 * bi + 1] : nullptr;
    long long* nbt = buffers ? (long long*)buffers[3 * bi + 2] : nullptr;
    if (run()) {
      if (io->training) {
        if (!have_stats) check(crfr_norm_stats(y.p, 1, (int)count, y.c, y.ld, io->eps, stats, scratch, scratch_bytes, st));
        if (rmean && rvar)
          check(crfr_bn_update_running(stats, rmean, rvar, nbt, y.c, count, io->momentum, io->eps, st));
      } else {
        check(crfr_bn_running_to_stats(rmean, rvar, y.c, io->eps, stats, st));
      }
      check(crfr_norm_act_fwd(y.p, y.ld, stats, params[g_idx], params[g_idx + 1],
                              alpha_idx >= 0 ? params[alpha_idx] : nullptr, relu, res ? res->p : nullptr,
                              res ? res->ld : 8, out.p, out.ld, 1, (int)count, y.c, st));
    }
    Op op;
    op.kind = OP_BN;
    op.a = y; op.out = out; op.stats = stats; op.g_idx = g_idx; op.beta_idx = g_idx + 1; op.alpha_idx = alpha_idx;
    op.relu = relu != 0;
    op.has_res = res != nullptr;
    if (res) op.b = *res;
    tape.push_back(op);
    return out;
  }

  Tensor block(const Tensor& x, int planes, int stride, bool down) {   // BasicBlock, model/resnet.py:18-47
    const int p0 = pcur;
    pcur += down ? 9 : 6;
    Tensor y1 = conv(x, p0 + 0, planes, 3, stride, 1, true);
    Tensor a1 = bn(y1, p0 + 1, 1, nullptr);
    Tensor y2 = conv(a1, p0 + 3, planes, 3, 1, 1, true);
    // module order of the BatchNorms is bn1, bn2, downsample.1: reserve bn2's slot before the downsample branch
    const int bn2 = bncur++;
    Tensor res = x;
    if (down) {
      Tensor yd = conv(x, p0 + 6, planes, 1, stride, 0, true);
      res = bn(yd, p0 + 7, 0, nullptr);
    }
    const int save = bncur;
    bncur = bn2;
    Tensor out = bn(y2, p0 + 4, 1, &res);
    bncur = save;
    return out;
  }

  Tensor linear(const Tensor& a, int w_index = -1) {
    const int B = a.n, K = a.h * a.w * a.c;
    Tensor y = new_tensor(B, 1, 1, kEmb);
    wp = (bf16*)alloc((size_t)kEmb * K * sizeof(bf16));
    wpt = io->training ? (bf16*)alloc((size_t)kEmb * K * sizeof(bf16)) : nullptr;
    const int w_idx = w_index >= 0 ? w_index : pcur;
    if (w_index < 0) pcur += 2;
    if (run()) {
      const long long total = (long long)kEmb * K;
      linear_pack_kernel<<<crfr_cdiv(total, 256), 256, 0, st>>>(params[w_idx], wp, wpt, kEmb, a.c, a.h * a.w);
      CRFR_COUNT_LAUNCH();
      check_cuda(cudaGetLastError());
      TcGemm g{a.p, B, 1, 1, K, K, wp, 1, 0, 1, kEmb, 64, y.p, kEmb, 0, params[w_idx + 1]};
      check(crfr_tc_gemm(g, st));
    }
    Op op;
    op.kind = OP_LINEAR;
    op.a = a; op.out = y; op.w_idx = w_idx; op.b_idx = w_idx + 1;
    tape.push_back(op);
    return y;
  }

  void to_nchw(const Tensor& t, float* dst) {
    if (dst && run()) check(crfr_nhwc_bf16_to_nchw_f32(t.p, dst, t.n, t.c, t.h, t.w, t.ld, st));
  }

  size_t scratch_need(int B, int S) const {
    size_t m = crfr_norm_ws_bytes(1, B * (S / 2) * (S / 2), 64);
    const int q = S / 2;
    const crfr_conv_desc shapes[] = {
        {B, S, S, 3, 64, 7, 2, 3, q, q, 4, 64, 0},
        {B, q, q, 64, 64, 3, 1, 1, q, q, 64, 64, 0},
        {B, q, q, 64, 128, 3, 2, 1, q / 2, q / 2, 64, 128, 0},
        {B, q / 2, q / 2, 128, 128, 3, 1, 1, q / 2, q / 2, 128, 128, 0},
        {B, q / 2, q / 2, 128, 256, 3, 2, 1, q / 4, q / 4, 128, 256, 0},
        {B, q / 4, q / 4, 256, 256, 3, 1, 1, q / 4, q / 4, 256, 256, 0},
        {B, q / 4, q / 4, 256, 512, 3, 2, 1, q / 8, q / 8, 256, 512, 0},
        {B, q / 8, q / 8, 512, 512, 3, 1, 1, q / 8, q / 8, 512, 512, 0}};
    for (const crfr_conv_desc& d : shapes) {
      const size_t b = crfr_conv_workspace_bytes(&d);
      if (b > m) m = b;
    }
    const size_t lin = sizeof(float) * (size_t)kEmb * kFeat * (q / 8) * (q / 8) + 4096;   // linear wgrad accumulator
    return (m > lin ? m : lin) + 4096;
  }

  void forward() {
    const int B = io->batch, S = io->size;
    pcur = 0; bncur = 0;
    scratch_bytes = scratch_need(B, S);
    scratch = alloc(scratch_bytes);
    Tensor x4 = new_tensor(B, S, S, 3);
    if (run()) check(crfr_nchw_f32_to_nhwc_bf16(io->x, x4.p, B, 3, S, S, 4, 4, st));
    // stem (model/resnet.py:208-211; the max-pool is commented out in the reference)
    Tensor y = conv(x4, 0, 64, 7, 2, 3, false);
    pcur = 1;
    Tensor a = bn(y, 1, 1, nullptr);
    pcur = 3;
    const int layers[4] = {3, 4, 6, 3}, planes[4] = {64, 128, 256, 512};
    for (int l = 0; l < 4; ++l) {
      for (int b = 0; b < layers[l]; ++b) a = block(a, planes[l], (l > 0 && b == 0) ? 2 : 1, l > 0 && b == 0);
      feat[l] = a;
      to_nchw(a, io->feat[l]);
    }
    Tensor o1 = bn(a, pcur, 0, nullptr);      // bn_o1
    pcur += 2;
    Tensor yfc = linear(o1);                  // fc (pcur += 2 inside)
    emb = bn(yfc, pcur, 0, nullptr);          // bn_o2 (BatchNorm1d)
    pcur += 2;
    to_nchw(emb, io->emb);
  }

  // ---- IR_50 (eval-mode BatchNorm) ----
  int last() const { return (int)tape.size() - 1; }
  Tensor prelu(const Tensor& y, int alpha_idx, float* ident) {   // plain PReLU pass
    Tensor out = new_tensor(y.n, y.h, y.w, y.c);
    if (run())
      check(crfr_norm_act_fwd(y.p, y.ld, ident, nullptr, nullptr, params[alpha_idx], 0, nullptr, 8, out.p, out.ld, 1,
                              y.n * y.h * y.w, y.c, st));
    Op op;
    op.kind = OP_PRELU;
    op.a = y; op.out = out; op.alpha_idx = alpha_idx;
    tape.push_back(op);
    return out;
  }
  Tensor subsample2(const Tensor& x) {
    Tensor out = new_tensor(x.n, x.h / 2, x.w / 2, x.c);
    if (run()) {
      const long long total = (long long)out.n * out.h * out.w * (x.c / 8);
      subsample2_kernel<<<crfr_cdiv(total, 256), 256, 0, st>>>(x.p, x.ld, out.p, out.ld, out.h, out.w, x.c / 8, total);
      CRFR_COUNT_LAUNCH();
      check_cuda(cudaGetLastError());
    }
    Op op;
    op.kind = OP_SUB2;
    op.a = x; op.out = out;
    tape.push_back(op);
    return out;
  }
  // res_layer.4 (eval-mode BatchNorm, parameters g_idx, g_idx + 1) + res_layer.5 (SEModule, fc1 / fc2 at fc1_idx,
  // fc1_idx + 1) + the shortcut res; sq: the squeeze statistics of y from its convolution
  Tensor se_unit_out(const Tensor& y, int g_idx, int bn_index, int fc1_idx, const Tensor& res, float* sq) {
    Tensor out = new_tensor(y.n, y.h, y.w, y.c);
    float* stats = (float*)alloc((size_t)y.c * 2 * sizeof(float));
    float* e = (float*)alloc((size_t)y.n * y.c * sizeof(float));
    float* ea = (float*)alloc((size_t)y.n * y.c * sizeof(float));
    float* eb = (float*)alloc((size_t)y.n * y.c * sizeof(float));
    if (run()) {
      check(crfr_bn_running_to_stats((const float*)buffers[3 * bn_index], (const float*)buffers[3 * bn_index + 1], y.c,
                                     io->eps, stats, st));
      se_excite_kernel<<<y.n, 256, 0, st>>>(sq, stats, params[g_idx], params[g_idx + 1], params[fc1_idx],
                                            params[fc1_idx + 1], y.c, y.c / kSeReduction, e, ea, eb);
      CRFR_COUNT_LAUNCH();
      check_cuda(cudaGetLastError());
      const long long total = (long long)y.n * y.h * y.w * (y.c / 8);
      se_apply_kernel<<<crfr_cdiv(total, 256), 256, 0, st>>>(y.p, y.ld, ea, eb, res.p, res.ld, out.p, out.ld, y.h * y.w,
                                                             y.c / 8, total);
      CRFR_COUNT_LAUNCH();
      check_cuda(cudaGetLastError());
    }
    Op op;
    op.kind = OP_SE;
    op.a = y; op.b = res; op.out = out; op.has_res = true;
    op.stats = e; op.bn_stats = stats; op.squeeze = sq;
    op.g_idx = g_idx; op.beta_idx = g_idx + 1; op.w_idx = fc1_idx;
    tape.push_back(op);
    return out;
  }

  // parameter order (named_parameters): input_layer (4), output_layer (6), body blocks (7, or 10 with a conv shortcut,
  // + 2 with SE: res_layer.5.fc1 / fc2); BatchNorm order (named_buffers): input_layer.1, output_layer.0, output_layer.4,
  // then per block [shortcut_layer.1], res_layer.0, res_layer.4.  The variant is (ir_layers, ir_se); IR_50 is (50, 0).
  void forward_ir() {
    const int B = io->batch, S = io->size;
    scratch_bytes = scratch_need_ir50(B, S);
    if (ir_se) {   // the squeeze statistics of res_layer.3 may take a separate per-image pass (crfr_norm_stats)
      const int q = S / 2;
      const crfr_conv_desc shapes[] = {
          {B, S, S, 64, 64, 3, 2, 1, q, q, 64, 64, 0},
          {B, q, q, 64, 64, 3, 1, 1, q, q, 64, 64, 0},
          {B, q, q, 128, 128, 3, 2, 1, q / 2, q / 2, 128, 128, 0},
          {B, q / 2, q / 2, 128, 128, 3, 1, 1, q / 2, q / 2, 128, 128, 0},
          {B, q / 2, q / 2, 256, 256, 3, 2, 1, q / 4, q / 4, 256, 256, 0},
          {B, q / 4, q / 4, 256, 256, 3, 1, 1, q / 4, q / 4, 256, 256, 0},
          {B, q / 4, q / 4, 512, 512, 3, 2, 1, q / 8, q / 8, 512, 512, 0}};
      for (const crfr_conv_desc& d : shapes) {
        const size_t b = crfr_conv_workspace_bytes(&d) + 4096;
        if (b > scratch_bytes) scratch_bytes = b;
      }
    }
    scratch = alloc(scratch_bytes);
    float* ident = (float*)alloc(512 * 2 * sizeof(float));
    if (run()) {
      identity_stats_kernel<<<4, 128, 0, st>>>(ident, 512);
      CRFR_COUNT_LAUNCH();
    }
    Tensor x4 = new_tensor(B, S, S, 3);
    if (run()) check(crfr_nchw_f32_to_nhwc_bf16(io->x, x4.p, B, 3, S, S, 4, 4, st));
    Tensor a = bn(conv(x4, 0, 64, 3, 1, 1, false), 1, 0, nullptr, 3, 0);     // input_layer: conv, BN, PReLU
    ir_stem_conv = last() - 1; ir_stem_bn = last();
    ir_units.clear();
    int p = 10, bi = 3;
    int units[4];
    ir_units_of(ir_layers, units);
    const int depth[4] = {64, 128, 256, 512};
    int in_ch = 64;
    for (int l = 0; l < 4; ++l)
      for (int u = 0; u < units[l]; ++u) {   // bottleneck_IR(_SE), model_irse.py:49-66
        const int stride = u == 0 ? 2 : 1, d = depth[l];
        const bool conv_sc = in_ch != d;
        IrUnit un;
        Tensor sc = a;
        if (conv_sc) {
          sc = bn(conv(a, p, d, 1, stride, 0, false), p + 1, 0, nullptr, -1, bi);
          un.sc_conv = last() - 1; un.sc_bn = last();
          p += 3; bi += 1;
        } else if (stride == 2) {
          sc = subsample2(a);
          un.sub = last();
        }
        Tensor r = bn(a, p, 0, nullptr, -1, bi);                       // res_layer.0
        un.bn0 = last();
        r = prelu(conv(r, p + 2, d, 3, 1, 1, false), p + 3, ident);    // res_layer.1, .2
        un.conv1 = last() - 1; un.prelu = last();
        float* sq = ir_se ? (float*)alloc((size_t)B * d * 2 * sizeof(float)) : nullptr;
        r = conv(r, p + 4, d, 3, stride, 1, false, sq);                // res_layer.3 (+ the SE squeeze)
        un.conv2 = last();
        if (ir_se) {
          a = se_unit_out(r, p + 5, bi + 1, p + 7, sc, sq);            // res_layer.4 + .5 (SE) + shortcut
          un.fc1 = p + 7;
        } else {
          a = bn(r, p + 5, 0, &sc, -1, bi + 1);                        // res_layer.4 + shortcut
        }
        un.bn4 = last();
        ir_units.push_back(un);
        p += ir_se ? 9 : 7; bi += 2;
        in_ch = d;
        if (u == units[l] - 1) {   // stage output: 64@56^2, 128@28^2, 256@14^2, 512@7^2 - the shapes of ResNet_34's x1..x4,
          feat[l] = a;             // i.e. the t_k of the residual-KD loss when IR is the teacher (distill_main.py:59,68-69)
          to_nchw(a, io->feat[l]);
        }
      }
    Tensor o = bn(a, 4, 0, nullptr, -1, 1);                            // output_layer.0 (Dropout: identity in eval)
    ir_head_bn0 = last();
    Tensor y = linear(o, 6);                                           // output_layer.3
    ir_head_lin = last();
    emb = bn(y, 8, 0, nullptr, -1, 2);                                 // output_layer.4 (BatchNorm1d)
    ir_head_bn1 = last();
    to_nchw(emb, io->emb);
  }

  size_t scratch_need_ir50(int B, int S) const {
    size_t m = crfr_norm_ws_bytes(1, B * S * S, 64);
    const int q = S / 2;
    const crfr_conv_desc shapes[] = {
        {B, S, S, 3, 64, 3, 1, 1, S, S, 4, 64, 0},
        {B, S, S, 64, 64, 3, 2, 1, q, q, 64, 64, 0},
        {B, q, q, 64, 128, 3, 2, 1, q / 2, q / 2, 64, 128, 0},
        {B, q, q, 64, 128, 1, 2, 0, q / 2, q / 2, 64, 128, 0},
        {B, q / 2, q / 2, 128, 256, 3, 2, 1, q / 4, q / 4, 128, 256, 0},
        {B, q / 4, q / 4, 256, 512, 3, 2, 1, q / 8, q / 8, 256, 512, 0},
        {B, q / 8, q / 8, 512, 512, 3, 1, 1, q / 8, q / 8, 512, 512, 0}};
    for (const crfr_conv_desc& d : shapes) {
      const size_t b = crfr_conv_workspace_bytes(&d);
      if (b > m) m = b;
    }
    return m + 4096;
  }

  // ---- IR input gradient (after a forward_ir over the same arena; parameters stay frozen) ----
  Tensor map_like(const Tensor& t) { return Tensor{(bf16*)alloc((size_t)t.n * t.h * t.w * t.ld * sizeof(bf16)), t.n, t.h, t.w, t.c, t.ld}; }
  float* bn_scale(const Op& b) {
    float* s = (float*)alloc((size_t)b.a.c * sizeof(float));
    if (run()) {
      bn_scale_kernel<<<crfr_cdiv(b.a.c, 128), 128, 0, st>>>(b.kind == OP_SE ? b.bn_stats : b.stats, params[b.g_idx],
                                                             b.a.c, s);
      CRFR_COUNT_LAUNCH();
      check_cuda(cudaGetLastError());
    }
    return s;
  }
  // transposed pack [tap][cin][cout] of a convolution, with the optional folded scales (rscale: cin, sscale: cout)
  bf16* dgrad_pack(const Op& cv, const float* rscale, const float* sscale, std::vector<crfr_pack_job>& jobs) {
    const crfr_conv_desc& d = cv.cd;
    const int T = d.k * d.k;
    bf16* wt = (bf16*)alloc((size_t)T * d.cin * d.cout * sizeof(bf16));
    crfr_pack_job j{params ? params[cv.w_idx] : nullptr, wt, T, d.cin, d.cout, d.cout, T, (long long)d.cin * T, 0, 0, rscale, sscale};
    jobs.push_back(j);
    return wt;
  }
  void dgrad(const Op& cv, const Slot& dy, const bf16* wt, const Tensor& dx, bool stem = false) {
    crfr_conv_desc d = cv.cd;
    d.out_ld = dy.ld;
    d.in_ld = dx.ld;
    if (!run()) return;
    if (stem && engine != CRFR_ENGINE_DIRECT && crfr_lowered_recipe(&d) == 1 && d.cout == 64 && d.h % 8 == 0)
      check(crfr_lowered_dgrad_cin3(&d, dy.p, wt, dx.p, scratch, scratch_bytes, st));
    else
      check(crfr_conv_dgrad(engine, &d, dy.p, wt, d.cout, dx.p, scratch, scratch_bytes, st));
  }
  // out = s * act'(z) * g (+ add): see ir50_bwd_ew_kernel; bn (may be null) supplies stats / gamma / beta; nscale /
  // nshift: per-(image, channel) factor and shift instead (the SE unit)
  void ew(const Slot& g, const Tensor& y, const Op* bn, int alpha_idx, const Slot* add, int add_mode, const Tensor& out,
          const float* nscale = nullptr, const float* nshift = nullptr) {
    if (!run()) return;
    const float* alpha = alpha_idx >= 0 ? params[alpha_idx] : nullptr;
    const long long total = (long long)out.n * out.h * out.w * (out.c / 8);
    ir50_bwd_ew_kernel<<<crfr_cdiv(total, 256), 256, 0, st>>>(
        g.p, g.ld, y.p, y.ld, bn ? bn->stats : nullptr, bn ? params[bn->g_idx] : nullptr,
        bn ? params[bn->beta_idx] : nullptr, alpha, add ? add->p : nullptr, add ? add->ld : 8, add_mode, out.p, out.ld,
        out.h, out.w, out.c / 8, total, nscale, nshift);
    CRFR_COUNT_LAUNCH();
    check_cuda(cudaGetLastError());
  }

  // one entry of the gradient tape (crfr_irnet_grad_tape): the bf16 gradient at p (pixel stride ld) with respect to the
  // stored forward tensor `of`, and an optional fp32 side result; offsets are bytes from the workspace base
  void record_grad(int kind, int unit, const Tensor& of, const bf16* p, int ld, const float* stats = nullptr) {
    if (!grad_tape) return;
    crfr_tape_entry e;
    e.kind = kind;
    e.n = of.n; e.h = of.h; e.w = of.w; e.c = of.c; e.ld = ld;
    e.out_off = (long long)((const uint8_t*)p - ws);
    e.in_off = (long long)((const uint8_t*)of.p - ws);
    e.stats_off = stats ? (long long)((const uint8_t*)stats - ws) : -1;
    e.w_idx = unit;
    e.has_res = 0;
    grad_tape->push_back(e);
  }

  // SE unit: the gradient dr at the SE input r from the unit's output gradient g (dr = e * g + W1^T dh / hw, see
  // se_bwd_tail_kernel) - a deterministic per-(image, channel) reduction, the tiny per-image tail, one element-wise pass
  Tensor se_grad(const Op& se, const Slot& g, int unit) {
    const Tensor& y = se.a;
    const int hw = y.h * y.w, chunks = se_chunks(hw), hid = y.c / kSeReduction;
    float* part = (float*)alloc((size_t)y.n * chunks * 2 * y.c * sizeof(float));
    float* shift = (float*)alloc((size_t)y.n * y.c * sizeof(float));
    Tensor dr = map_like(y);
    if (run()) {
      se_bwd_reduce_kernel<<<dim3(chunks, y.n), 256, 0, st>>>(g.p, g.ld, y.p, y.ld, hw, y.c, part);
      CRFR_COUNT_LAUNCH();
      check_cuda(cudaGetLastError());
      se_bwd_tail_kernel<<<y.n, 256, 0, st>>>(part, chunks, se.squeeze, se.bn_stats, params[se.g_idx], params[se.beta_idx],
                                              params[se.w_idx], params[se.w_idx + 1], se.stats, y.c, hid, hw, shift);
      CRFR_COUNT_LAUNCH();
      check_cuda(cudaGetLastError());
    }
    ew(g, Tensor{}, nullptr, -1, nullptr, 0, dr, se.stats, shift);
    record_grad(13, unit, y, dr.p, dr.ld, shift);
    return dr;
  }

  // Per unit, from the unit's output gradient g: res_layer.4's scale is folded into res_layer.3's dgrad weights and
  // res_layer.0's into res_layer.1's, the shortcut BatchNorm's into its 1x1 convolution, output_layer.0's and the
  // BatchNorm1d's into the transposed linear weights; what remains element-wise (PReLU masks, the stem's BatchNorm +
  // PReLU, the gradient sum at each unit's input) is ir50_bwd_ew_kernel.  In an SE unit the per-(image, channel)
  // excitation cannot be folded: se_grad turns g into the residual branch's gradient first.
  void backward_ir(const float* d_emb, const float* const* d_feat, float* dx) {
    const int B = io->batch;
    size_t need = crfr_lowered_dgrad_cin3_ws_bytes(&tape[ir_stem_conv].cd);
    for (const Op& op : tape)
      if (op.kind == OP_CONV) {
        const size_t b = crfr_conv_workspace_bytes(&op.cd);
        if (b > need) need = b;
      }
    if (need > scratch_bytes) {   // the forward's scratch is reused where it is large enough
      scratch_bytes = need;
      scratch = alloc(need);
    }
    // folded scales and weight packs, all issued before the walk (one batched pack launch)
    std::vector<crfr_pack_job> jobs;
    std::vector<bf16*> w1(ir_units.size()), w2(ir_units.size()), wsc(ir_units.size(), nullptr);
    for (size_t u = 0; u < ir_units.size(); ++u) {
      const IrUnit& U = ir_units[u];
      w2[u] = dgrad_pack(tape[U.conv2], nullptr, bn_scale(tape[U.bn4]), jobs);
      w1[u] = dgrad_pack(tape[U.conv1], bn_scale(tape[U.bn0]), nullptr, jobs);
      if (U.sc_conv >= 0) wsc[u] = dgrad_pack(tape[U.sc_conv], nullptr, bn_scale(tape[U.sc_bn]), jobs);
    }
    bf16* w0 = dgrad_pack(tape[ir_stem_conv], nullptr, nullptr, jobs);
    const Op& lin = tape[ir_head_lin];
    const Tensor& a4 = tape[ir_head_bn0].a;
    const int K = a4.h * a4.w * a4.c;
    bf16* wlt = nullptr;
    if (d_emb) {
      const float* s_o0 = bn_scale(tape[ir_head_bn0]);
      const float* s_emb = bn_scale(tape[ir_head_bn1]);
      wlt = (bf16*)alloc((size_t)kEmb * K * sizeof(bf16));
      if (run()) {
        const long long total = (long long)kEmb * K;
        linear_pack_kernel<<<crfr_cdiv(total, 256), 256, 0, st>>>(params[lin.w_idx], nullptr, wlt, kEmb, a4.c,
                                                                  a4.h * a4.w, s_emb, s_o0);
        CRFR_COUNT_LAUNCH();
        check_cuda(cudaGetLastError());
      }
    }
    if (run()) check(crfr_pack_weight_batch(jobs.data(), (int)jobs.size(), st));

    // head: d a4 = s_o0 * W^T (s_emb * d_emb)
    if (d_emb) {
      seed_grad(emb, d_emb);
      const Slot de = slots[emb.id][0];
      Tensor da = map_like(a4);
      if (run()) {
        TcGemm g{de.p, B, 1, 1, kEmb, de.ld, wlt, 1, 0, 1, K, 0, da.p, K, 0, nullptr};
        check(crfr_tc_gemm(g, st));
      }
      record_grad(11, -1, a4, da.p, da.ld);
      add_slot(a4, da.p, da.ld);
    }
    for (int l = 0; l < 4; ++l) seed_grad(feat[l], d_feat ? d_feat[l] : nullptr);

    for (int u = (int)ir_units.size() - 1; u >= 0 && ok(); --u) {
      const IrUnit& U = ir_units[u];
      const Op& b4 = tape[U.bn4];
      const Op& pr = tape[U.prelu];
      const Tensor& in = tape[U.bn0].a;
      if (!has_grad(b4.out)) continue;
      squash(b4.out, 1);
      const Slot g = slots[b4.out.id][0];
      record_grad(12, u, b4.out, g.p, g.ld);
      Tensor d_r2 = map_like(pr.out);
      if (U.fc1 >= 0) {
        const Tensor dr = se_grad(b4, g, u);                               // res_layer.5
        dgrad(tape[U.conv2], Slot{dr.p, dr.ld}, w2[u], d_r2);             // res_layer.4 + .3
      } else {
        dgrad(tape[U.conv2], g, w2[u], d_r2);                             // res_layer.4 + .3
      }
      const Slot s_r2{d_r2.p, d_r2.ld};
      ew(s_r2, pr.a, nullptr, pr.alpha_idx, nullptr, 0, d_r2);     // res_layer.2, in place
      record_grad(14, u, pr.a, d_r2.p, d_r2.ld);
      Tensor d_in = map_like(in);
      dgrad(tape[U.conv1], s_r2, w1[u], d_in);                            // res_layer.1 + .0
      const Slot s_in{d_in.p, d_in.ld};
      if (U.sc_conv >= 0) {                                                // conv1x1 + BN shortcut
        Tensor d_sc = map_like(in);
        dgrad(tape[U.sc_conv], g, wsc[u], d_sc);
        const Slot s_sc{d_sc.p, d_sc.ld};
        ew(s_in, Tensor{}, nullptr, -1, &s_sc, 1, d_in);
      } else {                                                             // identity / MaxPool2d(1, 2)
        ew(s_in, Tensor{}, nullptr, -1, &g, U.sub >= 0 ? 2 : 1, d_in);
      }
      record_grad(15, u, in, d_in.p, d_in.ld);
      add_slot(in, d_in.p, d_in.ld);
    }

    // stem: BatchNorm + PReLU, then the dgrad of the 3 -> 64 convolution into the 4-channel input
    const Op& sb = tape[ir_stem_bn];
    const Op& s0 = tape[ir_stem_conv];
    if (!has_grad(sb.out)) {
      if (run()) check_cuda(cudaMemsetAsync(dx, 0, sizeof(float) * (size_t)B * 3 * io->size * io->size, st));
      return;
    }
    squash(sb.out, 1);
    Tensor dy0 = map_like(sb.a);
    ew(slots[sb.out.id][0], sb.a, &sb, sb.alpha_idx, nullptr, 0, dy0);
    record_grad(16, -1, sb.a, dy0.p, dy0.ld);
    Tensor dx4 = map_like(s0.a);
    dgrad(s0, Slot{dy0.p, dy0.ld}, w0, dx4, true);
    if (run()) check(crfr_nhwc_bf16_to_nchw_f32(dx4.p, dx, B, 3, dx4.h, dx4.w, dx4.ld, st));
  }

  // ---- backward ----
  void add_slot(const Tensor& t, bf16* p, int ld) { slots[t.id].push_back({p, ld}); }
  bool has_grad(const Tensor& t) const { return t.id >= 0 && !slots[t.id].empty(); }
  void squash(const Tensor& t, size_t max_slots) {
    std::vector<Slot>& s = slots[t.id];
    while (s.size() > max_slots) {
      const bool three = s.size() >= 3;
      bf16* out = (bf16*)alloc((size_t)t.n * t.h * t.w * t.ld * sizeof(bf16));
      const size_t k = s.size();
      Slot a = s[k - 1], b = s[k - 2], c = three ? s[k - 3] : Slot{nullptr, t.ld};
      if (run()) check(crfr_add_n(a.p, a.ld, b.p, b.ld, c.p, c.ld, out, t.ld, (long long)t.n * t.h * t.w, t.ld, st));
      s.resize(k - (three ? 3 : 2));
      s.push_back({out, t.ld});
    }
  }
  void seed_grad(const Tensor& t, const float* g) {   // external gradient of an output (fp32 NCHW)
    if (!g) return;
    bf16* d = (bf16*)alloc((size_t)t.n * t.h * t.w * t.ld * sizeof(bf16));
    if (run()) check(crfr_nchw_f32_to_nhwc_bf16(g, d, t.n, t.c, t.h, t.w, t.ld, t.ld, st));
    add_slot(t, d, t.ld);
  }

  void backward() {
    for (int i = (int)tape.size() - 1; i >= 0 && ok(); --i) {
      Op& op = tape[i];
      if (!has_grad(op.out)) continue;
      switch (op.kind) {
        case OP_BN: {
          squash(op.out, 2);
          std::vector<Slot>& s = slots[op.out.id];
          const Tensor& y = op.a;
          const long long count = (long long)y.n * y.h * y.w;
          const size_t bytes = (size_t)count * y.ld * sizeof(bf16);
          bf16* dz = (op.has_res || s.size() > 1) ? (bf16*)alloc(bytes) : nullptr;   // only if somebody consumes it
          bf16* dy = (bf16*)alloc(bytes);
          if (run())
            check(crfr_norm_act_bwd(s[0].p, s[0].ld, s.size() > 1 ? s[1].p : nullptr, s.size() > 1 ? s[1].ld : 8, y.p, y.ld,
                                    op.stats, params[op.g_idx], params[op.beta_idx], nullptr, op.relu ? 1 : 0,
                                    op.has_res ? op.b.p : nullptr, op.has_res ? op.b.ld : 8, dz, y.ld, dy, y.ld,
                                    grad(op.g_idx), grad(op.beta_idx), nullptr, 1, (int)count, y.c, scratch, scratch_bytes,
                                    st));
          add_slot(y, dy, y.ld);
          if (op.has_res) add_slot(op.b, dz, y.ld);
          break;
        }
        case OP_CONV: {
          squash(op.out, 1);
          Slot dy = slots[op.out.id][0];
          crfr_conv_desc d = op.cd;
          d.out_ld = dy.ld;
          if (run()) check(crfr_conv_wgrad(engine, &d, op.a.p, dy.p, grad(op.w_idx), nullptr, scratch, scratch_bytes, st));
          if (op.x_needs_grad) {
            const Tensor& x = op.a;
            bf16* dx = (bf16*)alloc((size_t)x.n * x.h * x.w * x.ld * sizeof(bf16));
            const int T = d.k * d.k;
            void* wt = alloc((size_t)T * d.cin * d.cout * sizeof(bf16));
            if (collect && ok()) collect->push_back({params[op.w_idx], wt, T, d.cin, d.cout, d.cout, T, (long long)d.cin * T, 0, 0});
            if (run()) {
              if (!packs_done)
                check(crfr_pack_weight(params[op.w_idx], wt, T, d.cin, d.cout, d.cout, T, (long long)d.cin * T, 1, st));
              check(crfr_conv_dgrad(engine, &d, dy.p, wt, d.cout, dx, scratch, scratch_bytes, st));
            }
            add_slot(x, dx, x.ld);
          }
          break;
        }
        case OP_LINEAR: {
          squash(op.out, 1);
          Slot dy = slots[op.out.id][0];
          const Tensor& a = op.a;
          const int B = a.n, K = a.h * a.w * a.c;
          bf16* da = (bf16*)alloc((size_t)B * K * sizeof(bf16));
          if (run()) {
            TcGemm g{dy.p, B, 1, 1, kEmb, dy.ld, wpt, 1, 0, 1, K, 0, da, K, 0, nullptr};
            check(crfr_tc_gemm(g, st));
            float* G = (float*)scratch;
            check_cuda(cudaMemsetAsync(G, 0, sizeof(float) * (size_t)K * kEmb, st));
            TcWgrad wg{a.p, B, 1, 1, K, K, dy.p, kEmb, dy.ld, 0, G};
            check(crfr_tc_wgrad_raw(wg, st));
            if (grad(op.w_idx)) {
              const long long total = (long long)kEmb * K;
              linear_unpack_kernel<<<crfr_cdiv(total, 256), 256, 0, st>>>(G, grad(op.w_idx), kEmb, a.c, a.h * a.w);
              CRFR_COUNT_LAUNCH();
              check_cuda(cudaGetLastError());
            }
            if (grad(op.b_idx)) check(crfr_colsum(dy.p, dy.ld, kEmb, B, grad(op.b_idx), scratch, scratch_bytes, st));
          }
          add_slot(a, da, K / (a.h * a.w));
          break;
        }
      }
    }
  }
};

int check_io(const crfr_resnet_io* io, const char* who) {
  CRFR_CHECK_ARG(io && io->batch > 0 && io->size == 112, "%s: batch/size invalid (input must be [B,3,112,112])", who);
  CRFR_CHECK_ARG(io->x && io->emb, "%s: null tensor pointer", who);
  CRFR_CHECK_ARG(io->eps > 0.f && io->momentum >= 0.f && io->momentum <= 1.f, "%s: eps/momentum invalid", who);
  return CRFR_OK;
}

void init_net(Net& net, int engine, const float* const* params, float* const* grads, void* const* buffers,
              const crfr_resnet_io* io, void* ws, size_t ws_bytes, cudaStream_t st, bool exec) {
  net.engine = engine; net.params = params; net.grads = grads; net.buffers = buffers; net.io = io; net.st = st;
  net.ws = (uint8_t*)ws; net.ws_bytes = ws_bytes; net.exec = exec;
}

}  // namespace

extern "C" size_t crfr_resnet34_workspace_bytes(int batch, int size, int training) {
  if (batch <= 0 || size != 112) return 0;
  crfr_resnet_io io = {};
  io.batch = batch; io.size = size; io.training = training; io.momentum = 0.1f; io.eps = 1e-5f;
  static float dummy = 0.f;   // non-null marker so that the dry run sizes every optional buffer
  Net net;
  init_net(net, CRFR_ENGINE_AUTO, nullptr, nullptr, nullptr, &io, nullptr, ~(size_t)0 >> 2, nullptr, false);
  net.forward();
  if (training) {
    for (int l = 0; l < 4; ++l) net.seed_grad(net.feat[l], &dummy);
    net.seed_grad(net.emb, &dummy);
    net.backward();
  }
  return net.off + 65536;
}

// Layout of the stored forward tensors of the ResNet_34 program in the workspace (a dry run: nothing is launched): one
// entry per recorded op in program order - kind 0 convolution, 1 BatchNorm (+ residual) (+ ReLU), 7 linear head; out_off /
// in_off / stats_off are bytes from the workspace base.  The parity tests read the stored bf16 activations through this
// table and replay them into the CPU oracle (teacher-forced forward / backward checks, tests/test_resnet_forced_gpu.py).
namespace {
// kinds: 0 convolution, 1 BatchNorm (+ residual) (+ ReLU / PReLU), 7 linear head, 8 PReLU pass, 9 stride-2 subsampling,
// 10 SE unit output (BatchNorm + excitation + residual; stats_off: the excitation e [n][c] fp32).
// Gradient tape of the IR backward (crfr_irnet_grad_tape; in_off: out_off of the stored forward tensor differentiated,
// w_idx: the unit, -1 outside the body): 11 the head's input gradient (at output_layer.0's input), 12 a unit's summed
// output gradient g, 13 an SE unit's dr at r = BN_4(y) (in_off: y; stats_off: shift [n][c] fp32 = dpool / hw), 14 the
// gradient at res_layer.1's output (after the PReLU pass), 15 a unit's input gradient, 16 the stem's dy0 (at
// input_layer.0's output)
int fill_tape(const Net& net, crfr_tape_entry* entries, int max_entries) {
  const int count = (int)net.tape.size();
  for (int i = 0; i < count && i < max_entries && entries; ++i) {
    const Op& op = net.tape[i];
    crfr_tape_entry& e = entries[i];
    const Tensor& t = op.out;
    e.kind = op.kind == OP_CONV ? 0 : op.kind == OP_BN ? 1 : op.kind == OP_LINEAR ? 7 : op.kind == OP_PRELU ? 8
           : op.kind == OP_SUB2 ? 9 : 10;
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

extern "C" int crfr_resnet34_tape(int batch, int size, int training, crfr_tape_entry* entries, int max_entries) {
  if (batch <= 0 || size != 112) return -1;
  crfr_resnet_io io = {};
  io.batch = batch; io.size = size; io.training = training; io.momentum = 0.1f; io.eps = 1e-5f;
  Net net;
  init_net(net, CRFR_ENGINE_AUTO, nullptr, nullptr, nullptr, &io, nullptr, ~(size_t)0 >> 2, nullptr, false);
  net.forward();
  return fill_tape(net, entries, max_entries);
}

namespace {
bool ir_variant_ok(int num_layers, int se) {
  int units[4];
  return ir_units_of(num_layers, units) && (se == 0 || se == 1);
}
int check_ir_variant(int num_layers, int se, const char* who) {
  CRFR_CHECK_ARG(ir_variant_ok(num_layers, se), "%s: unsupported IR variant (num_layers %d, se %d): 50, 100 or 152 layers, "
                 "se 0 or 1", who, num_layers, se);
  return CRFR_OK;
}
// a dry run of the IR program's forward (and, with grad, of its input gradient) at (batch, 112): arena offsets and tape
void ir_dry_run(Net& net, crfr_resnet_io& io, int num_layers, int se, int batch, int size, bool grad) {
  io = {};
  io.batch = batch; io.size = size; io.training = 0; io.momentum = 0.1f; io.eps = 1e-5f;
  init_net(net, CRFR_ENGINE_AUTO, nullptr, nullptr, nullptr, &io, nullptr, ~(size_t)0 >> 2, nullptr, false);
  net.ir_layers = num_layers; net.ir_se = se;
  net.forward_ir();
  if (grad) {
    static float dummy = 0.f;   // non-null marker so that the dry run sizes every optional buffer
    const float* feats[4] = {&dummy, &dummy, &dummy, &dummy};
    net.backward_ir(&dummy, feats, &dummy);
  }
}
}  // namespace

extern "C" int crfr_irnet_sizes(int num_layers, int se, int* n_params, int* n_bn) {
  CRFR_TRY(check_ir_variant(num_layers, se, "irnet_sizes"));
  int units[4];
  ir_units_of(num_layers, units);
  const int n = units[0] + units[1] + units[2] + units[3];
  if (n_params) *n_params = 10 + n * (se ? 9 : 7) + 3 * 3;   // three units have a conv1x1 + BN shortcut
  if (n_bn) *n_bn = 3 + 2 * n + 3;
  return CRFR_OK;
}

// The same table for the IR programs (eval mode): every stored tensor of crfr_irnet_forward in program order, for the
// teacher-forced parity tests of the input gradient (tests/test_ir50_grad_gpu.py, tests/test_irnet_gpu.py).
extern "C" int crfr_irnet_tape(int num_layers, int se, int batch, int size, crfr_tape_entry* entries, int max_entries) {
  if (!ir_variant_ok(num_layers, se) || batch <= 0 || size != 112) return -1;
  crfr_resnet_io io;
  Net net;
  ir_dry_run(net, io, num_layers, se, batch, size, false);
  return fill_tape(net, entries, max_entries);
}
// Where crfr_irnet_backward leaves each stored gradient: the dry run that the call performs (forward, then backward_ir
// with exec false), recorded from inside backward_ir, so the offsets are those of the real call.  seed_mask: which upstream
// gradients are given (1 = d_emb, 2 / 4 / 8 / 16 = d_feat[0..3]); the layout depends on it.
extern "C" int crfr_irnet_grad_tape(int num_layers, int se, int batch, int size, int seed_mask, crfr_tape_entry* entries,
                                    int max_entries) {
  if (!ir_variant_ok(num_layers, se) || batch <= 0 || size != 112 || seed_mask <= 0 || seed_mask > 31) return -1;
  crfr_resnet_io io;
  Net net;
  ir_dry_run(net, io, num_layers, se, batch, size, false);
  std::vector<crfr_tape_entry> rec;
  net.grad_tape = &rec;
  static float dummy = 0.f;   // non-null marker of a given seed
  const float* feats[4];
  for (int l = 0; l < 4; ++l) feats[l] = (seed_mask >> (l + 1)) & 1 ? &dummy : nullptr;
  net.backward_ir(seed_mask & 1 ? &dummy : nullptr, feats, &dummy);
  const int count = (int)rec.size();
  for (int i = 0; i < count && i < max_entries && entries; ++i) entries[i] = rec[i];
  return count;
}
extern "C" int crfr_ir50_tape(int batch, int size, crfr_tape_entry* entries, int max_entries) {
  return crfr_irnet_tape(50, 0, batch, size, entries, max_entries);
}

extern "C" int crfr_resnet34_forward(int engine, const float* const* host_params, void* const* host_buffers,
                                     const crfr_resnet_io* io, void* ws, size_t ws_bytes, void* stream) {
  CRFR_TRY(check_io(io, "resnet34_forward"));
  CRFR_CHECK_ARG(host_params && ws, "resnet34_forward: null pointer");
  CRFR_CHECK_ARG(io->training || host_buffers, "resnet34_forward: eval mode needs the running statistics");
  Net net;
  init_net(net, engine, host_params, nullptr, host_buffers, io, ws, ws_bytes, (cudaStream_t)stream, true);
  net.forward();
  return net.err;
}

// ------------------------------------------------------------------------------------------------------------
// Residual knowledge-distillation step (distill_main.py:59-74, evaluated on one forward: SURVEY.md 8c-iii):
// teacher forward (eval), student + assistant forward (train), the six MSE terms on the NHWC bf16 features as they
// sit in the workspace (no fp32 NCHW round trip), and both backward passes - one native call.
// ------------------------------------------------------------------------------------------------------------
namespace {

__global__ void kd_total_kernel(const float* __restrict__ parts, float* __restrict__ losses) {
  losses[0] = parts[0];
  losses[1] = ((parts[1] + parts[2]) + (parts[3] + parts[4])) + parts[5];
}

struct KdLayout {
  size_t teacher, train, scratch, total;
};
// ir_layers = 0: a ResNet_34 teacher, else the IR variant (ir_layers, ir_se)
KdLayout kd_layout(int batch, int size, int ir_layers = 0, int ir_se = 0) {
  KdLayout l;
  l.teacher = ((ir_layers ? crfr_irnet_workspace_bytes(ir_layers, ir_se, batch, size)
                          : crfr_resnet34_workspace_bytes(batch, size, 0)) + 4095) & ~(size_t)4095;
  // + room for the second embedding-gradient slot of the student (L_s and L_a both reach s_emb)
  l.train = (crfr_resnet34_workspace_bytes(batch, size, 1) + (size_t)batch * kEmb * 2 + (4u << 20)) & ~(size_t)4095;
  l.scratch = 1 << 20;
  l.total = l.teacher + 2 * l.train + l.scratch;
  return l;
}

}  // namespace

extern "C" size_t crfr_kd_workspace_bytes(int batch, int size) {
  if (batch <= 0 || size != 112) return 0;
  return kd_layout(batch, size).total;
}
extern "C" size_t crfr_kd_workspace_bytes_ex(int batch, int size, int teacher_ir50) {
  if (batch <= 0 || size != 112) return 0;
  return kd_layout(batch, size, teacher_ir50 ? 50 : 0).total;
}
extern "C" size_t crfr_kd_workspace_bytes_ir(int batch, int size, int teacher_ir_layers, int teacher_ir_se) {
  if (batch <= 0 || size != 112 || !ir_variant_ok(teacher_ir_layers, teacher_ir_se)) return 0;
  return kd_layout(batch, size, teacher_ir_layers, teacher_ir_se).total;
}

extern "C" int crfr_kd_train_step(int engine, const float* const* teacher_params, void* const* teacher_buffers,
                                  const float* const* student_params, void* const* student_buffers,
                                  float* const* student_grads, const float* const* assistant_params,
                                  void* const* assistant_buffers, float* const* assistant_grads, const crfr_kd_io* kio,
                                  float* losses, void* ws, size_t ws_bytes, void* stream) {
  CRFR_CHECK_ARG(kio && kio->batch > 0 && kio->size == 112 && kio->x, "kd_train_step: batch/size/x invalid");
  CRFR_CHECK_ARG(teacher_params && teacher_buffers && student_params && student_grads && assistant_params &&
                     assistant_grads && losses && ws,
                 "kd_train_step: null pointer");
  const int t_layers = kio->teacher_ir50 ? (kio->teacher_ir_layers ? kio->teacher_ir_layers : 50) : 0;
  const int t_se = kio->teacher_ir50 ? kio->teacher_ir_se : 0;
  if (t_layers) CRFR_TRY(check_ir_variant(t_layers, t_se, "kd_train_step"));
  const KdLayout lay = kd_layout(kio->batch, kio->size, t_layers, t_se);
  if (ws_bytes < lay.total) {
    crfr_set_error("kd_train_step: workspace %zu < %zu", ws_bytes, lay.total);
    return CRFR_EWORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  uint8_t* base = (uint8_t*)ws;
  crfr_resnet_io io_eval = {}, io_train = {};
  io_eval.batch = io_train.batch = kio->batch;
  io_eval.size = io_train.size = kio->size;
  io_eval.x = kio->x;                                  // HR batch for the teacher
  io_train.x = kio->x_lr ? kio->x_lr : kio->x;         // LR batch (or the same one, as distill_main.py:59-61 feeds it)
  io_eval.momentum = io_train.momentum = kio->momentum;
  io_eval.eps = io_train.eps = kio->eps;
  io_eval.training = 0;
  io_train.training = 1;
  // The program of one step over three networks; real = false: dry run (arena offsets and weight-pack jobs only)
  auto program = [&](Net& T, Net& S, Net& A, bool real) -> int {
    if (t_layers) {
      T.ir_layers = t_layers; T.ir_se = t_se;
      T.forward_ir();
    } else {
      T.forward();
    }
    if (!T.ok()) return T.err;
    S.forward();
    if (!S.ok()) return S.err;
    A.forward();
    if (!A.ok()) return A.err;

    float* parts = (float*)(base + lay.teacher + 2 * lay.train);   // [6] loss terms, then the reduction scratch
    void* lws = parts + 64;
    const size_t lws_bytes = lay.scratch - 64 * sizeof(float);
    const bool to_student = kio->assistant_grad_to_student != 0;
    auto grad_buf = [](Net& net, const Tensor& t) {
      bf16* g = (bf16*)net.alloc((size_t)t.n * t.h * t.w * t.ld * sizeof(bf16));
      net.add_slot(t, g, t.ld);
      return g;
    };
    // student loss: MSE(s_emb, t_emb.detach())
    {
      const long long numel = (long long)S.emb.n * S.emb.c;
      bf16* d_s = grad_buf(S, S.emb);
      if (real)
        CRFR_TRY(crfr_loss_kd(S.emb.p, nullptr, T.emb.p, numel, 0, 1.f, parts + 0, d_s, nullptr, nullptr, lws, lws_bytes, stream));
    }
    // assistant loss: sum_k MSE(t_k - s_k, a_k) over the four stage features and the embedding
    for (int k = 0; k < 5; ++k) {
      const Tensor& t = k < 4 ? T.feat[k] : T.emb;
      const Tensor& s_ = k < 4 ? S.feat[k] : S.emb;
      const Tensor& a = k < 4 ? A.feat[k] : A.emb;
      const long long numel = (long long)t.n * t.h * t.w * t.c;
      bf16* d_s = to_student ? grad_buf(S, s_) : nullptr;
      bf16* d_a = grad_buf(A, a);
      if (real)
        CRFR_TRY(crfr_loss_kd(t.p, s_.p, a.p, numel, 0, 1.f, parts + 1 + k, nullptr, d_s, d_a, lws, lws_bytes, stream));
    }
    if (!S.ok()) return S.err;
    if (!A.ok()) return A.err;
    if (real) {
      kd_total_kernel<<<1, 1, 0, st>>>(parts, losses);
      CRFR_COUNT_LAUNCH();
      CRFR_LAUNCH_CHECK();
    }
    S.backward();
    if (!S.ok()) return S.err;
    if (real && kio->events[0]) CRFR_CUDA(cudaEventRecord((cudaEvent_t)kio->events[0], st));   // student gradients are final
    A.backward();
    if (real && A.ok() && kio->events[1]) CRFR_CUDA(cudaEventRecord((cudaEvent_t)kio->events[1], st));
    return A.err;
  };
  {   // all weight packs of the step (three networks, both directions: ~180) as three launches
    std::vector<crfr_pack_job> jobs;
    Net T, S, A;
    init_net(T, engine, teacher_params, nullptr, teacher_buffers, &io_eval, base, lay.teacher, st, false);
    init_net(S, engine, student_params, student_grads, student_buffers, &io_train, base + lay.teacher, lay.train, st, false);
    init_net(A, engine, assistant_params, assistant_grads, assistant_buffers, &io_train, base + lay.teacher + lay.train,
             lay.train, st, false);
    T.collect = S.collect = A.collect = &jobs;
    CRFR_TRY(program(T, S, A, false));
    CRFR_TRY(crfr_pack_weight_batch(jobs.data(), (int)jobs.size(), st));
  }
  Net T, S, A;
  init_net(T, engine, teacher_params, nullptr, teacher_buffers, &io_eval, base, lay.teacher, st, true);
  init_net(S, engine, student_params, student_grads, student_buffers, &io_train, base + lay.teacher, lay.train, st, true);
  init_net(A, engine, assistant_params, assistant_grads, assistant_buffers, &io_train, base + lay.teacher + lay.train,
           lay.train, st, true);
  T.packs_done = S.packs_done = A.packs_done = true;
  return program(T, S, A, true);
}

extern "C" size_t crfr_irnet_workspace_bytes(int num_layers, int se, int batch, int size) {
  if (!ir_variant_ok(num_layers, se) || batch <= 0 || size != 112) return 0;
  crfr_resnet_io io;
  Net net;
  ir_dry_run(net, io, num_layers, se, batch, size, false);
  return net.off + 65536;
}
extern "C" size_t crfr_ir50_workspace_bytes(int batch, int size) { return crfr_irnet_workspace_bytes(50, 0, batch, size); }

extern "C" int crfr_irnet_forward(int engine, int num_layers, int se, const float* const* host_params,
                                  void* const* host_buffers, const crfr_resnet_io* io, void* ws, size_t ws_bytes,
                                  void* stream) {
  CRFR_TRY(check_ir_variant(num_layers, se, "irnet_forward"));
  CRFR_TRY(check_io(io, "irnet_forward"));
  CRFR_CHECK_ARG(host_params && host_buffers && ws, "irnet_forward: null pointer");
  CRFR_CHECK_ARG(!io->training, "irnet_forward: the teacher runs in eval mode only (train-mode Dropout is stochastic)");
  Net net;
  init_net(net, engine, host_params, nullptr, host_buffers, io, ws, ws_bytes, (cudaStream_t)stream, true);
  net.ir_layers = num_layers; net.ir_se = se;
  net.forward_ir();
  return net.err;
}
extern "C" int crfr_ir50_forward(int engine, const float* const* host_params, void* const* host_buffers,
                                 const crfr_resnet_io* io, void* ws, size_t ws_bytes, void* stream) {
  return crfr_irnet_forward(engine, 50, 0, host_params, host_buffers, io, ws, ws_bytes, stream);
}

// forward arena of crfr_irnet_workspace_bytes (same layout), then the input-gradient buffers
extern "C" size_t crfr_irnet_grad_workspace_bytes(int num_layers, int se, int batch, int size) {
  if (!ir_variant_ok(num_layers, se) || batch <= 0 || size != 112) return 0;
  crfr_resnet_io io;
  Net net;
  ir_dry_run(net, io, num_layers, se, batch, size, true);
  return net.off + 65536;
}
extern "C" size_t crfr_ir50_grad_workspace_bytes(int batch, int size) {
  return crfr_irnet_grad_workspace_bytes(50, 0, batch, size);
}

extern "C" int crfr_irnet_backward(int engine, int num_layers, int se, const float* const* host_params,
                                   void* const* host_buffers, const crfr_resnet_io* io, const float* d_emb,
                                   const float* const* d_feat, float* dx, void* ws, size_t ws_bytes, void* stream) {
  CRFR_TRY(check_ir_variant(num_layers, se, "irnet_backward"));
  CRFR_TRY(check_io(io, "irnet_backward"));
  CRFR_CHECK_ARG(host_params && dx && ws, "irnet_backward: null pointer");
  CRFR_CHECK_ARG(!io->training, "irnet_backward: the forward must have run in eval mode");
  const size_t need = crfr_irnet_grad_workspace_bytes(num_layers, se, io->batch, io->size);
  if (ws_bytes < need) {
    crfr_set_error("irnet_backward: workspace %zu < %zu (crfr_irnet_grad_workspace_bytes)", ws_bytes, need);
    return CRFR_EWORKSPACE;
  }
  Net net;
  init_net(net, engine, host_params, nullptr, host_buffers, io, ws, ws_bytes, (cudaStream_t)stream, false);
  net.ir_layers = num_layers; net.ir_se = se;
  net.forward_ir();   // dry run: rebuild the tape and the saved-activation offsets
  if (!net.ok()) return net.err;
  net.exec = true;
  net.backward_ir(d_emb, d_feat, dx);
  return net.err;
}
extern "C" int crfr_ir50_backward(int engine, const float* const* host_params, void* const* host_buffers,
                                  const crfr_resnet_io* io, const float* d_emb, const float* const* d_feat, float* dx,
                                  void* ws, size_t ws_bytes, void* stream) {
  return crfr_irnet_backward(engine, 50, 0, host_params, host_buffers, io, d_emb, d_feat, dx, ws, ws_bytes, stream);
}

extern "C" int crfr_resnet34_backward(int engine, const float* const* host_params, float* const* host_grads,
                                      const crfr_resnet_io* io, const float* d_emb, const float* const* d_feat,
                                      void* ws, size_t ws_bytes, void* stream) {
  CRFR_TRY(check_io(io, "resnet34_backward"));
  CRFR_CHECK_ARG(host_params && host_grads && ws, "resnet34_backward: null pointer");
  CRFR_CHECK_ARG(io->training, "resnet34_backward: the forward must have run in training mode");
  Net net;
  init_net(net, engine, host_params, host_grads, nullptr, io, ws, ws_bytes, (cudaStream_t)stream, false);
  net.forward();   // dry run: rebuild the tape and the saved-activation offsets
  if (!net.ok()) return net.err;
  net.exec = true;
  for (int l = 0; l < 4; ++l) net.seed_grad(net.feat[l], d_feat ? d_feat[l] : nullptr);
  net.seed_grad(net.emb, d_emb);
  if (!net.ok()) return net.err;
  net.backward();
  return net.err;
}
