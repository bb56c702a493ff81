// Fused loss forward+backward kernels (HBM-bound, one pass over the prediction and target, deterministic
// two-stage reductions: per-block partials in the workspace, fixed-order finalisation in double).
// ref: loss/loss.py:7-15 (MSELossFunc), :17-32 (MSELoss_Landmark), :34-62 (CrossEntropyLoss2d),
//      distill_main.py:63,68-70 (nn.MSELoss residual-KD terms).
#include "common.cuh"
#include "crfr.h"
#include "internal.h"

namespace {

constexpr int kT = 256;

__device__ __forceinline__ void block_partial(float v, float* partial) {
  __shared__ float sm[kT / 32];
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int i = 0; i < kT / 32; ++i) s += sm[i];
    partial[blockIdx.x] = s;
  }
}

__global__ void finalize_kernel(const float* __restrict__ partial, int nblocks, double scale, float* __restrict__ loss) {
  __shared__ double sm[kT];
  double s = 0.0;
  for (int i = threadIdx.x; i < nblocks; i += kT) s += (double)partial[i];
  sm[threadIdx.x] = s;
  __syncthreads();
  for (int o = kT / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) sm[threadIdx.x] += sm[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) loss[0] = (float)(sm[0] * scale);
}

// partial layout: [1 + (dchan ? c : 0)][gridDim.x] - squared-error partials first, then per-channel sums of (x - t)
__global__ void __launch_bounds__(kT)
mse97_kernel(const float* __restrict__ x, const float* __restrict__ t, long long npix, int hw, int c, float gcoef,
             bf16* __restrict__ dx, int dx_ld, float* __restrict__ partial, int want_chan) {
  long long i = (long long)blockIdx.x * kT + threadIdx.x;
  float acc = 0.f;
  float dsum[4] = {0.f, 0.f, 0.f, 0.f};
  if (i < npix) {
    long long n = i / hw;
    int p = (int)(i - n * hw);
    const float* xs = x + n * (long long)c * hw + p;
    const float* ts = t + n * (long long)c * hw + p;
    for (int ch = 0; ch < c; ++ch) {
      float d = xs[(long long)ch * hw] - ts[(long long)ch * hw];
      acc += d * d;
      if (ch < 4) dsum[ch] = d;
      if (dx) dx[i * dx_ld + ch] = __float2bfloat16_rn(gcoef * d);
    }
    if (dx)
      for (int ch = c; ch < dx_ld; ++ch) dx[i * dx_ld + ch] = __float2bfloat16_rn(0.f);
  }
  block_partial(acc, partial);
  if (want_chan)
    for (int ch = 0; ch < c && ch < 4; ++ch) {
      __syncthreads();
      block_partial(dsum[ch], partial + (size_t)(1 + ch) * gridDim.x);
    }
}

// dchan[ch] += scale * sum(partial[ch][0..nblocks)) in double, fixed order (one block per channel)
__global__ void chan_finalize_kernel(const float* __restrict__ partial, int nblocks, double scale,
                                     float* __restrict__ dchan) {
  __shared__ double sm[kT];
  const float* pp = partial + (size_t)blockIdx.x * nblocks;
  double s = 0.0;
  for (int i = threadIdx.x; i < nblocks; i += kT) s += (double)pp[i];
  sm[threadIdx.x] = s;
  __syncthreads();
  for (int o = kT / 2; o > 0; o >>= 1) {
    if (threadIdx.x < o) sm[threadIdx.x] += sm[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) dchan[blockIdx.x] += (float)(sm[0] * scale);
}

// One thread per window pixel: dx at the pixel = bf16(gcoef * (x - t) + g), the first term computed exactly as
// mse97_kernel does (so that g = 0 reproduces its bits); partial[ch][block] = the block's sum of g (c <= 4)
__global__ void __launch_bounds__(kT)
mse97_window_kernel(const float* __restrict__ x, const float* __restrict__ t, int c, int h, int w, float gcoef,
                    const bf16* __restrict__ g, int gh, int gw, int g_ld, int oy, int ox, bf16* __restrict__ dx, int dx_ld,
                    long long npix, float* __restrict__ partial) {
  const long long i = (long long)blockIdx.x * kT + threadIdx.x;
  float gsum[4] = {0.f, 0.f, 0.f, 0.f};
  if (i < npix) {
    const long long n = i / ((long long)gh * gw);
    const int p = (int)(i - n * gh * gw), y = p / gw, xx = p - (p / gw) * gw;
    const long long q = (n * h + oy + y) * w + ox + xx;     // pixel of the full image
    const long long hw = (long long)h * w;
    for (int ch = 0; ch < c; ++ch) {
      const long long e = (n * c + ch) * hw + (q - n * hw);
      const float d = x[e] - t[e];
      const float gi = __bfloat162float(g[i * g_ld + ch]);
      gsum[ch] = gi;
      dx[q * dx_ld + ch] = __float2bfloat16_rn(__fmaf_rn(gcoef, d, gi));
    }
  }
  if (partial)
    for (int ch = 0; ch < c; ++ch) {
      if (ch) __syncthreads();
      block_partial(gsum[ch], partial + (size_t)ch * gridDim.x);
    }
}

// per-(block, channel) partial sums of an fp32 NCHW tensor: grid (chunks, c), partial[c][chunks]
__global__ void __launch_bounds__(kT)
nchw_chansum_kernel(const float* __restrict__ g, int n, int c, int hw, float* __restrict__ partial) {
  const int ch = blockIdx.y;
  const long long total = (long long)n * hw;
  float acc = 0.f;
  for (long long i = (long long)blockIdx.x * kT + threadIdx.x; i < total; i += (long long)gridDim.x * kT) {
    const long long img = i / hw;
    acc += g[(img * c + ch) * hw + (i - img * hw)];
  }
  block_partial(acc, partial + (size_t)ch * gridDim.x);
}

__global__ void __launch_bounds__(kT)
landmark_kernel(const float* __restrict__ x, const float* __restrict__ t, long long npix, int hw, int c, float gcoef,
                bf16* __restrict__ dx, int dx_ld, int coff, float* __restrict__ partial) {
  long long i = (long long)blockIdx.x * kT + threadIdx.x;
  float acc = 0.f, d = 0.f;
  if (i < npix) {
    long long n = i / hw;
    int p = (int)(i - n * hw);
    const float* xs = x + n * (long long)c * hw + p;
    float s = 0.f;
#pragma unroll 8
    for (int ch = 0; ch < c; ++ch) s += xs[(long long)ch * hw];   // same order as written; the loads are independent
    d = s - t[i];
    acc = d * d;
  }
  if (dx) {
    // every channel of a pixel gets the same gradient: the warp writes its 32 pixels' rows one after the other, each lane
    // a 4-byte pair of the row (coalesced), instead of every lane walking its own row with 2-byte stores 2 * dx_ld bytes
    // apart from its neighbours' (137 us for 128 images)
    const unsigned short gb = __bfloat16_as_ushort(__float2bfloat16_rn(gcoef * d));
    const int lane = threadIdx.x & 31;
    const long long wbase = i - lane;
    for (int k = 0; k < 32; ++k) {
      const unsigned short gk = (unsigned short)__shfl_sync(0xffffffffu, (int)gb, k);
      const long long ik = wbase + k;
      if (ik >= npix) break;                                    // warp-uniform
      unsigned short* row = reinterpret_cast<unsigned short*>(dx) + ik * dx_ld + coff;
      const int head = (int)(((uintptr_t)row >> 1) & 1);        // the row starts in the middle of a 4-byte word
      if (head && lane == 0) row[0] = gk;
      const int pairs = (c - head) >> 1;
      uint32_t* rw = reinterpret_cast<uint32_t*>(row + head);
      const uint32_t gg = (uint32_t)gk | ((uint32_t)gk << 16);
      for (int w = lane; w < pairs; w += 32) rw[w] = gg;
      if (((c - head) & 1) && lane == 0) row[c - 1] = gk;
    }
  }
  block_partial(acc, partial);
}

__global__ void __launch_bounds__(kT)
ce2d_kernel(const float* __restrict__ x, const long long* __restrict__ target, long long npix, int hw, int c,
            float gcoef, bf16* __restrict__ dx, int dx_ld, int coff, float* __restrict__ partial) {
  long long i = (long long)blockIdx.x * kT + threadIdx.x;
  float acc = 0.f;
  if (i < npix) {
    long long n = i / hw;
    int p = (int)(i - n * hw);
    const float* xs = x + n * (long long)c * hw + p;
    float m = -INFINITY;
    for (int ch = 0; ch < c; ++ch) m = fmaxf(m, xs[(long long)ch * hw]);
    float se = 0.f;
    for (int ch = 0; ch < c; ++ch) se += expf(xs[(long long)ch * hw] - m);
    float lse = m + logf(se);
    const long long tl = target[i];
    // torch's NLLLoss raises on a label outside [0, c); a kernel cannot raise, so such a pixel poisons the loss with NaN
    // (loud, and no out-of-bounds read) and contributes no gradient
    const bool valid = tl >= 0 && tl < c;
    const int tg = valid ? (int)tl : 0;
    acc = valid ? lse - xs[(long long)tg * hw] : __int_as_float(0x7fc00000);
    if (dx)
      for (int ch = 0; ch < c; ++ch) {
        float sm = expf(xs[(long long)ch * hw] - lse);
        dx[i * dx_ld + coff + ch] = __float2bfloat16_rn(valid ? gcoef * (sm - (ch == tg ? 1.f : 0.f)) : 0.f);
      }
  }
  block_partial(acc, partial);
}

template <typename T> __device__ __forceinline__ float ldf(const T* p, long long i);
template <> __device__ __forceinline__ float ldf<float>(const float* p, long long i) { return p[i]; }
template <> __device__ __forceinline__ float ldf<bf16>(const bf16* p, long long i) { return __bfloat162float(p[i]); }
__device__ __forceinline__ void stf(float* p, long long i, float v) { p[i] = v; }
__device__ __forceinline__ void stf(bf16* p, long long i, float v) { p[i] = __float2bfloat16_rn(v); }

template <typename T>
__global__ void __launch_bounds__(kT)
kd_kernel(const T* __restrict__ t, const T* __restrict__ s, const T* __restrict__ a, long long numel, float gcoef,
          T* __restrict__ dt, T* __restrict__ ds, T* __restrict__ da, float* __restrict__ partial) {
  float acc = 0.f;
  for (long long i = (long long)blockIdx.x * kT + threadIdx.x; i < numel; i += (long long)gridDim.x * kT) {
    float r = ldf(t, i) - (s ? ldf(s, i) : 0.f) - ldf(a, i);
    acc += r * r;
    float g = gcoef * r;
    if (dt) stf(dt, i, g);
    if (ds) stf(ds, i, -g);
    if (da) stf(da, i, -g);
  }
  block_partial(acc, partial);
}

int check_ws(const char* who, void* ws, size_t ws_bytes, int blocks) {
  if (!ws || ws_bytes < sizeof(float) * (size_t)blocks) {
    crfr_set_error("%s: workspace %zu < %zu", who, ws_bytes, sizeof(float) * (size_t)blocks);
    return CRFR_EWORKSPACE;
  }
  return CRFR_OK;
}

}  // namespace

// dchan (optional, c <= 4): dchan[ch] += sum over all pixels of the fp32 loss gradient of channel ch (the bias gradient of
// the convolution that produced x; kept in fp32 because the bf16-rounded map sums with heavy cancellation)
int crfr_loss_mse97_chan(const float* x, const float* t, int n, int c, int hw, float gscale, float* loss, void* dx,
                         int dx_ld, float* dchan, void* ws, size_t ws_bytes, cudaStream_t st) {
  CRFR_CHECK_ARG(x && t && loss && n > 0 && c > 0 && hw > 0 && (!dx || dx_ld >= c) && (!dchan || c <= 4),
                 "loss_mse97: bad argument");
  long long npix = (long long)n * hw;
  int blocks = crfr_cdiv(npix, kT);
  CRFR_TRY(check_ws("loss_mse97", ws, ws_bytes, blocks * (dchan ? 1 + c : 1)));
  double numel = (double)npix * c;
  const double gcoef = gscale * 2.0 * 97.0 / numel;
  mse97_kernel<<<blocks, kT, 0, st>>>(x, t, npix, hw, c, (float)gcoef, (bf16*)dx, dx_ld, (float*)ws, dchan ? 1 : 0);
  CRFR_COUNT_LAUNCH();
  finalize_kernel<<<1, kT, 0, st>>>((const float*)ws, blocks, 97.0 / numel, loss);
  CRFR_COUNT_LAUNCH();
  if (dchan) {
    chan_finalize_kernel<<<c, kT, 0, st>>>((const float*)ws + blocks, blocks, gcoef, dchan);
    CRFR_COUNT_LAUNCH();
  }
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

extern "C" int crfr_loss_mse97(const float* x, const float* t, int n, int c, int hw, float gscale, float* loss,
                               void* dx, int dx_ld, void* ws, size_t ws_bytes, void* stream) {
  return crfr_loss_mse97_chan(x, t, n, c, hw, gscale, loss, dx, dx_ld, nullptr, ws, ws_bytes, (cudaStream_t)stream);
}

int crfr_mse97_add_window_grad(const float* x, const float* t, int n, int c, int h, int w, float gscale, const void* g,
                               int gh, int gw, int g_ld, int oy, int ox, void* dx, int dx_ld, float* dchan, void* ws,
                               size_t ws_bytes, cudaStream_t st) {
  CRFR_CHECK_ARG(x && t && g && dx && n > 0 && c > 0 && c <= 4 && g_ld >= c && dx_ld >= c && oy >= 0 && ox >= 0 &&
                     oy + gh <= h && ox + gw <= w && gh > 0 && gw > 0,
                 "mse97_add_window_grad: bad argument");
  const long long npix = (long long)n * gh * gw;
  const int blocks = crfr_cdiv(npix, kT);
  if (dchan) CRFR_TRY(check_ws("mse97_add_window_grad", ws, ws_bytes, blocks * c));
  const double gcoef = gscale * 2.0 * 97.0 / ((double)n * h * w * c);   // as crfr_loss_mse97_chan
  mse97_window_kernel<<<blocks, kT, 0, st>>>(x, t, c, h, w, (float)gcoef, (const bf16*)g, gh, gw, g_ld, oy, ox, (bf16*)dx,
                                             dx_ld, npix, dchan ? (float*)ws : nullptr);
  CRFR_COUNT_LAUNCH();
  if (dchan) {
    chan_finalize_kernel<<<c, kT, 0, st>>>((const float*)ws, blocks, 1.0, dchan);
    CRFR_COUNT_LAUNCH();
  }
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

// out[ch] += sum over (n, h, w) of g[n][ch][h][w]  (fp32 NCHW), deterministic two-stage reduction
int crfr_nchw_chansum(const float* g, int n, int c, int hw, float* out, void* ws, size_t ws_bytes, cudaStream_t st) {
  CRFR_CHECK_ARG(g && out && n > 0 && c > 0 && hw > 0, "nchw_chansum: bad argument");
  long long total = (long long)n * hw;
  int chunks = (int)((total + kT * 8 - 1) / (kT * 8));
  if (chunks > 592) chunks = 592;
  if (chunks < 1) chunks = 1;
  CRFR_TRY(check_ws("nchw_chansum", ws, ws_bytes, chunks * c));
  nchw_chansum_kernel<<<dim3(chunks, c), kT, 0, st>>>(g, n, c, hw, (float*)ws);
  CRFR_COUNT_LAUNCH();
  chan_finalize_kernel<<<c, kT, 0, st>>>((const float*)ws, chunks, 1.0, out);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

extern "C" int crfr_loss_landmark(const float* x, const float* t, int n, int c, int hw, float gscale, float* loss,
                                  void* dx, int dx_ld, int dx_coff, void* ws, size_t ws_bytes, void* stream) {
  CRFR_CHECK_ARG(x && t && loss && n > 0 && c > 0 && hw > 0 && (!dx || dx_ld >= dx_coff + c),
                 "loss_landmark: bad argument");
  long long npix = (long long)n * hw;
  int blocks = crfr_cdiv(npix, kT);
  CRFR_TRY(check_ws("loss_landmark", ws, ws_bytes, blocks));
  cudaStream_t st = (cudaStream_t)stream;
  landmark_kernel<<<blocks, kT, 0, st>>>(x, t, npix, hw, c, (float)(gscale * 2.0 * 97.0 / (double)npix), (bf16*)dx,
                                         dx_ld, dx_coff, (float*)ws);
  CRFR_COUNT_LAUNCH();
  finalize_kernel<<<1, kT, 0, st>>>((const float*)ws, blocks, 97.0 / (double)npix, loss);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

extern "C" int crfr_loss_ce2d(const float* logits, const long long* target, int n, int c, int hw, float gscale,
                              float* loss, void* dx, int dx_ld, int dx_coff, void* ws, size_t ws_bytes,
                              void* stream) {
  CRFR_CHECK_ARG(logits && target && loss && n > 0 && c > 0 && hw > 0 && (!dx || dx_ld >= dx_coff + c),
                 "loss_ce2d: bad argument");
  long long npix = (long long)n * hw;
  int blocks = crfr_cdiv(npix, kT);
  CRFR_TRY(check_ws("loss_ce2d", ws, ws_bytes, blocks));
  cudaStream_t st = (cudaStream_t)stream;
  ce2d_kernel<<<blocks, kT, 0, st>>>(logits, target, npix, hw, c, (float)(gscale / (double)npix), (bf16*)dx, dx_ld,
                                     dx_coff, (float*)ws);
  CRFR_COUNT_LAUNCH();
  finalize_kernel<<<1, kT, 0, st>>>((const float*)ws, blocks, 1.0 / (double)npix, loss);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

extern "C" int crfr_loss_kd(const void* t, const void* s, const void* a, long long numel, int is_f32, float gscale,
                            float* loss, void* dt, void* ds, void* da, void* ws, size_t ws_bytes, void* stream) {
  CRFR_CHECK_ARG(t && a && loss && numel > 0, "loss_kd: bad argument");
  int blocks = (int)((numel + kT - 1) / kT);
  if (blocks > 148 * 16) blocks = 148 * 16;
  CRFR_TRY(check_ws("loss_kd", ws, ws_bytes, blocks));
  cudaStream_t st = (cudaStream_t)stream;
  float gcoef = (float)(gscale * 2.0 / (double)numel);
  if (is_f32)
    kd_kernel<float><<<blocks, kT, 0, st>>>((const float*)t, (const float*)s, (const float*)a, numel, gcoef,
                                            (float*)dt, (float*)ds, (float*)da, (float*)ws);
  else
    kd_kernel<bf16><<<blocks, kT, 0, st>>>((const bf16*)t, (const bf16*)s, (const bf16*)a, numel, gcoef, (bf16*)dt,
                                           (bf16*)ds, (bf16*)da, (float*)ws);
  CRFR_COUNT_LAUNCH();
  finalize_kernel<<<1, kT, 0, st>>>((const float*)ws, blocks, 1.0 / (double)numel, loss);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}
