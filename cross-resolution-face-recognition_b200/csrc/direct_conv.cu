// Generic CUDA-core convolution family: any kernel size / stride / padding, Conv2d and ConvTranspose2d, forward,
// dgrad and wgrad.  It serves (a) the edge layers whose channel counts do not fill a tcgen05 tile (3-channel
// images, the 108-wide prior heads) and (b) as an on-GPU cross-check for the tcgen05 engine.
//
// Geometry vocabulary: a convolution couples a "big" grid (conv input / deconv output, bh x bw) with a "small"
// grid (conv output / deconv input, sh x sw):  big = small * stride - pad + tap.
//   gather_down : small[p][r] = bias[r] + sum_{tap,s} big[p*stride - pad + tap][s] * W[tap][r][s]
//                 (Conv2d forward, ConvTranspose2d dgrad)
//   gather_up   : big[P][r]   = bias[r] + sum_{tap valid,s} small[(P + pad - tap)/stride][s] * W[tap][r][s]
//                 (Conv2d dgrad, ConvTranspose2d forward)
//   wgrad       : G[a][b][tap] += sum_p small[p][a] * big[p*stride - pad + tap][b]
// ref: nn.Conv2d / nn.ConvTranspose2d call sites listed in include/crfr.h.
#include "common.cuh"
#include "crfr.h"

namespace {

struct Geo {
  int n, bh, bw, sh, sw, k, stride, pad;
};

// ------------------------------------------------------------------------------------------------
// load S_VEC source channels starting at element pointer p into f[]
template <int V> __device__ __forceinline__ void load_vec(const bf16* p, float* f);
template <> __device__ __forceinline__ void load_vec<8>(const bf16* p, float* f) {
  unpack8(*reinterpret_cast<const bf16x8*>(p), f);
}
template <> __device__ __forceinline__ void load_vec<4>(const bf16* p, float* f) {
  bf16x4 v = *reinterpret_cast<const bf16x4*>(p);
  float2 a = __bfloat1622float2(v.v[0]), b = __bfloat1622float2(v.v[1]);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y;
}
template <int V> __device__ __forceinline__ void load_vec_ldg(const bf16* p, float* f);
template <> __device__ __forceinline__ void load_vec_ldg<8>(const bf16* p, float* f) {
  uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
  unpack8(*reinterpret_cast<const bf16x8*>(&u), f);
}
template <> __device__ __forceinline__ void load_vec_ldg<4>(const bf16* p, float* f) {
  uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
  bf16x4 v = *reinterpret_cast<const bf16x4*>(&u);
  float2 a = __bfloat1622float2(v.v[0]), b = __bfloat1622float2(v.v[1]);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y;
}

template <int COG>
__device__ __forceinline__ void store_result(const float* acc, int r0, int R, long long pix, bf16* y, int y_ld,
                                             float* y_nchw, long long n, int p_in_img, int img_pix) {
  if (y) {
    if (COG == 8 && r0 + 8 <= R && (y_ld & 7) == 0) {
      *reinterpret_cast<bf16x8*>(y + pix * y_ld + r0) = pack8(acc);
    } else {
#pragma unroll
      for (int j = 0; j < COG; ++j) {
        if (r0 + j < R) y[pix * y_ld + r0 + j] = __float2bfloat16_rn(acc[j]);
        else if (r0 + j < y_ld) y[pix * y_ld + r0 + j] = __float2bfloat16_rn(0.f);  // zero the channel padding
      }
    }
  }
  if (y_nchw) {
#pragma unroll
    for (int j = 0; j < COG; ++j)
      if (r0 + j < R) y_nchw[(n * R + r0 + j) * img_pix + p_in_img] = acc[j];
  }
}

// small[p][r] = bias[r] + sum big[...] * W[tap][r][s]
template <int COG, int V>
__global__ void __launch_bounds__(128)
gather_down_kernel(Geo g, const bf16* __restrict__ big, int big_ld, const bf16* __restrict__ w, int R, int s_pad,
                   const float* __restrict__ bias, bf16* __restrict__ y, int y_ld, float* __restrict__ y_nchw) {
  const long long npix = (long long)g.n * g.sh * g.sw;
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int rgroups = (R + COG - 1) / COG;
  if (idx >= npix * rgroups) return;
  const int rg = (int)(idx / npix);
  const long long pix = idx - (long long)rg * npix;
  const int sx = (int)(pix % g.sw);
  const long long q = pix / g.sw;
  const int sy = (int)(q % g.sh);
  const long long n = q / g.sh;
  const int r0 = rg * COG;
  float acc[COG];
#pragma unroll
  for (int j = 0; j < COG; ++j) acc[j] = (bias && r0 + j < R) ? bias[r0 + j] : 0.f;
  for (int ky = 0; ky < g.k; ++ky) {
    const int by = sy * g.stride - g.pad + ky;
    if (by < 0 || by >= g.bh) continue;
    for (int kx = 0; kx < g.k; ++kx) {
      const int bx = sx * g.stride - g.pad + kx;
      if (bx < 0 || bx >= g.bw) continue;
      const bf16* src = big + ((n * g.bh + by) * g.bw + bx) * big_ld;
      const bf16* wt = w + ((long long)(ky * g.k + kx) * R + r0) * s_pad;
      for (int s = 0; s < s_pad; s += V) {
        float xv[V];
        load_vec<V>(src + s, xv);
#pragma unroll
        for (int j = 0; j < COG; ++j) {
          if (r0 + j < R) {
            float wv[V];
            load_vec_ldg<V>(wt + (long long)j * s_pad + s, wv);
#pragma unroll
            for (int e = 0; e < V; ++e) acc[j] = fmaf(xv[e], wv[e], acc[j]);
          }
        }
      }
    }
  }
  store_result<COG>(acc, r0, R, pix, y, y_ld, y_nchw, n, sy * g.sw + sx, g.sh * g.sw);
}

// big[P][r] = bias[r] + sum_{valid taps} small[(P + pad - tap)/stride][s] * W[tap][r][s]
template <int COG, int V>
__global__ void __launch_bounds__(128)
gather_up_kernel(Geo g, const bf16* __restrict__ small, int small_ld, const bf16* __restrict__ w, int R, int s_pad,
                 const float* __restrict__ bias, bf16* __restrict__ y, int y_ld, float* __restrict__ y_nchw) {
  const long long npix = (long long)g.n * g.bh * g.bw;
  long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int rgroups = (R + COG - 1) / COG;
  if (idx >= npix * rgroups) return;
  const int rg = (int)(idx / npix);
  const long long pix = idx - (long long)rg * npix;
  const int bx = (int)(pix % g.bw);
  const long long q = pix / g.bw;
  const int by = (int)(q % g.bh);
  const long long n = q / g.bh;
  const int r0 = rg * COG;
  float acc[COG];
#pragma unroll
  for (int j = 0; j < COG; ++j) acc[j] = (bias && r0 + j < R) ? bias[r0 + j] : 0.f;
  for (int ky = 0; ky < g.k; ++ky) {
    const int ty = by + g.pad - ky;
    if (ty < 0 || ty % g.stride) continue;
    const int sy = ty / g.stride;
    if (sy >= g.sh) continue;
    for (int kx = 0; kx < g.k; ++kx) {
      const int tx = bx + g.pad - kx;
      if (tx < 0 || tx % g.stride) continue;
      const int sx = tx / g.stride;
      if (sx >= g.sw) continue;
      const bf16* src = small + ((n * g.sh + sy) * g.sw + sx) * small_ld;
      const bf16* wt = w + ((long long)(ky * g.k + kx) * R + r0) * s_pad;
      for (int s = 0; s < s_pad; s += V) {
        float xv[V];
        load_vec<V>(src + s, xv);
#pragma unroll
        for (int j = 0; j < COG; ++j) {
          if (r0 + j < R) {
            float wv[V];
            load_vec_ldg<V>(wt + (long long)j * s_pad + s, wv);
#pragma unroll
            for (int e = 0; e < V; ++e) acc[j] = fmaf(xv[e], wv[e], acc[j]);
          }
        }
      }
    }
  }
  store_result<COG>(acc, r0, R, pix, y, y_ld, y_nchw, n, by * g.bw + bx, g.bh * g.bw);
}

// G[chunk][(a*B + b)*T + tap] = sum over the chunk's pixels p of small[p][a] * big[p*stride - pad + tap][b]
// grid: (pixel chunks, taps, pair blocks); each thread owns up to MAXP (a, 4 consecutive b) pairs.  Every chunk stores its own
// slice; sum_chunks_kernel adds the slices in chunk order (no float atomics: the same bits on every run).
constexpr int kWgThreads = 256;
constexpr int kMaxPairs = 4;
__global__ void __launch_bounds__(kWgThreads)
wgrad_kernel(Geo g, const bf16* __restrict__ small, int small_ld, int A, const bf16* __restrict__ big, int big_ld,
             int B, int chunk_pix, float* __restrict__ G) {
  const int b4n = (B + 3) >> 2;
  const int npairs = A * b4n;
  const int tap = blockIdx.y, ky = tap / g.k, kx = tap - ky * g.k;
  const int T = g.k * g.k;
  int pa[kMaxPairs], pb[kMaxPairs];
  bool live[kMaxPairs];
  float acc[kMaxPairs][4];
#pragma unroll
  for (int m = 0; m < kMaxPairs; ++m) {
    int pr = (blockIdx.z * kMaxPairs + m) * kWgThreads + threadIdx.x;
    live[m] = pr < npairs;
    pa[m] = live[m] ? pr / b4n : 0;
    pb[m] = live[m] ? (pr - pa[m] * b4n) * 4 : 0;
#pragma unroll
    for (int e = 0; e < 4; ++e) acc[m][e] = 0.f;
  }
  const long long npix = (long long)g.n * g.sh * g.sw;
  G += (long long)blockIdx.x * A * B * T;
  const long long p0 = (long long)blockIdx.x * chunk_pix;
  const long long p1 = min(npix, p0 + (long long)chunk_pix);
  for (long long p = p0; p < p1; ++p) {
    const int sx = (int)(p % g.sw);
    const long long q = p / g.sw;
    const int sy = (int)(q % g.sh);
    const long long n = q / g.sh;
    const int by = sy * g.stride - g.pad + ky, bx = sx * g.stride - g.pad + kx;
    if (by < 0 || by >= g.bh || bx < 0 || bx >= g.bw) continue;  // uniform across the CTA
    const bf16* sp = small + p * small_ld;
    const bf16* bp = big + ((n * g.bh + by) * g.bw + bx) * big_ld;
#pragma unroll
    for (int m = 0; m < kMaxPairs; ++m) {
      if (live[m]) {
        float sv = __bfloat162float(sp[pa[m]]);
        float bv[4];
        load_vec<4>(bp + pb[m], bv);
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[m][e] = fmaf(sv, bv[e], acc[m][e]);
      }
    }
  }
#pragma unroll
  for (int m = 0; m < kMaxPairs; ++m) {
    if (live[m]) {
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (pb[m] + e < B) G[((long long)pa[m] * B + pb[m] + e) * T + tap] = acc[m][e];
    }
  }
}

// part[chunk][c] = sum over the chunk's pixels of t[pix][c]
__global__ void __launch_bounds__(256)
colsum_kernel(const bf16* __restrict__ t, int ld, int c_total, long long npix, int chunk_pix, float* __restrict__ part) {
  extern __shared__ float sm[];  // [lanes][c]
  // blockIdx.y selects a block of up to 256 channels
  const int coff = blockIdx.y * 256;
  const int c = min(256, c_total - coff);
  const int lanes = 256 / c > 0 ? 256 / c : 1;
  const int ch = threadIdx.x % c, lane = threadIdx.x / c;
  float acc = 0.f;
  const long long p0 = (long long)blockIdx.x * chunk_pix, p1 = min(npix, p0 + (long long)chunk_pix);
  if (lane < lanes)
    for (long long p = p0 + lane; p < p1; p += lanes) acc += __bfloat162float(t[p * ld + coff + ch]);
  if (lane < lanes) sm[lane * c + ch] = acc;
  __syncthreads();
  if (threadIdx.x < c) {
    float s = 0.f;
    for (int l = 0; l < lanes; ++l) s += sm[l * c + threadIdx.x];
    part[(long long)blockIdx.x * c_total + coff + threadIdx.x] = s;
  }
}

// out[i] += sum over the chunks of part[chunk][i], in chunk order
__global__ void sum_chunks_kernel(const float* __restrict__ part, int chunks, long long n, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = out[i];
  for (int k = 0; k < chunks; ++k) s += part[k * n + i];
  out[i] = s;
}

// as many chunks of the pixel range as `want` asks for and the workspace holds `slice` floats each (at least one)
long long fit_chunks(long long want, long long slice, size_t ws_bytes) {
  const long long fit = (long long)(ws_bytes / (sizeof(float) * (size_t)slice));
  return want < fit ? want : (fit > 1 ? fit : 1);
}

int sum_chunks(const float* part, long long chunks, long long n, float* out, cudaStream_t st) {
  sum_chunks_kernel<<<crfr_cdiv(n, 256), 256, 0, st>>>(part, (int)chunks, n, out);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

template <typename K>
int launch_gather(K kern, const Geo& g, long long npix, int R, int cog, cudaStream_t st, const bf16* src, int src_ld,
                  const bf16* w, int s_pad, const float* bias, bf16* y, int y_ld, float* y_nchw) {
  long long total = npix * ((R + cog - 1) / cog);
  kern<<<crfr_cdiv(total, 128), 128, 0, st>>>(g, src, src_ld, w, R, s_pad, bias, y, y_ld, y_nchw);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

}  // namespace

// ---- internal entry points used by conv_api.cu ---------------------------------------------------
// down != 0: gather_down (result on the small grid), else gather_up (result on the big grid)
int crfr_direct_gather(int down, int n, int bh, int bw, int sh, int sw, int k, int stride, int pad, const void* src,
                       int src_ld, const void* w, int R, int s_pad, const float* bias, void* y, int y_ld,
                       float* y_nchw, cudaStream_t st) {
  Geo g{n, bh, bw, sh, sw, k, stride, pad};
  const bf16* s = (const bf16*)src;
  const bf16* wp = (const bf16*)w;
  bf16* yo = (bf16*)y;
  long long npix = (long long)n * (down ? sh * sw : bh * bw);
  if ((s_pad & 7) == 0 && (src_ld & 7) == 0) {
    if (R >= 8)
      return down ? launch_gather(gather_down_kernel<8, 8>, g, npix, R, 8, st, s, src_ld, wp, s_pad, bias, yo, y_ld, y_nchw)
                  : launch_gather(gather_up_kernel<8, 8>, g, npix, R, 8, st, s, src_ld, wp, s_pad, bias, yo, y_ld, y_nchw);
    return down ? launch_gather(gather_down_kernel<4, 8>, g, npix, R, 4, st, s, src_ld, wp, s_pad, bias, yo, y_ld, y_nchw)
                : launch_gather(gather_up_kernel<4, 8>, g, npix, R, 4, st, s, src_ld, wp, s_pad, bias, yo, y_ld, y_nchw);
  }
  if ((s_pad & 3) == 0 && (src_ld & 3) == 0) {
    if (R >= 8)
      return down ? launch_gather(gather_down_kernel<8, 4>, g, npix, R, 8, st, s, src_ld, wp, s_pad, bias, yo, y_ld, y_nchw)
                  : launch_gather(gather_up_kernel<8, 4>, g, npix, R, 8, st, s, src_ld, wp, s_pad, bias, yo, y_ld, y_nchw);
    return down ? launch_gather(gather_down_kernel<4, 4>, g, npix, R, 4, st, s, src_ld, wp, s_pad, bias, yo, y_ld, y_nchw)
                : launch_gather(gather_up_kernel<4, 4>, g, npix, R, 4, st, s, src_ld, wp, s_pad, bias, yo, y_ld, y_nchw);
  }
  crfr_set_error("direct conv: source channel padding %d / ld %d must be a multiple of 4", s_pad, src_ld);
  return CRFR_EUNSUPPORTED;
}

int crfr_direct_wgrad(int n, int bh, int bw, int sh, int sw, int k, int stride, int pad, const void* small,
                      int small_ld, int A, const void* big, int big_ld, int B, float* G, void* ws, size_t ws_bytes,
                      cudaStream_t st) {
  if ((big_ld & 3) != 0) {
    crfr_set_error("direct wgrad: big-side ld %d must be a multiple of 4", big_ld);
    return CRFR_EUNSUPPORTED;
  }
  Geo g{n, bh, bw, sh, sw, k, stride, pad};
  long long npix = (long long)n * sh * sw;
  int npairs = A * ((B + 3) / 4);
  int pair_blocks = crfr_cdiv(npairs, kWgThreads * kMaxPairs);
  int T = k * k;
  // enough CTAs to fill the GPU a few times, chunks of >= 256 pixels
  long long want = (148LL * 16) / ((long long)T * pair_blocks) + 1;
  long long chunks = npix / 256 < 1 ? 1 : npix / 256;
  if (chunks > want) chunks = want;
  const long long slice = (long long)A * B * T;
  CRFR_CHECK_ARG(ws && ws_bytes >= sizeof(float) * (size_t)slice, "direct wgrad: workspace %zu < %zu", ws_bytes,
                 sizeof(float) * (size_t)slice);
  chunks = fit_chunks(chunks, slice, ws_bytes);
  int chunk_pix = (int)((npix + chunks - 1) / chunks);
  chunks = (npix + chunk_pix - 1) / chunk_pix;
  wgrad_kernel<<<dim3((unsigned)chunks, T, pair_blocks), kWgThreads, 0, st>>>(g, (const bf16*)small, small_ld, A,
                                                                               (const bf16*)big, big_ld, B,
                                                                               chunk_pix, (float*)ws);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return sum_chunks((const float*)ws, chunks, slice, G, st);
}

int crfr_colsum(const void* t, int ld, int c, long long npix, float* out, void* ws, size_t ws_bytes, cudaStream_t st) {
  CRFR_CHECK_ARG(ws && ws_bytes >= sizeof(float) * (size_t)c, "colsum: workspace %zu < %zu", ws_bytes, sizeof(float) * (size_t)c);
  long long chunks = npix / 512 < 1 ? 1 : npix / 512;
  if (chunks > 148 * 4) chunks = 148 * 4;
  chunks = fit_chunks(chunks, c, ws_bytes);
  int chunk_pix = (int)((npix + chunks - 1) / chunks);
  chunks = (npix + chunk_pix - 1) / chunk_pix;
  const int cb = c < 256 ? c : 256;
  const int lanes = 256 / cb > 0 ? 256 / cb : 1;
  colsum_kernel<<<dim3((unsigned)chunks, (unsigned)((c + 255) / 256)), 256, sizeof(float) * lanes * cb, st>>>(
      (const bf16*)t, ld, c, npix, chunk_pix, (float*)ws);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return sum_chunks((const float*)ws, chunks, c, out, st);
}
