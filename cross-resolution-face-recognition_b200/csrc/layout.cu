// Layout conversions at the nn.Module boundary and weight packing.
#include "common.cuh"
#include "crfr.h"
#include "internal.h"

namespace {

__global__ void nchw_to_nhwc_kernel(const float* __restrict__ src, bf16* __restrict__ dst, long long npix, int hw,
                                    int c, int ld, int c_zero_to) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  long long n = i / hw;
  int p = (int)(i - n * hw);
  const float* s = src + n * (long long)c * hw + p;
  bf16* d = dst + i * ld;
  for (int ch = 0; ch < c; ++ch) d[ch] = __float2bfloat16_rn(s[(long long)ch * hw]);
  for (int ch = c; ch < c_zero_to; ++ch) d[ch] = __float2bfloat16_rn(0.f);
}

__global__ void nhwc_to_nchw_kernel(const bf16* __restrict__ src, float* __restrict__ dst, long long npix, int hw,
                                    int c, int ld) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npix) return;
  long long n = i / hw;
  int p = (int)(i - n * hw);
  const bf16* s = src + i * ld;
  float* d = dst + n * (long long)c * hw + p;
  for (int ch = 0; ch < c; ++ch) d[(long long)ch * hw] = __bfloat162float(s[ch]);
}

// Tiled transposes for feature maps (c >= 32): a 32 pixel x 32 channel tile goes through shared memory so that both the
// fp32 NCHW side (contiguous along pixels) and the bf16 NHWC side (contiguous along channels) are accessed in whole
// lines.  The per-pixel kernels above walk the channels with a stride of hw floats on one side and 2-byte stores on the
// other (190 us for a [256, 64, 56, 56] map); they remain for the 3-channel images.
__global__ void __launch_bounds__(256)
nchw_to_nhwc_tiled_kernel(const float* __restrict__ src, bf16* __restrict__ dst, int hw, int c, int ld, int c_zero_to) {
  __shared__ float tile[32][33];
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const long long n = blockIdx.z;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int ch = c0 + ty + 8 * k, p = p0 + tx;
    tile[ty + 8 * k][tx] = (ch < c && p < hw) ? src[(n * c + ch) * hw + p] : 0.f;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int p = p0 + ty + 8 * k, ch = c0 + tx;
    if (p < hw && ch < c_zero_to) dst[(n * hw + p) * ld + ch] = __float2bfloat16_rn(tile[tx][ty + 8 * k]);
  }
}

__global__ void __launch_bounds__(256)
nhwc_to_nchw_tiled_kernel(const bf16* __restrict__ src, float* __restrict__ dst, int hw, int c, int ld) {
  __shared__ float tile[32][33];
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const long long n = blockIdx.z;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int p = p0 + ty + 8 * k, ch = c0 + tx;
    tile[ty + 8 * k][tx] = (p < hw && ch < c) ? __bfloat162float(src[(n * hw + p) * ld + ch]) : 0.f;
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int ch = c0 + ty + 8 * k, p = p0 + tx;
    if (ch < c && p < hw) dst[(n * c + ch) * hw + p] = tile[tx][ty + 8 * k];
  }
}

__global__ void pack_weight_kernel(const float* __restrict__ src, bf16* __restrict__ dst, int T, int R, int S,
                                   int s_pad, long long rs, long long ss, long long ts) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = (long long)T * R * s_pad;
  if (i >= total) return;
  int s = (int)(i % s_pad);
  long long q = i / s_pad;
  int r = (int)(q % R);
  int t = (int)(q / R);
  float v = (s < S) ? src[r * rs + s * ss + t * ts] : 0.f;
  dst[i] = __float2bfloat16_rn(v);
}

// every job of a batch in one launch: block -> job through the (ascending) first-block table in the kernel parameters
__global__ void pack_weight_batch_kernel(const __grid_constant__ crfr_pack_batch b) {
  int lo = 0, hi = b.njobs - 1;   // largest job whose first block is <= blockIdx.x (binary search: the table is sorted)
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if ((int)blockIdx.x >= b.job[mid].block0) lo = mid;
    else hi = mid - 1;
  }
  const crfr_pack_job& J = b.job[lo];
  const long long i = (long long)((int)blockIdx.x - J.block0) * 256 + threadIdx.x;
  if (i >= (long long)J.T * J.R * J.s_pad) return;
  const int s = (int)(i % J.s_pad);
  const long long q = i / J.s_pad;
  const int r = (int)(q % J.R), t = (int)(q / J.R);
  float v = 0.f;
  if (s < J.S) {
    v = J.src[r * J.rs + s * J.ss + t];
    if (J.rscale) v *= J.rscale[r];
    if (J.sscale) v *= J.sscale[s];
  }
  reinterpret_cast<bf16*>(J.dst)[i] = __float2bfloat16_rn(v);
}

}  // namespace

// internal.h: the weight packs of a whole network program (one per convolution and direction, ~120 per FSRNet step)
// as ceil(n / 64) launches instead of n
int crfr_pack_weight_batch(const crfr_pack_job* jobs, int n, cudaStream_t st) {
  for (int first = 0; first < n; first += CRFR_PACK_BATCH) {
    crfr_pack_batch b;
    b.njobs = n - first < CRFR_PACK_BATCH ? n - first : CRFR_PACK_BATCH;
    int blocks = 0;
    for (int k = 0; k < b.njobs; ++k) {
      b.job[k] = jobs[first + k];
      b.job[k].block0 = blocks;
      blocks += crfr_cdiv((long long)b.job[k].T * b.job[k].R * b.job[k].s_pad, 256);
    }
    pack_weight_batch_kernel<<<blocks, 256, 0, st>>>(b);
    CRFR_COUNT_LAUNCH();
    CRFR_LAUNCH_CHECK();
  }
  return CRFR_OK;
}

extern "C" int crfr_nchw_f32_to_nhwc_bf16(const float* src, void* dst, int n, int c, int h, int w, int dst_ld,
                                          int c_zero_to, void* stream) {
  CRFR_CHECK_ARG(src && dst && n > 0 && c > 0 && h > 0 && w > 0, "nchw_to_nhwc: bad argument");
  CRFR_CHECK_ARG(dst_ld >= c && c_zero_to <= dst_ld, "nchw_to_nhwc: ld %d < c %d", dst_ld, c);
  long long npix = (long long)n * h * w;
  if (c >= 32 && n <= 65535) {
    const int cz = c_zero_to > c ? c_zero_to : c;
    nchw_to_nhwc_tiled_kernel<<<dim3(crfr_cdiv(h * w, 32), crfr_cdiv(cz, 32), n), 256, 0, (cudaStream_t)stream>>>(
        src, (bf16*)dst, h * w, c, dst_ld, cz);
    CRFR_COUNT_LAUNCH();
    CRFR_LAUNCH_CHECK();
    return CRFR_OK;
  }
  nchw_to_nhwc_kernel<<<crfr_cdiv(npix, 256), 256, 0, (cudaStream_t)stream>>>(src, (bf16*)dst, npix, h * w, c,
                                                                              dst_ld, c_zero_to);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

extern "C" int crfr_nhwc_bf16_to_nchw_f32(const void* src, float* dst, int n, int c, int h, int w, int src_ld,
                                          void* stream) {
  CRFR_CHECK_ARG(src && dst && n > 0 && c > 0 && h > 0 && w > 0 && src_ld >= c, "nhwc_to_nchw: bad argument");
  long long npix = (long long)n * h * w;
  if (c >= 32 && n <= 65535) {
    nhwc_to_nchw_tiled_kernel<<<dim3(crfr_cdiv(h * w, 32), crfr_cdiv(c, 32), n), 256, 0, (cudaStream_t)stream>>>(
        (const bf16*)src, dst, h * w, c, src_ld);
    CRFR_COUNT_LAUNCH();
    CRFR_LAUNCH_CHECK();
    return CRFR_OK;
  }
  nhwc_to_nchw_kernel<<<crfr_cdiv(npix, 256), 256, 0, (cudaStream_t)stream>>>((const bf16*)src, dst, npix, h * w, c,
                                                                              src_ld);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

extern "C" int crfr_pack_weight(const float* src, void* dst, int T, int R, int S, int s_pad, long long r_stride,
                                long long s_stride, long long t_stride, void* stream) {
  CRFR_CHECK_ARG(src && dst && T > 0 && R > 0 && S > 0 && s_pad >= S, "pack_weight: bad argument");
  long long total = (long long)T * R * s_pad;
  pack_weight_kernel<<<crfr_cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(src, (bf16*)dst, T, R, S, s_pad,
                                                                              r_stride, s_stride, t_stride);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}
