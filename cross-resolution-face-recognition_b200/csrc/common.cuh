// Shared device/host helpers for the CRFR sm_100a kernels.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

typedef __nv_bfloat16 bf16;

// ------------------------------------------------------------------------------------------------
// error plumbing (C-ABI convention: int return, message through crfr_last_error())
// ------------------------------------------------------------------------------------------------
extern "C" const char* crfr_last_error(void);
void crfr_set_error(const char* fmt, ...);

#define CRFR_OK 0
#define CRFR_EINVAL 1
#define CRFR_ECUDA 2
#define CRFR_EWORKSPACE 3
#define CRFR_EUNSUPPORTED 4

#define CRFR_CHECK_ARG(cond, ...)                                                   \
  do {                                                                              \
    if (!(cond)) {                                                                  \
      crfr_set_error(__VA_ARGS__);                                                  \
      return CRFR_EINVAL;                                                           \
    }                                                                               \
  } while (0)

#define CRFR_CUDA(call)                                                             \
  do {                                                                              \
    cudaError_t e__ = (call);                                                       \
    if (e__ != cudaSuccess) {                                                       \
      crfr_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
      return CRFR_ECUDA;                                                            \
    }                                                                               \
  } while (0)

#define CRFR_LAUNCH_CHECK() CRFR_CUDA(cudaGetLastError())

#define CRFR_TRY(call)                                                              \
  do {                                                                              \
    int rc__ = (call);                                                              \
    if (rc__ != CRFR_OK) return rc__;                                               \
  } while (0)

static inline int crfr_cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// launch counter (bench.py reports gpu_launches from this)
extern unsigned long long g_crfr_launches;
#define CRFR_COUNT_LAUNCH() (++g_crfr_launches)

// ------------------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------------------
#ifdef __CUDACC__
struct alignas(16) bf16x8 { __nv_bfloat162 v[4]; };
struct alignas(8) bf16x4 { __nv_bfloat162 v[2]; };

__device__ __forceinline__ void unpack8(const bf16x8& p, float* f) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __bfloat1622float2(p.v[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ bf16x8 pack8(const float* f) {
  bf16x8 p;
#pragma unroll
  for (int i = 0; i < 4; ++i) p.v[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  return p;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }
// (mean, rstd) from the sums of x and x^2 over hw samples.  Explicitly rounded operations: the kernels that finalise
// statistics (stats_finalize_kernel, the forward pass of norm_stream.cu) must agree bit for bit, whatever the compiler
// would contract into an FMA in each of them.
__device__ __forceinline__ void crfr_mean_rstd(float sum, float sumsq, float inv_hw, float eps, float& mean, float& rstd) {
  mean = __fmul_rn(sum, inv_hw);
  const float var = fmaxf(__fsub_rn(__fmul_rn(sumsq, inv_hw), __fmul_rn(mean, mean)), 0.f);
  rstd = rsqrtf(__fadd_rn(var, eps));
}
#endif
