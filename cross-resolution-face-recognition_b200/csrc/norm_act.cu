// InstanceNorm / BatchNorm statistics and the fused normalise + affine + residual + PReLU/ReLU pass, forward and
// backward.  HBM-bound: every pass reads/writes 16-byte (8 x bf16) vectors, one channel-group per thread, so a
// warp touches whole 128-byte lines of the NHWC rows.  Reductions are deterministic: per-chunk partials in a
// workspace, fixed-order finalisation (no float atomics).
//
// ref: nn.InstanceNorm2d + nn.PReLU + torch.add in _Residual_Block (model/FSRnet.py:75-98) and BasicBlock
//      (:105-135); nn.BatchNorm2d + ReLU in model/resnet.py:18-47 (groups: n = 1, hw = N*H*W).
#include <stdlib.h>

#include "common.cuh"
#include "crfr.h"
#include "internal.h"

namespace {

constexpr int kThreads = 256;

__device__ __forceinline__ bf16x8 ld_stream(const bf16* p) {
  uint4 u;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w)
               : "l"(p));
  return *reinterpret_cast<bf16x8*>(&u);
}

struct ChunkPlan {
  int chunks;      // partials per image
  int chunk_pix;   // pixels per chunk
};

inline ChunkPlan plan_chunks(int n, int hw) {
  // The grid is n x chunks CTAs; these passes run 2-4 CTAs per SM.  A grid that is "a little more than a whole
  // number of waves" wastes up to a full wave (measured: 640 CTAs on 296 slots = 2.16 waves -> 72 % efficiency), so
  // pick the chunk count whose CTA total packs best into whole waves for every occupancy in 2..4, among chunk sizes
  // of >= 512 pixels (fewer only when the image is smaller).
  const int sms = 148;
  int maxc = hw / 512;
  if (maxc < 1) maxc = 1;
  if (maxc > 2048) maxc = 2048;
  int best = 1;
  double best_eff = -1.0;
  for (int c = 1; c <= maxc; ++c) {
    const long long ctas = (long long)n * c;
    double eff = 1.0;
    for (int occ = 2; occ <= 4; ++occ) {
      const long long conc = (long long)sms * occ;
      const long long waves = (ctas + conc - 1) / conc;
      const double e = (double)ctas / (double)(waves * conc);
      if (e < eff) eff = e;
    }
    if (eff > best_eff + 1e-9) {
      best_eff = eff;
      best = c;
    }
  }
  int chunk_pix = (hw + best - 1) / best;
  int chunks = (hw + chunk_pix - 1) / chunk_pix;
  return {chunks, chunk_pix};
}

// Reduce K per-thread 8-vectors across the pixel lanes of the CTA and store [K][C] at dst.
template <int K>
__device__ __forceinline__ void cta_reduce_store(float (&acc)[K][8], float* smem, int cg, int lane, int lanes, int c,
                                                 float* dst) {
  // smem layout [K][lanes][C]
#pragma unroll
  for (int k = 0; k < K; ++k)
#pragma unroll
    for (int j = 0; j < 8; ++j) smem[(k * lanes + lane) * c + cg * 8 + j] = acc[k][j];
  __syncthreads();
  for (int i = threadIdx.x; i < K * c; i += kThreads) {
    int k = i / c, ch = i - k * c;
    float s = 0.f;
    for (int l = 0; l < lanes; ++l) s += smem[(k * lanes + l) * c + ch];
    dst[k * c + ch] = s;
  }
}

__global__ void __launch_bounds__(kThreads)
stats_partial_kernel(const bf16* __restrict__ y, int ld, int hw, int c, int chunk_pix, float* __restrict__ partial) {
  extern __shared__ float smem[];
  const int groups = c >> 3, lanes = kThreads / groups;
  const int cg = threadIdx.x % groups, lane = threadIdx.x / groups;
  const int n = blockIdx.y, chunk = blockIdx.x;
  const int p0 = chunk * chunk_pix, p1 = min(hw, p0 + chunk_pix);
  const bf16* base = y + ((long long)n * hw) * ld + cg * 8;
  float acc[2][8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[0][j] = acc[1][j] = 0.f;
  for (int p = p0 + lane; p < p1; p += 4 * lanes) {
    bf16x8 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (p + u * lanes < p1) v[u] = ld_stream(base + (long long)(p + u * lanes) * ld);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (p + u * lanes < p1) {
        float f[8];
        unpack8(v[u], f);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          acc[0][j] += f[j];
          acc[1][j] += f[j] * f[j];
        }
      }
    }
  }
  cta_reduce_store<2>(acc, smem, cg, lane, lanes, c, partial + ((long long)n * gridDim.x + chunk) * 2 * c);
}

// grid (image, slab of 8 channels): 256 threads = 32 chunk lanes x 8 channels; deterministic two-level sum over the
// chunk partials (lane-strided, then lanes in order).  BatchNorm (one group over the whole batch) has hundreds of
// chunks: the slabs keep its finalisation parallel instead of one CTA walking every channel.
__global__ void __launch_bounds__(kThreads)
stats_finalize_kernel(const float* __restrict__ partial, int chunks, int c, float inv_hw, float eps,
                      float* __restrict__ stats) {
  __shared__ float sm[2][kThreads];
  const int n = blockIdx.x, ch = blockIdx.y * 8 + (threadIdx.x & 7), lane = threadIdx.x >> 3;
  const float* p = partial + (long long)n * chunks * 2 * c;
  float s = 0.f, q = 0.f;
  for (int k = lane; k < chunks; k += 32) {
    s += p[(k * 2 + 0) * c + ch];
    q += p[(k * 2 + 1) * c + ch];
  }
  sm[0][threadIdx.x] = s;
  sm[1][threadIdx.x] = q;
  __syncthreads();
  if (threadIdx.x < 8) {
    float ts = 0.f, tq = 0.f;
    for (int l = 0; l < 32; ++l) {
      ts += sm[0][l * 8 + threadIdx.x];
      tq += sm[1][l * 8 + threadIdx.x];
    }
    float mean, rstd;
    crfr_mean_rstd(ts, tq, inv_hw, eps, mean, rstd);
    stats[2 * (n * c + ch)] = mean;
    stats[2 * (n * c + ch) + 1] = rstd;
  }
}

// streaming (evict-first) 16-byte store: the activation is not re-read before ~100 MB of other traffic went by
__device__ __forceinline__ void st_stream(bf16* p, const bf16x8& v) {
  const uint4 u = *reinterpret_cast<const uint4*>(&v);
  asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(u.x), "r"(u.y), "r"(u.z), "r"(u.w) : "memory");
}

// 8 independent 16-byte loads per input in flight per thread and streaming stores: measured 6.0 TB/s against 5.5 TB/s
// for the 4-deep variant with default stores (2 reads + 1 write, 128 images of 64 x 128 x 128)
constexpr int kFwdUnroll = 8;

__global__ void __launch_bounds__(kThreads)
norm_act_fwd_kernel(const bf16* __restrict__ y, int y_ld, const float* __restrict__ stats,
                    const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ alpha,
                    int relu, const bf16* __restrict__ res, int res_ld, bf16* __restrict__ out, int out_ld, int hw,
                    int c, int chunk_pix) {
  const int groups = c >> 3, lanes = kThreads / groups;
  const int cg = threadIdx.x % groups, lane = threadIdx.x / groups;
  const int n = blockIdx.y;
  const int p0 = blockIdx.x * chunk_pix, p1 = min(hw, p0 + chunk_pix);
  float sc[8], sh[8], al[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    int ch = cg * 8 + j;
    float mean = stats[2 * (n * c + ch)], rstd = stats[2 * (n * c + ch) + 1];
    float g = gamma ? gamma[ch] : 1.f, b = beta ? beta[ch] : 0.f;
    sc[j] = g * rstd;
    sh[j] = b - mean * sc[j];
    al[j] = relu ? 0.f : (alpha ? alpha[ch] : 1.f);
  }
  const long long pix0 = (long long)n * hw;
  for (int p = p0 + lane; p < p1; p += kFwdUnroll * lanes) {
    bf16x8 vy[kFwdUnroll], vr[kFwdUnroll];
#pragma unroll
    for (int u = 0; u < kFwdUnroll; ++u) {
      const int pp = p + u * lanes;
      if (pp < p1) {
        vy[u] = ld_stream(y + (pix0 + pp) * y_ld + cg * 8);
        if (res) vr[u] = ld_stream(res + (pix0 + pp) * res_ld + cg * 8);
      }
    }
#pragma unroll
    for (int u = 0; u < kFwdUnroll; ++u) {
      const int pp = p + u * lanes;
      if (pp < p1) {
        float f[8], r[8];
        unpack8(vy[u], f);
        if (res) unpack8(vr[u], r);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float z = fmaf(f[j], sc[j], sh[j]);
          if (res) z += r[j];
          f[j] = z > 0.f ? z : z * al[j];
        }
        st_stream(out + (pix0 + pp) * out_ld + cg * 8, pack8(f));
      }
    }
  }
}

// backward pass 1: dz = dout * act'(z) (stored, bf16), partial sums of dz, dz*xhat, dout*min(z,0)
__global__ void __launch_bounds__(kThreads, 2)
norm_act_bwd_reduce_kernel(const bf16* __restrict__ da, int da_ld, const bf16* __restrict__ db, int db_ld,
                           const bf16* __restrict__ y, int y_ld, const float* __restrict__ stats,
                           const float* __restrict__ gamma, const float* __restrict__ beta,
                           const float* __restrict__ alpha, int relu, const bf16* __restrict__ res, int res_ld,
                           bf16* __restrict__ dz, int dz_ld, int hw, int c, int chunk_pix,
                           float* __restrict__ partial) {
  extern __shared__ float smem[];
  const int groups = c >> 3, lanes = kThreads / groups;
  const int cg = threadIdx.x % groups, lane = threadIdx.x / groups;
  const int n = blockIdx.y, chunk = blockIdx.x;
  const int p0 = chunk * chunk_pix, p1 = min(hw, p0 + chunk_pix);
  const bool act = relu || alpha;
  float mu[8], rs[8], sc[8], sh[8], al[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    int ch = cg * 8 + j;
    mu[j] = stats[2 * (n * c + ch)];
    rs[j] = stats[2 * (n * c + ch) + 1];
    float g = gamma ? gamma[ch] : 1.f, b = beta ? beta[ch] : 0.f;
    sc[j] = g * rs[j];
    sh[j] = b - mu[j] * sc[j];
    al[j] = relu ? 0.f : (alpha ? alpha[ch] : 1.f);
  }
  float acc[3][8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[0][j] = acc[1][j] = acc[2][j] = 0.f;
  const long long pix0 = (long long)n * hw;
  for (int p = p0 + lane; p < p1; p += 2 * lanes) {
    bf16x8 va[2], vb[2], vy[2], vr[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int pp = p + u * lanes;
      if (pp < p1) {
        va[u] = ld_stream(da + (pix0 + pp) * da_ld + cg * 8);
        if (db) vb[u] = ld_stream(db + (pix0 + pp) * db_ld + cg * 8);
        vy[u] = ld_stream(y + (pix0 + pp) * y_ld + cg * 8);
        if (act && res) vr[u] = ld_stream(res + (pix0 + pp) * res_ld + cg * 8);
      }
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int pp = p + u * lanes;
      if (pp < p1) {
        float g[8], f[8], r[8], g2[8];
        unpack8(va[u], g);
        if (db) {
          unpack8(vb[u], g2);
#pragma unroll
          for (int j = 0; j < 8; ++j) g[j] += g2[j];
        }
        unpack8(vy[u], f);
        if (act && res) unpack8(vr[u], r);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float d = g[j];
          if (act) {
            float z = fmaf(f[j], sc[j], sh[j]);
            if (res) z += r[j];
            if (!(z > 0.f)) {
              acc[2][j] += d * z;
              d *= al[j];
            }
          }
          d = bf16_round(d);
          g[j] = d;
          acc[0][j] += d;
          acc[1][j] += d * (f[j] - mu[j]) * rs[j];
        }
        if (dz) *reinterpret_cast<bf16x8*>(dz + (pix0 + pp) * dz_ld + cg * 8) = pack8(g);
      }
    }
  }
  cta_reduce_store<3>(acc, smem, cg, lane, lanes, c, partial + ((long long)n * gridDim.x + chunk) * 3 * c);
}

// grid (image, slab of 8 channels): fold the chunk partials -> bstats[n][ch] = (mean dz, mean dz*xhat); tot[n][3][c]
__global__ void __launch_bounds__(kThreads)
bwd_fold_kernel(const float* __restrict__ partial, int chunks, int c, float inv_hw, float* __restrict__ bstats,
                float* __restrict__ tot) {
  __shared__ float sm[3][kThreads];
  const int n = blockIdx.x, ch = blockIdx.y * 8 + (threadIdx.x & 7), lane = threadIdx.x >> 3;
  const float* p = partial + (long long)n * chunks * 3 * c;
  float s[3] = {0.f, 0.f, 0.f};
  for (int k = lane; k < chunks; k += 32)
#pragma unroll
    for (int j = 0; j < 3; ++j) s[j] += p[(k * 3 + j) * c + ch];
#pragma unroll
  for (int j = 0; j < 3; ++j) sm[j][threadIdx.x] = s[j];
  __syncthreads();
  if (threadIdx.x < 8) {
    float t[3] = {0.f, 0.f, 0.f};
    for (int l = 0; l < 32; ++l)
#pragma unroll
      for (int j = 0; j < 3; ++j) t[j] += sm[j][l * 8 + threadIdx.x];
    const int i = n * c + ch;
    bstats[2 * i] = t[0] * inv_hw;
    bstats[2 * i + 1] = t[1] * inv_hw;
#pragma unroll
    for (int j = 0; j < 3; ++j) tot[(n * 3 + j) * c + ch] = t[j];
  }
}

// backward pass 2: dy = gamma * rstd * (dz - mean(dz) - xhat * mean(dz * xhat)).
// dz == nullptr (layers without a residual branch: nobody else consumes dz): it is not stored by pass 1 but
// recomputed here from dout (da) and y with exactly the same arithmetic and rounding - one map less per layer.
__global__ void __launch_bounds__(kThreads)
norm_act_bwd_apply_kernel(const bf16* __restrict__ dz, int dz_ld, const bf16* __restrict__ y, int y_ld,
                          const float* __restrict__ stats, const float* __restrict__ bstats,
                          const float* __restrict__ gamma, bf16* __restrict__ dy, int dy_ld, int hw, int c,
                          int chunk_pix, const float* __restrict__ tot, int nimg, float* __restrict__ dgamma,
                          float* __restrict__ dbeta, float* __restrict__ dalpha, const bf16* __restrict__ da, int da_ld,
                          const float* __restrict__ beta, const float* __restrict__ alpha, int relu) {
  // CTA (0,0) also folds the per-image totals into the parameter gradients, in fixed order (deterministic)
  if (blockIdx.x == 0 && blockIdx.y == 0 && (dgamma || dbeta || dalpha)) {
    for (int ch = threadIdx.x; ch < c; ch += kThreads) {
      float t0 = 0.f, t1 = 0.f, t2 = 0.f;
      for (int i = 0; i < nimg; ++i) {
        t0 += tot[(i * 3 + 0) * c + ch];
        t1 += tot[(i * 3 + 1) * c + ch];
        t2 += tot[(i * 3 + 2) * c + ch];
      }
      if (dbeta) dbeta[ch] += t0;
      if (dgamma) dgamma[ch] += t1;
      if (dalpha) dalpha[ch] += t2;
    }
  }
  const int groups = c >> 3, lanes = kThreads / groups;
  const int cg = threadIdx.x % groups, lane = threadIdx.x / groups;
  const int n = blockIdx.y;
  const int p0 = blockIdx.x * chunk_pix, p1 = min(hw, p0 + chunk_pix);
  const bool recompute = dz == nullptr;
  const bool act = relu || alpha;
  const bf16* dsrc = recompute ? da : dz;
  const int dsrc_ld = recompute ? da_ld : dz_ld;
  float mu[8], rs[8], gr[8], m1[8], m2[8], bt[8], al[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    int ch = cg * 8 + j;
    mu[j] = stats[2 * (n * c + ch)];
    rs[j] = stats[2 * (n * c + ch) + 1];
    gr[j] = (gamma ? gamma[ch] : 1.f) * rs[j];
    m1[j] = bstats[2 * (n * c + ch)];
    m2[j] = bstats[2 * (n * c + ch) + 1];
    bt[j] = beta ? beta[ch] : 0.f;
    al[j] = relu ? 0.f : (alpha ? alpha[ch] : 1.f);
  }
  const long long pix0 = (long long)n * hw;
  for (int p = p0 + lane; p < p1; p += 4 * lanes) {
    bf16x8 vd[4], vy[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int pp = p + u * lanes;
      if (pp < p1) {
        vd[u] = ld_stream(dsrc + (pix0 + pp) * dsrc_ld + cg * 8);
        vy[u] = ld_stream(y + (pix0 + pp) * y_ld + cg * 8);
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int pp = p + u * lanes;
      if (pp < p1) {
        float d[8], f[8];
        unpack8(vd[u], d);
        unpack8(vy[u], f);
        if (recompute && act) {   // dz = dout * act'(z), z = gamma * xhat + beta written as in pass 1, rounded to bf16
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float z = fmaf(f[j], gr[j], bt[j] - mu[j] * gr[j]);
            if (!(z > 0.f)) d[j] *= al[j];
            d[j] = bf16_round(d[j]);
          }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float xh = (f[j] - mu[j]) * rs[j];
          d[j] = gr[j] * (d[j] - m1[j] - xh * m2[j]);
        }
        *reinterpret_cast<bf16x8*>(dy + (pix0 + pp) * dy_ld + cg * 8) = pack8(d);
      }
    }
  }
}

// implementation of crfr_norm_act_bwd: option norm_bwd_impl 0 = register-staged reduce + fold + apply kernels (below),
// 1 = persistent TMA-fed reduce + fold + apply kernels (norm_stream.cu; default wherever the views are TMA-addressable).

// BatchNorm buffer maintenance (one thread per channel)
__global__ void bn_update_running_kernel(const float* __restrict__ stats, float* __restrict__ rmean,
                                         float* __restrict__ rvar, long long* __restrict__ nbt, int c, float unbias,
                                         float momentum, float eps) {
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch == 0 && nbt) *nbt += 1;
  if (ch >= c) return;
  const float mean = stats[2 * ch], rstd = stats[2 * ch + 1];
  const float var = fmaxf(1.f / (rstd * rstd) - eps, 0.f);
  rmean[ch] = (1.f - momentum) * rmean[ch] + momentum * mean;
  rvar[ch] = (1.f - momentum) * rvar[ch] + momentum * var * unbias;
}

__global__ void bn_running_to_stats_kernel(const float* __restrict__ rmean, const float* __restrict__ rvar, int c,
                                           float eps, float* __restrict__ stats) {
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= c) return;
  stats[2 * ch] = rmean[ch];
  stats[2 * ch + 1] = rsqrtf(rvar[ch] + eps);
}

inline bool channels_ok(int c) { return c >= 8 && c <= 2048 && (c & 7) == 0 && (kThreads % (c >> 3)) == 0; }

}  // namespace

size_t crfr_norm_ws_bytes(int n, int hw, int c) {
  ChunkPlan pl = plan_chunks(n, hw);
  int chunks = pl.chunks;
  if (crfr_norm_stream_parts(n, hw, c) > chunks) chunks = crfr_norm_stream_parts(n, hw, c);
  // partials [n][chunks][3][c] + bstats [n][c][2] + tot [n][3][c]
  return sizeof(float) * ((size_t)n * chunks * 3 * c + (size_t)n * c * 2 + (size_t)n * 3 * c) + 256;
}

// Finalise (mean, rstd) from partials laid out [n][chunks][2][c]; shared with the conv epilogue statistics.
int crfr_norm_finalize(const float* partial, int n, int chunks, int hw, int c, float eps, float* stats,
                       cudaStream_t st) {
  stats_finalize_kernel<<<dim3(n, c / 8), kThreads, 0, st>>>(partial, chunks, c, 1.f / (float)hw, eps, stats);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

extern "C" int crfr_bn_update_running(const float* stats, float* running_mean, float* running_var,
                                      long long* num_batches_tracked, int c, long long count, float momentum,
                                      float eps, void* stream) {
  CRFR_CHECK_ARG(stats && running_mean && running_var && c > 0 && count > 0, "bn_update_running: bad argument");
  const float unbias = count > 1 ? (float)((double)count / (double)(count - 1)) : 1.f;
  bn_update_running_kernel<<<crfr_cdiv(c, 128), 128, 0, (cudaStream_t)stream>>>(stats, running_mean, running_var,
                                                                               num_batches_tracked, c, unbias,
                                                                               momentum, eps);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

extern "C" int crfr_bn_running_to_stats(const float* running_mean, const float* running_var, int c, float eps,
                                        float* stats, void* stream) {
  CRFR_CHECK_ARG(stats && running_mean && running_var && c > 0, "bn_running_to_stats: bad argument");
  bn_running_to_stats_kernel<<<crfr_cdiv(c, 128), 128, 0, (cudaStream_t)stream>>>(running_mean, running_var, c, eps,
                                                                                 stats);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

extern "C" size_t crfr_norm_workspace_bytes(int n, int hw, int c) { return crfr_norm_ws_bytes(n, hw, c); }


extern "C" int crfr_norm_stats(const void* y, int n, int hw, int c, int ld, float eps, float* stats, void* ws,
                               size_t ws_bytes, void* stream) {
  CRFR_CHECK_ARG(y && stats && n > 0 && hw > 0, "norm_stats: bad argument");
  CRFR_CHECK_ARG(channels_ok(c) && ld >= c && (ld & 7) == 0, "norm_stats: unsupported channels %d (ld %d)", c, ld);
  ChunkPlan pl = plan_chunks(n, hw);
  size_t need = sizeof(float) * (size_t)n * pl.chunks * 2 * c;
  if (!ws || ws_bytes < need) {
    crfr_set_error("norm_stats: workspace %zu < %zu", ws_bytes, need);
    return CRFR_EWORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  int lanes = kThreads / (c >> 3);
  size_t smem = sizeof(float) * 2 * lanes * c;
  stats_partial_kernel<<<dim3(pl.chunks, n), kThreads, smem, st>>>((const bf16*)y, ld, hw, c, pl.chunk_pix,
                                                                   (float*)ws);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return crfr_norm_finalize((const float*)ws, n, pl.chunks, hw, c, eps, stats, st);
}

extern "C" int crfr_norm_act_fwd(const void* y, int y_ld, const float* stats, const float* gamma, const float* beta,
                                 const float* alpha, int relu, const void* res, int res_ld, void* out, int out_ld,
                                 int n, int hw, int c, void* stream) {
  CRFR_CHECK_ARG(y && stats && out && n > 0 && hw > 0, "norm_act_fwd: bad argument");
  CRFR_CHECK_ARG(channels_ok(c) && y_ld >= c && out_ld >= c && ((y_ld | out_ld | res_ld) & 7) == 0,
                 "norm_act_fwd: unsupported channels %d", c);
  {
    const void* views[3] = {y, res, out};
    const int lds[3] = {y_ld, res_ld, out_ld};
    if (crfr_opt(CRFR_OPT_NORM_FWD_STREAM) && crfr_norm_stream_supported(c, (long long)n * hw, views, lds, 3))
      return crfr_norm_fwd_stream(y, y_ld, stats, gamma, beta, alpha, relu, res, res_ld, out, out_ld, n, hw, c,
                                  (cudaStream_t)stream);
  }
  ChunkPlan pl = plan_chunks(n, hw);
  norm_act_fwd_kernel<<<dim3(pl.chunks, n), kThreads, 0, (cudaStream_t)stream>>>(
      (const bf16*)y, y_ld, stats, gamma, beta, alpha, relu, (const bf16*)res, res_ld, (bf16*)out, out_ld, hw, c,
      pl.chunk_pix);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

extern "C" int crfr_norm_act_bwd(const void* dout_a, int da_ld, const void* dout_b, int db_ld, const void* y,
                                 int y_ld, const float* stats, const float* gamma, const float* beta,
                                 const float* alpha, int relu, const void* res, int res_ld, void* dz, int dz_ld,
                                 void* dy, int dy_ld, float* dgamma, float* dbeta, float* dalpha, int n, int hw,
                                 int c, void* ws, size_t ws_bytes, void* stream) {
  CRFR_CHECK_ARG(dout_a && y && stats && dy && n > 0 && hw > 0, "norm_act_bwd: bad argument");
  CRFR_CHECK_ARG(dz || (!res && !dout_b), "norm_act_bwd: dz may only be omitted without a residual / second gradient");
  CRFR_CHECK_ARG(channels_ok(c) && ((da_ld | db_ld | y_ld | res_ld | dz_ld | dy_ld) & 7) == 0,
                 "norm_act_bwd: unsupported channels %d", c);
  ChunkPlan pl = plan_chunks(n, hw);
  size_t need = crfr_norm_ws_bytes(n, hw, c);
  if (!ws || ws_bytes < need) {
    crfr_set_error("norm_act_bwd: workspace %zu < %zu", ws_bytes, need);
    return CRFR_EWORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  int lanes = kThreads / (c >> 3);
  const int impl = crfr_opt(CRFR_OPT_NORM_BWD_STREAM);
  const void* views[6] = {dout_a, dout_b, y, res, dz, dy};
  const int lds[6] = {da_ld, db_ld, y_ld, res_ld, dz_ld, dy_ld};
  const bool tma = impl >= 1 && crfr_norm_stream_supported(c, (long long)n * hw, views, lds, 6);
  const int chunks = tma ? crfr_norm_stream_parts(n, hw, c) : pl.chunks;
  float* partial = (float*)ws;
  float* bstats = partial + (size_t)n * chunks * 3 * c;
  float* tot = bstats + (size_t)n * c * 2;
  if (tma) {
    CRFR_TRY(crfr_norm_bwd_reduce_stream(dout_a, da_ld, dout_b, db_ld, y, y_ld, stats, gamma, beta, alpha, relu, res,
                                         res_ld, dz, dz_ld, n, hw, c, partial, st));
  } else {
    size_t smem = sizeof(float) * 3 * lanes * c;
    if (smem > 48 * 1024) {
      CRFR_CUDA(cudaFuncSetAttribute(norm_act_bwd_reduce_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    norm_act_bwd_reduce_kernel<<<dim3(pl.chunks, n), kThreads, smem, st>>>(
        (const bf16*)dout_a, da_ld, (const bf16*)dout_b, db_ld, (const bf16*)y, y_ld, stats, gamma, beta, alpha, relu,
        (const bf16*)res, res_ld, (bf16*)dz, dz_ld, hw, c, pl.chunk_pix, partial);
    CRFR_COUNT_LAUNCH();
    CRFR_LAUNCH_CHECK();
  }
  return crfr_norm_bwd_finish(partial, chunks, dz ? dz : dout_a, dz ? dz_ld : da_ld, dz == nullptr, y, y_ld, stats, gamma,
                              beta, alpha, relu, dy, dy_ld, dgamma, dbeta, dalpha, n, hw, c, bstats, tot, tma ? 1 : 0, st);
}

// Second half of the normalisation backward: fold the first pass' partials [n][chunks][3][c] (wherever that pass ran:
// the reduce kernels above / in norm_stream.cu, or the dgrad epilogue of rowconv2.cu), then the apply pass.
// dsrc = dz, or dout when recompute != 0 (dz is then rebuilt from dout and y with the first pass' arithmetic).
int crfr_norm_bwd_finish(const float* partial, int chunks, const void* dsrc, int dsrc_ld, int recompute, const void* y,
                         int y_ld, const float* stats, const float* gamma, const float* beta, const float* alpha, int relu,
                         void* dy, int dy_ld, float* dgamma, float* dbeta, float* dalpha, int n, int hw, int c,
                         float* bstats, float* tot, int use_stream, cudaStream_t st) {
  // the TMA-fed apply pass folds the partial sums itself where an image has few partial slots (InstanceNorm); with one
  // statistic group over the whole batch (BatchNorm: hundreds of slots) the fold stays a kernel of its own
  const bool fold_inside = use_stream && chunks <= 16;
  if (!fold_inside) {
    bwd_fold_kernel<<<dim3(n, c / 8), kThreads, 0, st>>>(partial, chunks, c, 1.f / (float)hw, bstats, tot);
    CRFR_COUNT_LAUNCH();
    CRFR_LAUNCH_CHECK();
  }
  if (use_stream)
    return crfr_norm_bwd_apply_stream(dsrc, dsrc_ld, recompute, y, y_ld, stats, partial, chunks, fold_inside ? nullptr : bstats,
                                      fold_inside ? nullptr : tot, gamma, beta, alpha, relu, dy, dy_ld, dgamma, dbeta, dalpha, n,
                                      hw, c, st);
  ChunkPlan pl = plan_chunks(n, hw);
  norm_act_bwd_apply_kernel<<<dim3(pl.chunks, n), kThreads, 0, st>>>(
      recompute ? nullptr : (const bf16*)dsrc, dsrc_ld, (const bf16*)y, y_ld, stats, bstats, gamma, (bf16*)dy, dy_ld, hw, c,
      pl.chunk_pix, tot, n, dgamma, dbeta, dalpha, recompute ? (const bf16*)dsrc : nullptr, dsrc_ld, beta, alpha, relu);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}
