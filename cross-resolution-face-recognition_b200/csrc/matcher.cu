// Eval matcher: cosine-similarity identification (bf16 tcgen05 GEMM with the top-k fused into the TMEM epilogue, so
// the [probes x gallery] score matrix is never materialised) and squared-L2 threshold verification.
//
// One CTA owns a tile of 128 probes (A operand, resident in smem for the CTA's lifetime: 128 x dim bf16) and walks a
// contiguous range of gallery blocks of 256 rows (B operand, streamed by TMA through a 4-stage ring; N = 256 MMAs:
// the A-operand fetch is paid once per 256 columns, which keeps the shared-memory port below saturation).  Scores
// accumulate in TMEM (two 256-column accumulators = all 512 columns, double buffered) and the 4 epilogue warps - one
// thread per probe row - drain them with tcgen05.ld and keep a register-resident sorted top-8 per probe.  The drain
// is written for a small instruction footprint: 8 scores are compared against the current 8th-best through one
// running maximum, and the insertion network is only entered for a group that contains a candidate (measured: the
// fully unrolled per-score insertion was 173 KB of SASS and instruction-fetch bound at 100 TFLOP/s).  Per-split
// results are merged by crfr_topk_merge (also used for gallery-sharded multi-GPU matching).
//
// ref: utils/eval.py:6-19 (accuracy -> output.topk(maxk, 1, True, True)), utils/utils.py:14-24,41-43 (threshold on
//      squared L2), DISTILLATION/model/model_irse.py:16-20 (l2_norm).
#include <cudaTypedefs.h>
#include <math.h>

#include "common.cuh"
#include "crfr.h"
#include "internal.h"
#include "sm100.cuh"

using namespace sm100;

namespace {

constexpr int kTopK = 8;        // register-resident candidates per probe
constexpr int kThreads = 192;   // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue
constexpr int kStages = 3;     // 3 x 32 KB gallery stages + 128 KB of resident probes fill the 227 KB of shared memory at dim 512
constexpr int kTile = 128 * 128;  // 16 KB: 128 rows x 64 bf16 (probe tile per K chunk)
constexpr int kGBlock = 256;      // gallery rows per MMA (N)
constexpr int kBTile = kGBlock * 128;  // 32 KB: 256 rows x 64 bf16

int make_rows_map(CUtensorMap* m, const void* ptr, long long rows, int dim, int box_rows) {
  const unsigned long long dims[2] = {(unsigned long long)dim, (unsigned long long)rows};
  const unsigned long long strides[1] = {(unsigned long long)dim * 2};
  const unsigned int box[2] = {64, (unsigned int)box_rows};
  return crfr_tmap_encode_bf16(m, ptr, 2, dims, strides, box, "embedding rows");
}

// ---- cluster primitives (CL form of the kernel)
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load whose box lands at the same shared-memory offset in every CTA of `mask` and signals the barrier at the same
// offset in each of them
__device__ __forceinline__ void tma_load_2d_multicast(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], "
      "[%2], %5;" ::"r"(smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(mask)
      : "memory");
}
// arrives on the barrier at this shared-memory offset in every CTA of `mask` once the MMAs issued so far have completed
__device__ __forceinline__ void umma_commit_multicast(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(mask)
               : "memory");
}

struct TopK {
  float v[kTopK];
  int i[kTopK];
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int j = 0; j < kTopK; ++j) {
      v[j] = -INFINITY;
      i[j] = -1;
    }
  }
  // candidates arrive in increasing index order; strict '>' keeps the lowest index first among equal scores
  __device__ __forceinline__ void push(float x, int idx) {
    if (x > v[kTopK - 1]) {
      v[kTopK - 1] = x;
      i[kTopK - 1] = idx;
#pragma unroll
      for (int j = kTopK - 1; j > 0; --j) {
        if (v[j] > v[j - 1]) {
          float tv = v[j]; v[j] = v[j - 1]; v[j - 1] = tv;
          int ti = i[j]; i[j] = i[j - 1]; i[j - 1] = ti;
        }
      }
    }
  }
};

struct MatchParams {
  int p;               // probes
  long long g;         // gallery rows
  int kchunks;         // dim / 64
  int nblocks;         // gallery blocks of kGBlock rows
  int blocks_per_split;
  int index_base;
  float* out_val;      // [splits][p][kTopK]
  int* out_idx;
};

// CL: clusters of two CTAs (two probe tiles, the same gallery range).  The TMA unit issues one request per 128-byte row of a
// box, and a K step of this kernel asks for 256 gallery rows per 4 MMAs of 128 cycles: the request rate, not the tensor pipe,
// bounded the single-CTA form at 0.62 of the bf16 peak.  In a cluster each CTA fetches HALF of every gallery block and
// multicasts it into both shared memories (tmG then has a box of 128 rows); a ring stage is free again when both CTAs'
// MMAs have consumed it (multicast tcgen05.commit on a barrier of count 2).
template <bool CL>
__global__ void __launch_bounds__(kThreads, 1)
cosine_topk_kernel(const __grid_constant__ CUtensorMap tmP, const __grid_constant__ CUtensorMap tmG, MatchParams mp) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = base;                                 // kchunks x 16 KB
  uint8_t* sB = base + mp.kchunks * kTile;            // kStages x 32 KB
  uint64_t* full = (uint64_t*)(sB + kStages * kBTile);
  uint64_t* empty = full + kStages;
  uint64_t* a_full = empty + kStages;
  uint64_t* acc_full = a_full + 1;    // [2]
  uint64_t* acc_empty = acc_full + 2; // [2]
  uint32_t* tmem_slot = (uint32_t*)(acc_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], CL ? 2 : 1);
    }
    mbar_init(a_full, 1);
    for (int b = 0; b < 2; ++b) {
      mbar_init(&acc_full[b], 1);
      mbar_init(&acc_empty[b], 4);  // one arrive per epilogue warp
    }
    fence_barrier_init();
    prefetch_tmap(&tmP);
    prefetch_tmap(&tmG);
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  if (CL) cluster_sync_all();   // the peer's barriers are initialised before anything is multicast to them
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const uint32_t crank = CL ? cluster_ctarank() : 0u;

  const int ptile = blockIdx.x, split = blockIdx.y;
  const int blk0 = split * mp.blocks_per_split;
  const int blk1 = min(mp.nblocks, blk0 + mp.blocks_per_split);
  const int nblk = max(0, blk1 - blk0);
  const int kch = mp.kchunks;

  if (warp == 0) {
    const bool leader = elect_one();
    if (leader) {
      mbar_expect_tx(a_full, (uint32_t)kch * kTile);
      for (int kc = 0; kc < kch; ++kc) tma_load_2d(sA + kc * kTile, &tmP, a_full, kc * 64, ptile * 128);
    }
    int it = 0;
    for (int b = 0; b < nblk; ++b)
      for (int kc = 0; kc < kch; ++kc, ++it) {
        const int s = it % kStages;
        mbar_wait(&empty[s], ((it / kStages) & 1) ^ 1);
        if (leader) {
          mbar_expect_tx(&full[s], kBTile);
          if (CL)   // this CTA's half of the block's rows, into both CTAs of the cluster
            tma_load_2d_multicast(sB + s * kBTile + crank * (kBTile / 2), &tmG, &full[s], kc * 64,
                                  (blk0 + b) * kGBlock + (int)crank * (kGBlock / 2), (uint16_t)3);
          else
            tma_load_2d(sB + s * kBTile, &tmG, &full[s], kc * 64, (blk0 + b) * kGBlock);
        }
      }
  } else if (warp == 1) {
    const bool leader = elect_one();
    const uint32_t idesc = make_idesc_bf16(128, kGBlock, 0, 0);
    const uint64_t adesc0 = make_smem_desc_sw128(smem_u32(sA), 16, 1024);
    const uint64_t bdesc0 = make_smem_desc_sw128(smem_u32(sB), 16, 1024);
    mbar_wait(a_full, 0);
    int it = 0;
    for (int b = 0; b < nblk; ++b) {
      const int buf = b & 1;
      mbar_wait(&acc_empty[buf], ((b >> 1) & 1) ^ 1);
      tc_fence_after();
      for (int kc = 0; kc < kch; ++kc, ++it) {
        const int s = it % kStages;
        mbar_wait(&full[s], (it / kStages) & 1);
        tc_fence_after();
        const uint64_t da = adesc0 + (uint64_t)((kc * kTile) >> 4), db = bdesc0 + (uint64_t)((s * kBTile) >> 4);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (leader) umma_bf16(tmem + buf * kGBlock, da + 2 * k, db + 2 * k, idesc, (uint32_t)((kc | k) != 0));
        if (leader) {
          if (CL) umma_commit_multicast(&empty[s], (uint16_t)3);   // frees the stage in both CTAs
          else umma_commit(&empty[s]);
        }
        __syncwarp();
      }
      if (leader) umma_commit(&acc_full[buf]);
      __syncwarp();
    }
  } else {
    const int q = warp & 3;
    const int row = ptile * 128 + q * 32 + lane;
    TopK top;
    top.init();
    for (int b = 0; b < nblk; ++b) {
      const int buf = b & 1;
      mbar_wait(&acc_full[buf], (b >> 1) & 1);
      tc_fence_after();
      const long long col0 = (long long)(blk0 + b) * kGBlock;
      const int valid = (int)min((long long)kGBlock, mp.g - col0);   // columns past the end of the gallery are masked
#pragma unroll 1
      for (int c0 = 0; c0 < kGBlock; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + buf * kGBlock + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int g8 = 0; g8 < 32; g8 += 8) {
          float x[8];
          float m = -INFINITY;
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            x[e] = (c0 + g8 + e < valid) ? __uint_as_float(v[g8 + e]) : -INFINITY;
            m = fmaxf(m, x[e]);
          }
          if (m > top.v[kTopK - 1]) {   // rare after the first few blocks: one compare per 8 scores on the hot path
#pragma unroll
            for (int e = 0; e < 8; ++e) top.push(x[e], (int)(col0 + c0 + g8 + e) + mp.index_base);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[buf]);
    }
    if (row < mp.p) {
      float* ov = mp.out_val + ((long long)split * mp.p + row) * kTopK;
      int* oi = mp.out_idx + ((long long)split * mp.p + row) * kTopK;
#pragma unroll
      for (int j = 0; j < kTopK; ++j) {
        ov[j] = top.v[j];
        oi[j] = top.i[j];
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (CL) cluster_sync_all();   // nobody leaves while the peer may still multicast into this CTA or arrive on its barriers
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem);
  }
}

// merge `parts` sorted candidate lists of width kin per probe into the top kout (ties: lowest index first)
__global__ void topk_merge_kernel(const float* __restrict__ vals, const int* __restrict__ idx, int parts, int p,
                                  int kin, int kout, float* __restrict__ out_val, int* __restrict__ out_idx) {
  int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= p) return;
  TopK top;
  top.init();
  for (int s = 0; s < parts; ++s) {
    const float* v = vals + ((long long)s * p + r) * kin;
    const int* ix = idx + ((long long)s * p + r) * kin;
    for (int j = 0; j < kin; ++j) {
      float x = v[j];
      int id = ix[j];
      if (id < 0) continue;
      // general merge: equal scores must be ordered by index, parts may arrive in any index order
      if (x > top.v[kTopK - 1] || (x == top.v[kTopK - 1] && id < top.i[kTopK - 1])) {
        top.v[kTopK - 1] = x;
        top.i[kTopK - 1] = id;
#pragma unroll
        for (int t = kTopK - 1; t > 0; --t) {
          bool ahead = top.v[t] > top.v[t - 1] || (top.v[t] == top.v[t - 1] && top.i[t] < top.i[t - 1] && top.i[t] >= 0);
          if (ahead) {
            float tv = top.v[t]; top.v[t] = top.v[t - 1]; top.v[t - 1] = tv;
            int ti = top.i[t]; top.i[t] = top.i[t - 1]; top.i[t - 1] = ti;
          }
        }
      }
    }
  }
  for (int j = 0; j < kout; ++j) {
    out_val[(long long)r * kout + j] = top.v[j];
    out_idx[(long long)r * kout + j] = top.i[j];
  }
}

__global__ void l2norm_kernel(const float* __restrict__ x, bf16* __restrict__ out, long long rows, int dim) {
  long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* s = x + r * dim;
  float acc = 0.f;
  for (int i = lane; i < dim; i += 32) acc += s[i] * s[i];
  acc = warp_sum(acc);
  float inv = 1.f / sqrtf(acc);
  for (int i = lane; i < dim; i += 32) out[r * dim + i] = __float2bfloat16_rn(s[i] * inv);
}

__global__ void pair_verify_kernel(const float* __restrict__ e1, const float* __restrict__ e2, long long pairs, int dim,
                                   float thr, float* __restrict__ dist, uint8_t* __restrict__ same) {
  long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (r >= pairs) return;
  float acc = 0.f;
  for (int i = lane; i < dim; i += 32) {
    float d = e1[r * dim + i] - e2[r * dim + i];
    acc += d * d;
  }
  acc = warp_sum(acc);
  if (lane == 0) {
    if (dist) dist[r] = acc;
    if (same) same[r] = acc < thr ? 1 : 0;
  }
}

// top-k of each row of a materialised score matrix (the drop-in for output.topk at utils/eval.py:11): one warp per
// row, each lane keeps a sorted top-8 of its strided columns, lane lists are merged through shared memory.
__global__ void __launch_bounds__(128)
topk_rows_kernel(const float* __restrict__ scores, int p, long long g, int k, float* __restrict__ out_val,
                 int* __restrict__ out_idx) {
  __shared__ float sv[4][32 * kTopK];
  __shared__ int si[4][32 * kTopK];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * 4 + w;
  if (row >= p) return;
  TopK top;
  top.init();
  const float* s = scores + (long long)row * g;
  for (long long c = lane; c < g; c += 32) top.push(s[c], (int)c);
#pragma unroll
  for (int j = 0; j < kTopK; ++j) {
    sv[w][lane * kTopK + j] = top.v[j];
    si[w][lane * kTopK + j] = top.i[j];
  }
  __syncwarp();
  if (lane == 0) {
    TopK m;
    m.init();
    for (int c = 0; c < 32 * kTopK; ++c) {
      float x = sv[w][c];
      int id = si[w][c];
      if (id < 0) continue;
      if (x > m.v[kTopK - 1] || (x == m.v[kTopK - 1] && id < m.i[kTopK - 1])) {
        m.v[kTopK - 1] = x;
        m.i[kTopK - 1] = id;
#pragma unroll
        for (int t = kTopK - 1; t > 0; --t) {
          bool ahead = m.v[t] > m.v[t - 1] || (m.v[t] == m.v[t - 1] && m.i[t] < m.i[t - 1] && m.i[t] >= 0);
          if (ahead) {
            float tv = m.v[t]; m.v[t] = m.v[t - 1]; m.v[t - 1] = tv;
            int ti = m.i[t]; m.i[t] = m.i[t - 1]; m.i[t - 1] = ti;
          }
        }
      }
    }
    for (int j = 0; j < k; ++j) {
      out_val[(long long)row * k + j] = m.v[j];
      out_idx[(long long)row * k + j] = m.i[j];
    }
  }
}

// counts[0..3] = tp, fp, tn, fn of (dist < thr) against issame (utils/utils.py:14-24)
__global__ void verify_counts_kernel(const float* __restrict__ dist, const uint8_t* __restrict__ issame, long long n,
                                     float thr, unsigned long long* __restrict__ counts) {
  unsigned int c[4] = {0, 0, 0, 0};
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    bool pred = dist[i] < thr, same = issame[i] != 0;
    c[pred ? (same ? 0 : 1) : (same ? 3 : 2)]++;
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    unsigned int v = c[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(&counts[j], (unsigned long long)v);
  }
}

// Threshold sweep of the verification protocol: counts[t][0..3] = tp, fp, tn, fn of (dist < thr[t]) vs issame, restricted
// to the pairs listed in `subset` (a K-fold train or test split; NULL = all pairs).  One thread per threshold; the pair
// data is staged through shared memory in tiles so that every block streams it once.
__global__ void __launch_bounds__(256)
verify_sweep_kernel(const float* __restrict__ dist, const uint8_t* __restrict__ issame, const int* __restrict__ subset,
                    int n, const float* __restrict__ thr, int nthr, unsigned int* __restrict__ counts) {
  __shared__ float sd[1024];
  __shared__ uint8_t ss[1024];
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const float th = t < nthr ? thr[t] : 0.f;
  unsigned int c[4] = {0u, 0u, 0u, 0u};
  for (int base = 0; base < n; base += 1024) {
    const int m = min(1024, n - base);
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
      const int src = subset ? subset[base + i] : base + i;
      sd[i] = dist[src];
      ss[i] = issame[src];
    }
    __syncthreads();
    for (int i = 0; i < m; ++i) {
      const bool pred = sd[i] < th, same = ss[i] != 0;
      c[pred ? (same ? 0 : 1) : (same ? 3 : 2)]++;
    }
    __syncthreads();
  }
  if (t < nthr)
    for (int j = 0; j < 4; ++j) counts[4 * t + j] = c[j];
}

struct SplitPlan {
  int tiles, nblocks, splits, blocks_per_split;
};
SplitPlan plan_splits(int p, long long g) {
  SplitPlan s;
  s.tiles = (p + 127) / 128;
  s.nblocks = (int)((g + kGBlock - 1) / kGBlock);
  // One CTA per SM at a time: the launch runs in waves of `sms` CTAs and costs waves x (blocks per split + the probe-tile load,
  // about 4 blocks' worth).  Pick the split count that minimises it: 10 k probes x 1 M rows = 79 (80 in clusters) tiles - 15
  // splits are 1 185 CTAs = 8.007 waves, i.e. NINE waves of 261 blocks; 13 splits are 7 waves of 301 (-10 %).
  const int sms = crfr_sm_count();
  const int tiles_eff = s.tiles >= 2 ? ((s.tiles + 1) & ~1) : s.tiles;   // clusters of two probe tiles
  int best = 1;
  long long best_cost = -1;
  for (int want = 1; want <= 64 && want <= s.nblocks; ++want) {
    const int bps = (s.nblocks + want - 1) / want;
    const int splits = (s.nblocks + bps - 1) / bps;
    const long long waves = ((long long)tiles_eff * splits + sms - 1) / sms;
    const long long cost = waves * (bps + 4);
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = want; }
  }
  s.blocks_per_split = (s.nblocks + best - 1) / best;
  s.splits = (s.nblocks + s.blocks_per_split - 1) / s.blocks_per_split;
  return s;
}

}  // namespace

extern "C" size_t crfr_cosine_topk_workspace_bytes(int p, long long g, int dim, int k) {
  (void)dim; (void)k;
  if (p <= 0 || g <= 0) return 0;
  SplitPlan s = plan_splits(p, g);
  return (size_t)s.splits * p * kTopK * (sizeof(float) + sizeof(int)) + 256;
}

extern "C" int crfr_topk_merge(const float* vals, const int* idx, int parts, int p, int k, float* out_val,
                               int* out_idx, void* stream) {
  CRFR_CHECK_ARG(vals && idx && out_val && out_idx && parts > 0 && p > 0 && k > 0 && k <= kTopK, "topk_merge: bad argument");
  topk_merge_kernel<<<crfr_cdiv(p, 128), 128, 0, (cudaStream_t)stream>>>(vals, idx, parts, p, k, k, out_val, out_idx);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

extern "C" int crfr_cosine_topk(int engine, const void* probes, const void* gallery, int p, long long g, int dim, int k,
                                int index_base, float* top_val, int* top_idx, void* ws, size_t ws_bytes,
                                void* stream) {
  (void)engine;
  CRFR_CHECK_ARG(probes && gallery && top_val && top_idx && p > 0 && g > 0, "cosine_topk: bad argument");
  CRFR_CHECK_ARG(k >= 1 && k <= kTopK, "cosine_topk: k must be in [1, %d]", kTopK);
  CRFR_CHECK_ARG(dim % 64 == 0 && dim >= 64 && dim <= 512, "cosine_topk: dim %d must be a multiple of 64, <= 512", dim);
  CRFR_CHECK_ARG(g + index_base < 2147483647LL, "cosine_topk: gallery indices must fit int32");
  CRFR_CHECK_ARG((((uintptr_t)probes | (uintptr_t)gallery) & 15) == 0, "cosine_topk: pointers must be 16B aligned");
  SplitPlan s = plan_splits(p, g);
  size_t need = crfr_cosine_topk_workspace_bytes(p, g, dim, k);
  if (!ws || ws_bytes < need) {
    crfr_set_error("cosine_topk: workspace %zu < %zu", ws_bytes, need);
    return CRFR_EWORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const bool cl = s.tiles >= 2;
  CUtensorMap tmP, tmG;
  CRFR_TRY(make_rows_map(&tmP, probes, p, dim, 128));
  CRFR_TRY(make_rows_map(&tmG, gallery, g, dim, cl ? kGBlock / 2 : kGBlock));
  MatchParams mp;
  mp.p = p; mp.g = g; mp.kchunks = dim / 64; mp.nblocks = s.nblocks; mp.blocks_per_split = s.blocks_per_split;
  mp.index_base = index_base;
  mp.out_val = (float*)ws;
  mp.out_idx = (int*)((float*)ws + (size_t)s.splits * p * kTopK);
  const int smem = mp.kchunks * kTile + kStages * kBTile + 1024 + 256;
  // the dynamic shared-memory size depends on the embedding width: raise the per-device limit to the hardware maximum once
  static std::atomic<unsigned long long> attr_done{0}, attr_done_cl{0};
  CRFR_CUDA((cudaError_t)crfr_smem_attr(cosine_topk_kernel<false>, 232448, attr_done));
  CRFR_CUDA((cudaError_t)crfr_smem_attr(cosine_topk_kernel<true>, 232448, attr_done_cl));
  if (cl) {   // clusters of two probe tiles (an odd tile count gets one tile of padding: its probes do not exist, nothing is written)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((s.tiles + 1) & ~1, s.splits);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    CRFR_CUDA(cudaLaunchKernelEx(&cfg, cosine_topk_kernel<true>, tmP, tmG, mp));
  } else {
    cosine_topk_kernel<false><<<dim3(s.tiles, s.splits), kThreads, smem, st>>>(tmP, tmG, mp);
  }
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  topk_merge_kernel<<<crfr_cdiv(p, 128), 128, 0, st>>>(mp.out_val, mp.out_idx, s.splits, p, kTopK, k, top_val, top_idx);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

extern "C" int crfr_topk_rows(const float* scores, int p, long long g, int k, float* out_val, int* out_idx,
                              void* stream) {
  CRFR_CHECK_ARG(scores && out_val && out_idx && p > 0 && g > 0 && k >= 1 && k <= kTopK, "topk_rows: bad argument (k <= %d)", kTopK);
  topk_rows_kernel<<<crfr_cdiv(p, 4), 128, 0, (cudaStream_t)stream>>>(scores, p, g, k, out_val, out_idx);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

extern "C" int crfr_verify_counts(const float* dist, const uint8_t* issame, long long n, float thr,
                                  unsigned long long* counts, void* stream) {
  CRFR_CHECK_ARG(dist && issame && counts && n > 0, "verify_counts: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  CRFR_CUDA(cudaMemsetAsync(counts, 0, 4 * sizeof(unsigned long long), st));
  long long blocks = (n + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  verify_counts_kernel<<<(unsigned)blocks, 256, 0, st>>>(dist, issame, n, thr, counts);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

extern "C" int crfr_verify_sweep(const float* dist, const uint8_t* issame, const int* subset, int n,
                                 const float* thresholds, int nthr, unsigned int* counts, void* stream) {
  CRFR_CHECK_ARG(dist && issame && thresholds && counts && n > 0 && nthr > 0, "verify_sweep: bad argument");
  verify_sweep_kernel<<<crfr_cdiv(nthr, 256), 256, 0, (cudaStream_t)stream>>>(dist, issame, subset, n, thresholds, nthr,
                                                                              counts);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

extern "C" int crfr_l2norm_bf16(const float* x, void* out, long long rows, int dim, void* stream) {
  CRFR_CHECK_ARG(x && out && rows > 0 && dim > 0, "l2norm_bf16: bad argument");
  long long threads = rows * 32;
  l2norm_kernel<<<crfr_cdiv(threads, 256), 256, 0, (cudaStream_t)stream>>>(x, (bf16*)out, rows, dim);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

extern "C" int crfr_pair_verify(const float* e1, const float* e2, long long pairs, int dim, float thr, float* dist,
                                uint8_t* same, void* stream) {
  CRFR_CHECK_ARG(e1 && e2 && pairs > 0 && dim > 0 && (dist || same), "pair_verify: bad argument");
  long long threads = pairs * 32;
  pair_verify_kernel<<<crfr_cdiv(threads, 256), 256, 0, (cudaStream_t)stream>>>(e1, e2, pairs, dim, thr, dist, same);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}
