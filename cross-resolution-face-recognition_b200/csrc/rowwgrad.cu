// Persistent row-streaming weight gradient for the dominant FSRNet layer shape (3x3, 64 -> 64 channels, width 128).
//
//   dW[ky][kx][ci][co] = sum_{n,y,x} X[n][y+ky-1][x+kx-1][ci] * dY[n][y][x][co]
//
// Pixels are the GEMM K dimension, so both operands are MN-major views of NHWC rows (channels contiguous).  As in
// rowconv.cu the natural N = 64 MMA is avoided (it is capped at ~50 % of the tensor pipe, tools/micro/mma_bench.cu):
// for one input row q of X the three dY rows q-1, q, q+1 (= ky 2, 1, 0) are stacked along N through the descriptor's
// leading-byte-offset (consecutive slots of the dY ring), and two kx taps are stacked along M the same way - the kx
// shift of the X row (loaded once, with halo) is a 128-byte start offset, so the second M atom is simply LBO = 128 B
// away:
//     D1[(kx 0|1) x 64 ci][(ky 2|1|0) x 64 co] += X_q(shift 0|1)^T * [dY_{q-1} | dY_q | dY_{q+1}]      (M=128, N=192)
//     D2[(kx 2|-) x 64 ci][...]                 += X_q(shift 2|3)^T * [...]                               (upper half unused)
// 16 MMAs (K = 16 pixels each) per row instead of 48 N = 64 MMAs.  Rows outside the image are TMA zero fill.
// An M = 64 MMA costs the tensor pipe as much as M = 128, so D2 above runs at half use (the kernel at 75 %).  For an even image
// height the rows are therefore processed in PAIRS (q, q+1) and the two kx = 2 atoms share one MMA over the FOUR dY rows that
// the pair touches:
//     D2[(X_q | X_{q+1}) shift 2 x 64 ci][(dY_{q-1} | dY_q | dY_{q+1} | dY_{q+2}) x 64 co]               (M=128, N=256)
// (M atoms one X slot apart, N atoms one dY slot apart).  Six of its eight 64 x 64 blocks are wanted - X_q with dY_{q+2} and
// X_{q+1} with dY_{q-1} are no taps and are dropped by the epilogue - so a pair costs 2 x 192 + 256 = 640 accumulator columns
// per K step instead of 768: 90 % of the issued MMA work is useful instead of 75 %.  Measured (128 images, incl. the slab
// reduction): 154 -> 137.5 us.  ncu on the pair form (profiles/r2_rowwgrad_pair_ncu.txt, 124 us): tensor pipe 80 % of the active
// cycles, the tensor core's shared-memory reads - an SS-mode MMA streams (128 + N) x 32 bytes per N / 2 cycles - 59 % of their
// peak, DRAM 4.4 TB/s: no unit is saturated; the idle fifth is the prologue (TMEM zero fill, first loads), the slab epilogue
// and ring waits.  Deeper rings change nothing (6 X slots packed at 130 x 128 bytes - the swizzle is a function of the
// address, slot bases need only 128-byte alignment: verified - 135.6 us; dY ring 8: 139.9 us; L2 prefetch 2 / 4 / 8 rows ahead:
// 138.7 / 139.8 / 145.4 us).
//
// ref: the weight gradients of the nn.Conv2d sites model/FSRnet.py:79,85 (coarse / decoder residual stacks).
#include <cudaTypedefs.h>
#include <stdlib.h>

#include "common.cuh"
#include "crfr.h"
#include "internal.h"
#include "sm100.cuh"

using namespace sm100;

namespace {

constexpr int kW = 128;
constexpr int kC = 64;
constexpr int kXRowBytes = 132 * 128;      // X row with halo: x = -1 .. 130 (shift 3 of the unused atom stays inside)
constexpr int kXSlotBytes = 17 * 1024;
constexpr int kXSlots = 4;
constexpr int kDyRowBytes = 128 * 128;
constexpr int kDyRing = 6;                 // dY ring positions ...
constexpr int kDySlots = kDyRing + 2;      // ... plus two MIRROR slots: rows at ring positions 0 and 1 are also loaded behind the
                                           // last position, so the three consecutive dY rows of an X row are always contiguous
                                           // in shared memory (one N = 192 MMA, never a split where the ring wraps)
constexpr int kDone = 8;                   // ring of "X row consumed" barriers
constexpr int kPrefetch = 0;               // rows pulled into L2 ahead of the shared-memory rings.  0: with the mirror slots and the
                                           // lean issue loop the cursor only costs - 10 rows ahead the kernel read 765 MB from DRAM
                                           // per 128-image launch instead of the algorithmic 537 MB (542 MB without) and took
                                           // 165 us instead of 154 us (ncu dram__bytes_read, CUDA events incl. slab reduction)
constexpr int kThreads = 192;
constexpr int kSlabFloats = 9 * kC * kC;
constexpr int kSmemBytes = kXSlots * kXSlotBytes + kDySlots * kDyRowBytes + 1024 + 512;
static_assert(kSmemBytes <= 232448, "shared memory budget");

struct WgParams {
  int n, h, total_rows;
  float* slabs;   // [gridDim.x][9][64][64]
  int prefetch;   // rows pulled into L2 ahead of the rings
  int paired;     // even image height: rows in pairs, the kx = 2 taps of a pair in one M = 128, N = 256 MMA
};

// One MMA: descriptors that differ only in their low word (start address) from precomputed bases - the issuing warp is the
// serial resource of a single-issuer kernel (see rowconv2.cu): two 32-bit adds and one UTCHMMA per MMA.
__device__ __forceinline__ void umma_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %3};\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "setp.ne.b32 p, 1, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t}" ::"r"(d_tmem),
      "r"(a_lo), "r"(b_lo), "r"(desc_hi), "r"(idesc)
      : "memory");
}

__global__ void __launch_bounds__(kThreads, 1)
rowwgrad_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmDY, WgParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* sX = base;
  uint8_t* sDY = base + kXSlots * kXSlotBytes;
  uint64_t* full_x = (uint64_t*)(sDY + kDySlots * kDyRowBytes);
  uint64_t* full_dy = full_x + kXSlots;       // [kDyRing]
  uint64_t* done = full_dy + kDyRing;         // [kDone] the MMAs of X row g are complete: frees its X slot and dY row g - 1
  uint64_t* fin = done + kDone;
  uint32_t* tmem_slot = (uint32_t*)(fin + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kXSlots; ++s) mbar_init(&full_x[s], 1);
    for (int s = 0; s < kDyRing; ++s) mbar_init(&full_dy[s], 1);
    for (int s = 0; s < kDone; ++s) mbar_init(&done[s], 1);
    mbar_init(fin, 1);
    fence_barrier_init();
    prefetch_tmap(&tmX);
    prefetch_tmap(&tmDY);
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  if (warp >= 2) {   // the accumulators start at zero: every MMA of this kernel accumulates
    for (int c = 0; c < 512; c += 32) tmem_st32_zero(tmem + ((uint32_t)((warp & 3) * 32) << 16) + c);
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  // paired: ranges of whole row pairs (h even: an image boundary is a pair boundary too)
  const long long units = p.paired ? p.total_rows / 2 : p.total_rows;
  const long long r_begin = (units * blockIdx.x / gridDim.x) << p.paired;
  const long long r_end = (units * (blockIdx.x + 1) / gridDim.x) << p.paired;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    // Load order = use order: per segment dY rows y0-1 .. y0+seg (out-of-image rows are zero filled) interleaved with X
    // rows y0 .. y0+seg-1.  X row i (running index gx) uses dY rows i, i+1, i+2 of its segment; a dY row is free again
    // when the last X row that uses it is done, an X slot when its own row is done: both are the SAME event, the one
    // commit per X row on done[gx % kDone].  A prefetch cursor runs kPrefetch rows ahead and pulls rows into L2 (the
    // rings hold less than the DRAM latency x bandwidth product at the rate the MMAs consume rows).
    const bool leader = elect_one();
    int last_user[kDyRing];                       // running X index of the last user of the dY row in each ring position
#pragma unroll
    for (int i = 0; i < kDyRing; ++i) last_user[i] = -1;
    int gx = 0, gd = 0;
    long long r = r_begin, rp = r_begin;          // load cursor / prefetch cursor (segment starts)
    int pf_i = -1, pf_seg = 0, pf_n = 0, pf_y0 = 0, pf_ahead = 0;
    bool pf_valid = false;
    auto pf_start = [&]() {
      pf_valid = rp < r_end;
      if (!pf_valid) return;
      pf_n = (int)(rp / p.h); pf_y0 = (int)(rp % p.h);
      pf_seg = (int)min((long long)(p.h - pf_y0), r_end - rp);
      pf_i = -1;
      rp += pf_seg;
    };
    auto pf_step = [&]() {   // prefetch the dY row (and X row) of one step of the load order
      if (!pf_valid) return;
      const int yd = pf_y0 + pf_i;
      if (leader && yd >= 0 && yd < p.h) tma_prefetch_4d(&tmDY, 0, 0, yd, pf_n);
      if (leader && pf_i >= 1) tma_prefetch_4d(&tmX, 0, -1, pf_y0 + pf_i - 1, pf_n);
      if (++pf_i > pf_seg) pf_start();
    };
    pf_start();
    for (; pf_ahead < p.prefetch; ++pf_ahead) pf_step();
    while (r < r_end) {
      const int n = (int)(r / p.h), y0 = (int)(r % p.h);
      const int seg = (int)min((long long)(p.h - y0), r_end - r);
      const int gx0 = gx;
      for (int i = -1; i <= seg; ++i) {
        if (p.prefetch) pf_step();
        {
          const int pos = gd % kDyRing;
          const int lu = last_user[pos];
          if (lu >= 0) mbar_wait(&done[lu & (kDone - 1)], (lu / kDone) & 1);
          last_user[pos] = gx0 + min(i + 1, seg - 1);   // dY row j = i + 1 of the segment is used by X rows j-2 .. j
          if (leader) {
            const bool mirror = pos < 2;
            mbar_expect_tx(&full_dy[pos], mirror ? 2 * kDyRowBytes : kDyRowBytes);
            tma_load_4d(sDY + pos * kDyRowBytes, &tmDY, &full_dy[pos], 0, 0, y0 + i, n);
            if (mirror) tma_load_4d(sDY + (kDyRing + pos) * kDyRowBytes, &tmDY, &full_dy[pos], 0, 0, y0 + i, n);
          }
          ++gd;
        }
        if (i >= 1) {   // X row y0+i-1 is first needed once dY row y0+i has been requested
          const int s = gx % kXSlots;
          if (gx >= kXSlots) mbar_wait(&done[(gx - kXSlots) & (kDone - 1)], ((gx - kXSlots) / kDone) & 1);
          if (leader) {
            mbar_expect_tx(&full_x[s], kXRowBytes);
            tma_load_4d(sX + s * kXSlotBytes, &tmX, &full_x[s], 0, -1, y0 + i - 1, n);
          }
          ++gx;
        }
      }
      r += seg;
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    const bool leader = elect_one();
    // A: two 64-channel atoms 128 B apart (the kx and kx+1 views of the same row); B: N atoms one dY slot apart
    const uint64_t xdesc0 = make_smem_desc_sw128(smem_u32(sX), 128, 1024);
    const uint64_t dydesc0 = make_smem_desc_sw128(smem_u32(sDY), kDyRowBytes, 1024);
    const uint32_t desc_hi = (uint32_t)(xdesc0 >> 32), x_lo = (uint32_t)xdesc0, dy_lo = (uint32_t)dydesc0;
    const uint32_t idesc = make_idesc_bf16(128, 3 * kC, 1, 1);
    // paired form: A atoms = the kx = 2 views of two consecutive X slots, B = four dY slots
    const uint32_t x2_lo = (uint32_t)make_smem_desc_sw128(smem_u32(sX) + 256, kXSlotBytes, 1024);
    const uint32_t idesc4 = make_idesc_bf16(128, 4 * kC, 1, 1);
    int sx = 0;  uint32_t xph = 0;    // X ring slot of the current row and its parity
    int dp = 0;  uint32_t dph = 0;    // dY ring position of the current row's first dY row (q - 1), and its parity
    int dg = 0;
    long long r = r_begin;
    while (r < r_end) {
      const int y0 = (int)(r % p.h);
      const int seg = (int)min((long long)(p.h - y0), r_end - r);
      if (p.paired) {
        // dp is even here (even ring, even segments): positions dp .. dp + 3 are contiguous through the two mirror slots,
        // and so are dp + 1 .. dp + 3 for the second row of the pair
        for (int i = 0; i < seg; i += 2) {
          int p1 = dp + 1, p2 = dp + 2, p3 = dp + 3;
          uint32_t ph2 = dph;
          if (p2 >= kDyRing) { p2 -= kDyRing; p3 -= kDyRing; ph2 ^= 1; }
          if (i == 0) {
            mbar_wait(&full_dy[dp], dph);
            mbar_wait(&full_dy[p1], dph);
          }
          mbar_wait(&full_dy[p2], ph2);
          mbar_wait(&full_x[sx], xph);
          tc_fence_after();
          const uint32_t a0 = x_lo + (uint32_t)(sx * (kXSlotBytes >> 4));
          const uint32_t b0 = dy_lo + (uint32_t)(dp * (kDyRowBytes >> 4));
          if (leader) {
#pragma unroll
            for (int k = 0; k < 8; ++k)
              umma_lo(tmem, a0 + (uint32_t)(k * (2048 >> 4)), b0 + (uint32_t)(k * (2048 >> 4)), desc_hi, idesc);
          }
          __syncwarp();
          mbar_wait(&full_dy[p3], ph2);
          mbar_wait(&full_x[sx + 1], xph);
          tc_fence_after();
          if (leader) {
            const uint32_t a1 = a0 + (uint32_t)(kXSlotBytes >> 4), b1 = b0 + (uint32_t)(kDyRowBytes >> 4);
            const uint32_t a2 = x2_lo + (uint32_t)(sx * (kXSlotBytes >> 4));
#pragma unroll
            for (int k = 0; k < 8; ++k)
              umma_lo(tmem, a1 + (uint32_t)(k * (2048 >> 4)), b1 + (uint32_t)(k * (2048 >> 4)), desc_hi, idesc);
#pragma unroll
            for (int k = 0; k < 8; ++k)
              umma_lo(tmem + 256, a2 + (uint32_t)(k * (2048 >> 4)), b0 + (uint32_t)(k * (2048 >> 4)), desc_hi, idesc4);
            umma_commit(&done[dg]);          // both rows are released by the pair's last MMA
            umma_commit(&done[dg + 1]);
          }
          __syncwarp();
          sx += 2;
          if (sx == kXSlots) { sx = 0; xph ^= 1; }
          dp += 2;
          if (dp == kDyRing) { dp = 0; dph ^= 1; }
          dg = (dg + 2) & (kDone - 1);
        }
      } else
      for (int i = 0; i < seg; ++i) {
        // dY rows q-1, q, q+1 = ring positions dp, dp+1, dp+2 (mod kDyRing); the first two were waited for by the previous
        // row of the segment
        int p1 = dp + 1, p2 = dp + 2;
        uint32_t ph1 = dph, ph2 = dph;
        if (p1 >= kDyRing) { p1 -= kDyRing; ph1 ^= 1; }
        if (p2 >= kDyRing) { p2 -= kDyRing; ph2 ^= 1; }
        if (i == 0) {
          mbar_wait(&full_dy[dp], dph);
          mbar_wait(&full_dy[p1], ph1);
        }
        mbar_wait(&full_dy[p2], ph2);
        mbar_wait(&full_x[sx], xph);
        tc_fence_after();
        const uint32_t a01 = x_lo + (uint32_t)(sx * (kXSlotBytes >> 4));
        const uint32_t a2x = a01 + (uint32_t)(256 >> 4);
        const uint32_t b0 = dy_lo + (uint32_t)(dp * (kDyRowBytes >> 4));   // contiguous thanks to the mirror slots
        if (leader) {
#pragma unroll
          for (int k = 0; k < 8; ++k) {             // 8 x 16 pixels
            umma_lo(tmem, a01 + (uint32_t)(k * (2048 >> 4)), b0 + (uint32_t)(k * (2048 >> 4)), desc_hi, idesc);
            umma_lo(tmem + 256, a2x + (uint32_t)(k * (2048 >> 4)), b0 + (uint32_t)(k * (2048 >> 4)), desc_hi, idesc);
          }
          umma_commit(&done[dg]);
        }
        __syncwarp();
        if (++sx == kXSlots) { sx = 0; xph ^= 1; }
        if (++dp == kDyRing) { dp = 0; dph ^= 1; }
        dg = (dg + 1) & (kDone - 1);
      }
      // the segment's last two dY rows belong to no later X row of this segment
      dp += 2;
      if (dp >= kDyRing) { dp -= kDyRing; dph ^= 1; }
      r += seg;
    }
    if (leader) umma_commit(fin);
    __syncwarp();
  } else {
    // ------------------------------------------------------------------ epilogue: TMEM -> this CTA's slab
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int ci = row & 63;
    mbar_wait(fin, 0);
    tc_fence_after();
    float* slab = p.slabs + (size_t)blockIdx.x * kSlabFloats;
    if (p.paired) {
      // D2 lanes 0-63: X_q with dY_{q-1+b} in column block b -> ky = 2 - b (b = 3 is no tap); lanes 64-127: X_{q+1} with the
      // same dY rows -> ky = 3 - b (b = 0 is no tap).  Both halves belong to the same nine 64 x 64 gradients: the lower
      // lanes store, the upper lanes add after a barrier (fixed order: deterministic).
      const bool upper = row >= 64;                 // warp-uniform
#pragma unroll
      for (int phase = 0; phase < 2; ++phase) {
        if ((phase == 1) == upper) {
#pragma unroll
          for (int c0 = 0; c0 < 256; c0 += 32) {
            const int b = c0 / 64;
            const int ky = (upper ? 3 : 2) - b;
            if (ky < 0 || ky > 2) continue;
            uint32_t v[32];
            tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + 256 + c0, v);
            tmem_ld_wait();
            float* dst = slab + ((size_t)(ky * 3 + 2) * kC + ci) * kC + (c0 & 63);
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              float4 o = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]),
                                     __uint_as_float(v[j + 3]));
              if (upper) {
                const float4 t = *reinterpret_cast<const float4*>(dst + j);
                o.x += t.x; o.y += t.y; o.z += t.z; o.w += t.w;
              }
              *reinterpret_cast<float4*>(dst + j) = o;
            }
          }
        }
        if (phase == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
      }
    }
#pragma unroll
    for (int half = 0; half < (p.paired ? 1 : 2); ++half) {
      const int kx = half == 0 ? (row >> 6) : 2;
      const bool live = half == 0 || row < 64;      // warp-uniform
#pragma unroll
      for (int c0 = 0; c0 < 192; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + half * 256 + c0, v);
        tmem_ld_wait();
        if (live) {
          const int ky = 2 - c0 / 64;
          float* dst = slab + ((size_t)(ky * 3 + kx) * kC + ci) * kC + (c0 & 63);
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            *reinterpret_cast<float4*>(dst + j) = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]),
                                                              __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem);
  }
}

// dW[co][ci][t] += sum_slabs slab[s][t][ci][co]   (fixed order).  64 outputs per block; four thread groups each sum every
// fourth slab with four independent accumulators (the first version - one thread per output walking all 148 slabs - was a
// 14 us latency chain, 0.5 ms per training step), then the groups are folded in fixed order through shared memory.
__global__ void __launch_bounds__(256)
slab_reduce_kernel(const float* __restrict__ slabs, int nslabs, float* __restrict__ dw) {
  __shared__ float part[4][64];
  const int o = threadIdx.x & 63, grp = threadIdx.x >> 6;
  const int i = blockIdx.x * 64 + o;   // over [t][ci][co]
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  int s = grp;
  for (; s + 12 < nslabs; s += 16) {
    s0 += slabs[(size_t)s * kSlabFloats + i];
    s1 += slabs[(size_t)(s + 4) * kSlabFloats + i];
    s2 += slabs[(size_t)(s + 8) * kSlabFloats + i];
    s3 += slabs[(size_t)(s + 12) * kSlabFloats + i];
  }
  for (; s < nslabs; s += 4) s0 += slabs[(size_t)s * kSlabFloats + i];
  part[grp][o] = (s0 + s1) + (s2 + s3);
  __syncthreads();
  if (grp == 0) {
    const int co = i & 63, ci = (i >> 6) & 63, t = i >> 12;
    dw[((size_t)co * kC + ci) * 9 + t] += (part[0][o] + part[1][o]) + (part[2][o] + part[3][o]);
  }
}

int encode(CUtensorMap* m, const void* ptr, int n, int h, int ld, int box_w, const char* what) {
  const unsigned long long dims[4] = {(unsigned long long)kC, (unsigned long long)kW, (unsigned long long)h,
                                      (unsigned long long)n};
  const unsigned long long strides[3] = {(unsigned long long)ld * 2, (unsigned long long)kW * ld * 2,
                                         (unsigned long long)h * kW * ld * 2};
  const unsigned int box[4] = {64, (unsigned int)box_w, 1, 1};
  return crfr_tmap_encode_bf16(m, ptr, 4, dims, strides, box, what);
}

int grid_for(int total_rows, int h) {
  const int sms = crfr_sm_count();
  const int units = (h & 1) ? total_rows : total_rows / 2;   // even height: CTAs take whole row pairs
  return sms < units ? sms : units;
}

}  // namespace

int crfr_rowwgrad_supported(int h, int w, int cin, int cout, int k, int stride, int pad) {
  return w == kW && cin == kC && cout == kC && k == 3 && stride == 1 && pad == 1 && h >= 1;
}

size_t crfr_rowwgrad_ws_bytes(int n, int h) { return sizeof(float) * (size_t)grid_for(n * h, h) * kSlabFloats + 256; }

// x, dy: NHWC bf16 [n][h][128][64] views; dw: fp32 [64][64][3][3], accumulated.
int crfr_rowwgrad(const void* x, int x_ld, const void* dy, int dy_ld, int n, int h, float* dw, void* ws,
                  size_t ws_bytes, cudaStream_t st) {
  CRFR_CHECK_ARG(((uintptr_t)x & 15) == 0 && ((uintptr_t)dy & 15) == 0 && (x_ld & 7) == 0 && (dy_ld & 7) == 0,
                 "rowwgrad: pointers must be 16B aligned and ld a multiple of 8");
  const size_t need = crfr_rowwgrad_ws_bytes(n, h);
  if (!ws || ws_bytes < need) {
    crfr_set_error("rowwgrad: workspace %zu < %zu", ws_bytes, need);
    return CRFR_EWORKSPACE;
  }
  CUtensorMap tmX, tmDY;
  CRFR_TRY(encode(&tmX, x, n, h, x_ld, 132, "x"));
  CRFR_TRY(encode(&tmDY, dy, n, h, dy_ld, 128, "dy"));
  static std::atomic<unsigned long long> attr_done{0};
  CRFR_CUDA((cudaError_t)crfr_smem_attr(rowwgrad_kernel, kSmemBytes, attr_done));
  WgParams p;
  p.n = n; p.h = h; p.total_rows = n * h;
  p.slabs = (float*)ws;
  p.prefetch = kPrefetch;
  p.paired = (h & 1) ? 0 : 1;
  const int grid = grid_for(p.total_rows, h);
  rowwgrad_kernel<<<grid, kThreads, kSmemBytes, st>>>(tmX, tmDY, p);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  slab_reduce_kernel<<<kSlabFloats / 64, 256, 0, st>>>((const float*)ws, grid, dw);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}
