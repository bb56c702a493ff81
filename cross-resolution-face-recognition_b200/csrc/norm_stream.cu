// TMA-fed versions of the two InstanceNorm / BatchNorm backward passes (norm_act.cu holds the arithmetic contract).
//
// Why: the register-staged passes ran at 3.1 TB/s (reduce) and 5.3 TB/s (apply) against 6.45 TB/s.  They are not short
// of loads in flight - a first TMA-fed version with the same arithmetic was no faster - they are ISSUE bound: ~12
// instructions per channel (scalar fp32, per-load address arithmetic, two unpacks, a round trip through bf16, three
// accumulations) at ~5 channels per clock per SM.  Here:
//   * a producer warp streams [32 pixels x 64 channels] SWIZZLE_128B boxes of every input map (2-4 maps) through an
//     88 KB ring of 4 KB-per-map stages with cp.async.bulk.tensor + mbarrier complete_tx; two CTAs per SM;
//   * the 8 consumer warps read their 16 bytes per map with one ld.shared.v4 (no address arithmetic, no predication)
//     and do two channels per packed fp32x2 instruction (FFMA2 / FADD2, sm_100): sum(dz * xhat) is accumulated as
//     sum(dz * y) and centred once per segment, dz is rounded and packed by one cvt.rn.bf16x2, the apply pass is
//     ca * dz + cb * y + cc - about 8 instructions per channel;
//   * the kernels are persistent: CTA b owns the contiguous range [b R / G, (b + 1) R / G) of the flattened
//     (image, pixel) space (R = n x hw, G = 2 CTAs per SM), split into per-image segments.  The producer runs ahead
//     across segment boundaries, so the per-segment work of the consumers (the image's coefficients, folding the
//     partial sums) overlaps the loads of the next segment; the former (chunk, image) grid of ~600-pixel CTAs lost a
//     third of the bandwidth to start-up and reduction tails.
// Partial sums go to fixed (image, CTA) slots and are folded in fixed order by bwd_fold_kernel: deterministic.  Same
// arithmetic per element as norm_act_bwd_reduce/apply_kernel up to the association of the fp32 sums.
// Measured (profiles/r1_norm_stream_ncu_full.txt): 6.26 / 6.10 TB/s of DRAM traffic inside the reduce / apply kernel.
//
// ref: backward of nn.InstanceNorm2d + nn.PReLU + residual add (model/FSRnet.py:75-98, 105-135) and of train-mode
//      nn.BatchNorm2d + ReLU (model/resnet.py:24-45).
#include <cudaTypedefs.h>

#include "common.cuh"
#include "crfr.h"
#include "internal.h"
#include "sm100.cuh"

using namespace sm100;

namespace {

constexpr int kConsumers = 256;
constexpr int kThreads = kConsumers + 32;   // + one producer warp
constexpr int kTileBytes = 4096;            // one map, one stage, one pixel per consumer: 256 x 16 B; passes that stream
                                            // two maps use two pixels per consumer and stage (8 KB tiles): half the
                                            // per-stage barrier / address work in loops that are close to issue bound
constexpr int kRingBytes = 88 * 1024;       // stage ring per CTA (two CTAs per SM)
constexpr int kMaxStages = 16;
constexpr int kScratchBytes = 8192;         // [lanes][c] floats = 256 x 8 x 4 B

struct Maps {
  CUtensorMap t[4];
};

struct StreamArgs {
  int ntensors, stages, ring_bytes, tile_bytes;
  int hw, c, nimg, parts;
  long long total;                  // n x hw pixels
  int relu, has_b, has_res, recompute;
  const float* stats; const float* gamma; const float* beta; const float* alpha;
  const float* bstats; const float* tot;   // apply: folded sums (register-kernel contract), or NULL: fold `partial` here
  float inv_hw;
  bf16* out; int out_ld;            // reduce: dz (may be null); apply: dy
  float* partial;                   // reduce: [n][parts][3][c]
  float* dgamma; float* dbeta; float* dalpha;
};

__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void st_stream(bf16* p, const uint4& u) {
  asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(u.x), "r"(u.y), "r"(u.z), "r"(u.w) : "memory");
}
// bf16x2 word <-> two fp32 (low half = even channel)
__device__ __forceinline__ float2 up2(uint32_t w) {
  return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
}
__device__ __forceinline__ uint32_t pk2(float2 v) {
  const __nv_bfloat162 b = __floats2bfloat162_rn(v.x, v.y);
  return *reinterpret_cast<const uint32_t*>(&b);
}
__device__ __forceinline__ uint32_t word(const uint4& v, int i) { return i == 0 ? v.x : (i == 1 ? v.y : (i == 2 ? v.z : v.w)); }
__device__ __forceinline__ void set_word(uint4& v, int i, uint32_t w) {
  if (i == 0) v.x = w; else if (i == 1) v.y = w; else if (i == 2) v.z = w; else v.w = w;
}

// Byte offset, inside a stage's tile of one map, of the 16 bytes (8 channels) that consumer (channel group cg, pixel lane)
// reads.  The tile is c / 64 SWIZZLE_128B boxes of [P pixels][64 channels]; the swizzle XORs the 16-byte chunk index
// with bits 7..9 of the shared-memory address (tiles are 4 KB aligned), which is the pixel row only while a box is a
// whole number of 1 KB swizzle atoms - at 512 channels a box is 4 rows = 512 bytes.
__device__ __forceinline__ uint32_t sw128_offset(int cg, int lane, int P) {
  const uint32_t row = (uint32_t)((cg >> 3) * P + lane);            // 128-byte row inside the tile
  return row * 128 + ((((uint32_t)cg & 7) ^ (row & 7)) << 4);
}

// first CTA whose range [total b / G, total (b + 1) / G) contains pixel x
__device__ __forceinline__ int first_cta_of(long long x, long long total, int G) {
  return (int)(((x + 1) * G + total - 1) / total) - 1;
}

struct Setup {
  uint32_t ring;        // shared-window addresses
  uint32_t full, empty;
  float* scratch;
  int r_begin, r_end;   // this CTA's range of the flattened (image, pixel) space (n x hw < 2^31)
};

__device__ __forceinline__ uint64_t* bar_ptr(uint8_t* ring, int ring_bytes, int which, int s) {
  return (uint64_t*)(ring + ring_bytes + kScratchBytes) + which * kMaxStages + s;
}
__device__ __forceinline__ void mbar_wait_a(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  for (uint32_t i = 0; i < (1u << 24) && !ok; ++i)
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
  if (!ok) __trap();   // a protocol bug traps instead of hanging the GPU box
}
__device__ __forceinline__ void mbar_arrive_a(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ Setup setup(const StreamArgs& a, uint8_t* smem_raw) {
  Setup u;
  uint8_t* ring = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  u.ring = smem_u32(ring);
  u.scratch = (float*)(ring + a.ring_bytes);
  u.full = smem_u32(bar_ptr(ring, a.ring_bytes, 0, 0));
  u.empty = smem_u32(bar_ptr(ring, a.ring_bytes, 1, 0));
  u.r_begin = (int)(a.total * blockIdx.x / gridDim.x);
  u.r_end = (int)(a.total * (blockIdx.x + 1) / gridDim.x);
  if (threadIdx.x == 0) {
    for (int s = 0; s < a.stages; ++s) {
      mbar_init(bar_ptr(ring, a.ring_bytes, 0, s), 1);
      mbar_init(bar_ptr(ring, a.ring_bytes, 1, s), kConsumers / 32);
    }
    fence_barrier_init();
  }
  __syncthreads();
  return u;
}

// producer warp: stream every stage of this CTA's range, running ahead of the consumers across segment boundaries
__device__ __forceinline__ void produce(const Maps& maps, const StreamArgs& a, const Setup& u, int P) {
  const bool leader = elect_one();
  const int subs = a.c >> 6;
  const uint32_t stage_bytes = a.ntensors * a.tile_bytes;
  int s = 0;
  uint32_t phase = 1;
  int r = u.r_begin;
  while (r < u.r_end) {
    const int off = r % a.hw;
    const int seg = min(a.hw - off, u.r_end - r);
    const int nst = (seg + P - 1) / P;
    for (int k = 0; k < nst; ++k) {
      mbar_wait_a(u.empty + 8 * s, phase);
      if (leader) {
        const uint32_t fb = u.full + 8 * s;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(fb), "r"(stage_bytes) : "memory");
        const uint32_t stage = u.ring + s * stage_bytes;
        for (int t = 0; t < a.ntensors; ++t)
          for (int sub = 0; sub < subs; ++sub)
            asm volatile(
                "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                ::"r"(stage + t * a.tile_bytes + sub * (P * 128)), "l"(&maps.t[t]), "r"(fb), "r"(sub * 64), "r"(r + k * P)
                : "memory");
      }
      __syncwarp();
      if (++s == a.stages) { s = 0; phase ^= 1; }
    }
    r += seg;
  }
}

// pass 1: dz = dout * act'(z) (bf16), per-(image, CTA) partial sums of dz, dz * xhat, dout * min(z, 0).
// The inner loop is issue-bound, not bandwidth-bound, unless it is kept to ~8 instructions per channel: two channels
// per packed fp32x2 instruction (FFMA2 / FADD2), sum(dz * xhat) accumulated as sum(dz * y) and centred once per
// segment, rounding and packing of dz in one cvt.rn.bf16x2.
template <bool HAS_B, bool HAS_RES>
__device__ __forceinline__ void reduce_consume(const StreamArgs& a, const Setup& u, int P) {
  constexpr int PX = (HAS_B || HAS_RES) ? 1 : 2;   // pixels per consumer and stage
  constexpr int kTile = PX * kTileBytes;
  const int c = a.c, groups = c >> 3, lanes = kConsumers / groups;
  const int cg = threadIdx.x % groups, lane = threadIdx.x / groups;
  const bool act = a.relu || a.alpha;
  const uint32_t stage_bytes = a.ntensors * kTile;
  uint32_t my_off[PX];
#pragma unroll
  for (int h = 0; h < PX; ++h) my_off[h] = sw128_offset(cg, lane + h * lanes, P);
  constexpr int ty = HAS_B ? 2 : 1, tr = ty + 1;   // tensor order in a stage: dout_a, [dout_b], y, [res]
  int s = 0;
  uint32_t phase = 0;
  int r = u.r_begin;
  while (r < u.r_end) {
    const int img = r / a.hw, off = r - img * a.hw;
    const int seg = min(a.hw - off, u.r_end - r);
    const int nst = (seg + P - 1) / P;
    float2 sc[4], sh[4], al[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float t[6];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int ch = cg * 8 + 2 * i + e;
        const float mu = a.stats[2 * (img * c + ch)], rs = a.stats[2 * (img * c + ch) + 1];
        t[e] = (a.gamma ? a.gamma[ch] : 1.f) * rs;
        t[2 + e] = (a.beta ? a.beta[ch] : 0.f) - mu * t[e];
        t[4 + e] = a.relu ? 0.f : (a.alpha ? a.alpha[ch] : 1.f);
      }
      sc[i] = make_float2(t[0], t[1]);
      sh[i] = make_float2(t[2], t[3]);
      al[i] = make_float2(t[4], t[5]);
    }
    float2 acc0[4], acc1[4], acc2[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) acc0[i] = acc1[i] = acc2[i] = make_float2(0.f, 0.f);
    const bool store = a.out != nullptr;
    bf16* optr = a.out + ((long long)r + lane) * a.out_ld + cg * 8;
    const long long ostep = (long long)P * a.out_ld;
    for (int k = 0; k < nst; ++k) {
      mbar_wait_a(u.full + 8 * s, phase);
#pragma unroll
      for (int h = 0; h < PX; ++h) {
        const uint32_t addr = u.ring + s * stage_bytes + my_off[h];
        if (k * P + lane + h * lanes < seg) {
          const uint4 A = lds128(addr);
          uint4 B, R;
          if (HAS_B) B = lds128(addr + kTile);
          const uint4 Y = lds128(addr + ty * kTile);
          if (HAS_RES) R = lds128(addr + tr * kTile);
          uint4 O;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            float2 g = up2(word(A, i));
            if (HAS_B) g = __fadd2_rn(g, up2(word(B, i)));
            const float2 f = up2(word(Y, i));
            if (act) {
              float2 z = __ffma2_rn(f, sc[i], sh[i]);
              if (HAS_RES) z = __fadd2_rn(z, up2(word(R, i)));
              if (!(z.x > 0.f)) { acc2[i].x = fmaf(g.x, z.x, acc2[i].x); g.x *= al[i].x; }
              if (!(z.y > 0.f)) { acc2[i].y = fmaf(g.y, z.y, acc2[i].y); g.y *= al[i].y; }
            }
            const uint32_t w = pk2(g);
            set_word(O, i, w);
            const float2 d = up2(w);
            acc0[i] = __fadd2_rn(acc0[i], d);
            acc1[i] = __ffma2_rn(d, f, acc1[i]);
          }
          if (store) *reinterpret_cast<uint4*>(optr + (long long)h * lanes * a.out_ld) = O;
        }
      }
      optr += ostep;
      __syncwarp();
      if ((threadIdx.x & 31) == 0) mbar_arrive_a(u.empty + 8 * s);
      if (++s == a.stages) { s = 0; phase ^= 1; }
    }
    // centre and scale: sum(dz * xhat) = rstd * (sum(dz * y) - mean * sum(dz))
    float q[3][8];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int ch = cg * 8 + 2 * i + e;
        const float mu = a.stats[2 * (img * c + ch)], rs = a.stats[2 * (img * c + ch) + 1];
        const float s0 = e ? acc0[i].y : acc0[i].x, s1 = e ? acc1[i].y : acc1[i].x;
        q[0][2 * i + e] = s0;
        q[1][2 * i + e] = (s1 - mu * s0) * rs;
        q[2][2 * i + e] = e ? acc2[i].y : acc2[i].x;
      }
    }
    // fold the pixel lanes in fixed order, one quantity at a time through the [lanes][c] scratch, and publish this
    // CTA's partial of the image in its fixed slot
    const int part = blockIdx.x - first_cta_of((long long)img * a.hw, a.total, gridDim.x);
    float* dst = a.partial + ((long long)img * a.parts + part) * 3 * c;
#pragma unroll
    for (int qq = 0; qq < 3; ++qq) {
      named_bar_sync(1, kConsumers);
#pragma unroll
      for (int j = 0; j < 8; ++j) u.scratch[lane * c + cg * 8 + j] = q[qq][j];
      named_bar_sync(1, kConsumers);
      for (int ch = threadIdx.x; ch < c; ch += kConsumers) {
        float t = 0.f;
        for (int l = 0; l < lanes; ++l) t += u.scratch[l * c + ch];
        dst[qq * c + ch] = t;
      }
    }
    if (off + seg == a.hw)   // last CTA of this image: the unused slots must read as zero
      for (int z = part + 1; z < a.parts; ++z)
        for (int i = threadIdx.x; i < 3 * c; i += kConsumers) a.partial[((long long)img * a.parts + z) * 3 * c + i] = 0.f;
    r += seg;
  }
}

__global__ void __launch_bounds__(kThreads, 2)
norm_bwd_reduce_stream_kernel(const __grid_constant__ Maps maps, const __grid_constant__ StreamArgs a) {
  extern __shared__ uint8_t smem_raw[];
  const int P = a.tile_bytes / (2 * a.c);           // pixels per stage = pixel lanes of the consumers x 1 or 2
  const Setup u = setup(a, smem_raw);
  if ((threadIdx.x >> 5) == kConsumers / 32) {
    produce(maps, a, u, P);
    return;
  }
  if (a.has_b) {
    if (a.has_res) reduce_consume<true, true>(a, u, P);
    else reduce_consume<true, false>(a, u, P);
  } else {
    if (a.has_res) reduce_consume<false, true>(a, u, P);
    else reduce_consume<false, false>(a, u, P);
  }
}

// pass 2: dy = gamma * rstd * (dz - mean(dz) - xhat * mean(dz * xhat)) = ca * dz + cb * y + cc per channel;
// dz streamed back, or recomputed from dout (z = ca * y + shift, same rounding as pass 1)
__global__ void __launch_bounds__(kThreads, 2)
norm_bwd_apply_stream_kernel(const __grid_constant__ Maps maps, const __grid_constant__ StreamArgs a) {
  extern __shared__ uint8_t smem_raw[];
  constexpr int PX = 2, kTile = PX * kTileBytes;   // two maps per stage: two pixels per consumer and stage
  const int c = a.c, groups = c >> 3, lanes = kConsumers / groups;
  const int P = kTile / (2 * c);
  const Setup u = setup(a, smem_raw);
  if ((threadIdx.x >> 5) == kConsumers / 32) {
    produce(maps, a, u, P);
    return;
  }
  // The parameter gradients: 3 c sums over the images (folded totals) or over (image, partial slot), one warp each, spread
  // over the grid; lanes stride over the entries and fold by butterfly - a fixed order (deterministic)
  if (a.dgamma || a.dbeta || a.dalpha) {
    const int wl = threadIdx.x & 31, entries = a.tot ? a.nimg : a.nimg * a.parts;
    const float* src = a.tot ? a.tot : a.partial;
    for (int sidx = blockIdx.x * (kConsumers / 32) + (threadIdx.x >> 5); sidx < 3 * c; sidx += gridDim.x * (kConsumers / 32)) {
      const int qq = sidx / c, ch = sidx - qq * c;
      float* dst = qq == 0 ? a.dbeta : (qq == 1 ? a.dgamma : a.dalpha);
      if (!dst) continue;
      float t = 0.f;
      for (int e = wl; e < entries; e += 32) t += src[((long long)e * 3 + qq) * c + ch];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
      if (wl == 0) dst[ch] += t;
    }
  }
  const int cg = threadIdx.x % groups, lane = threadIdx.x / groups;
  const bool redo = a.recompute && (a.relu || a.alpha);
  const uint32_t stage_bytes = 2 * kTile;
  uint32_t my_off[PX];
#pragma unroll
  for (int h = 0; h < PX; ++h) my_off[h] = sw128_offset(cg, lane + h * lanes, P);
  int s = 0;
  uint32_t phase = 0;
  int r = u.r_begin;
  while (r < u.r_end) {
    const int img = r / a.hw, off = r - img * a.hw;
    const int seg = min(a.hw - off, u.r_end - r);
    const int nst = (seg + P - 1) / P;
    // mean dz, mean dz * xhat of this thread's 8 channels of the image
    float m1[8], m2[8];
    if (a.bstats) {               // folded by bwd_fold_kernel (many partial slots per image: BatchNorm)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        m1[j] = a.bstats[2 * (img * c + cg * 8 + j)];
        m2[j] = a.bstats[2 * (img * c + cg * 8 + j) + 1];
      }
    } else {                      // the few partial slots of an image in fixed order; slot loop outermost: 16 independent loads
#pragma unroll
      for (int j = 0; j < 8; ++j) m1[j] = m2[j] = 0.f;
      const float* ps = a.partial + (long long)img * a.parts * 3 * c + cg * 8;
#pragma unroll 2
      for (int k = 0; k < a.parts; ++k, ps += 3 * c) {
        const float4 u0 = *reinterpret_cast<const float4*>(ps), u1 = *reinterpret_cast<const float4*>(ps + 4);
        const float4 v0 = *reinterpret_cast<const float4*>(ps + c), v1 = *reinterpret_cast<const float4*>(ps + c + 4);
        m1[0] += u0.x; m1[1] += u0.y; m1[2] += u0.z; m1[3] += u0.w; m1[4] += u1.x; m1[5] += u1.y; m1[6] += u1.z; m1[7] += u1.w;
        m2[0] += v0.x; m2[1] += v0.y; m2[2] += v0.z; m2[3] += v0.w; m2[4] += v1.x; m2[5] += v1.y; m2[6] += v1.z; m2[7] += v1.w;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) { m1[j] *= a.inv_hw; m2[j] *= a.inv_hw; }
    }
    float2 ca[4], cb[4], cc[4], sh[4], al[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float t[10];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int ch = cg * 8 + 2 * i + e;
        const float mu = a.stats[2 * (img * c + ch)], rs = a.stats[2 * (img * c + ch) + 1];
        const float gr = (a.gamma ? a.gamma[ch] : 1.f) * rs;
        t[e] = gr;
        t[2 + e] = -gr * m2[2 * i + e] * rs;
        t[4 + e] = -gr * m1[2 * i + e] - t[2 + e] * mu;
        t[6 + e] = (a.beta ? a.beta[ch] : 0.f) - mu * gr;
        t[8 + e] = a.relu ? 0.f : (a.alpha ? a.alpha[ch] : 1.f);
      }
      ca[i] = make_float2(t[0], t[1]);
      cb[i] = make_float2(t[2], t[3]);
      cc[i] = make_float2(t[4], t[5]);
      sh[i] = make_float2(t[6], t[7]);
      al[i] = make_float2(t[8], t[9]);
    }
    bf16* optr = a.out + ((long long)r + lane) * a.out_ld + cg * 8;
    const long long ostep = (long long)P * a.out_ld;
    for (int k = 0; k < nst; ++k) {
      mbar_wait_a(u.full + 8 * s, phase);
#pragma unroll
      for (int h = 0; h < PX; ++h) {
        const uint32_t addr = u.ring + s * stage_bytes + my_off[h];
        if (k * P + lane + h * lanes < seg) {
          const uint4 D = lds128(addr), Y = lds128(addr + kTile);
          uint4 O;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            float2 d = up2(word(D, i));
            const float2 f = up2(word(Y, i));
            if (redo) {
              const float2 z = __ffma2_rn(f, ca[i], sh[i]);
              if (!(z.x > 0.f)) d.x *= al[i].x;
              if (!(z.y > 0.f)) d.y *= al[i].y;
              d = up2(pk2(d));
            }
            set_word(O, i, pk2(__ffma2_rn(ca[i], d, __ffma2_rn(cb[i], f, cc[i]))));
          }
          st_stream(optr + (long long)h * lanes * a.out_ld, O);
        }
      }
      optr += ostep;
      __syncwarp();
      if ((threadIdx.x & 31) == 0) mbar_arrive_a(u.empty + 8 * s);
      if (++s == a.stages) { s = 0; phase ^= 1; }
    }
    r += seg;
  }
}

// forward: out = act(gamma * (y - mean) * rstd + beta (+ res)), one or two maps in, one out; same ring, two pixels per
// consumer and stage
__global__ void __launch_bounds__(kThreads, 2)
norm_fwd_stream_kernel(const __grid_constant__ Maps maps, const __grid_constant__ StreamArgs a) {
  extern __shared__ uint8_t smem_raw[];
  constexpr int PX = 2, kTile = PX * kTileBytes;
  const int c = a.c, groups = c >> 3, lanes = kConsumers / groups;
  const int P = kTile / (2 * c);
  const Setup u = setup(a, smem_raw);
  if ((threadIdx.x >> 5) == kConsumers / 32) {
    produce(maps, a, u, P);
    return;
  }
  const int cg = threadIdx.x % groups, lane = threadIdx.x / groups;
  const bool has_res = a.has_res != 0;
  const uint32_t stage_bytes = a.ntensors * kTile;
  uint32_t my_off[PX];
#pragma unroll
  for (int h = 0; h < PX; ++h) my_off[h] = sw128_offset(cg, lane + h * lanes, P);
  int s = 0;
  uint32_t phase = 0;
  int r = u.r_begin;
  while (r < u.r_end) {
    const int img = r / a.hw, off = r - img * a.hw;
    const int seg = min(a.hw - off, u.r_end - r);
    const int nst = (seg + P - 1) / P;
    float2 sc[4], sh[4], al[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float t[6];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int ch = cg * 8 + 2 * i + e;
        const float mu = a.stats[2 * (img * c + ch)], rs = a.stats[2 * (img * c + ch) + 1];
        t[e] = (a.gamma ? a.gamma[ch] : 1.f) * rs;
        t[2 + e] = (a.beta ? a.beta[ch] : 0.f) - mu * t[e];
        t[4 + e] = a.relu ? 0.f : (a.alpha ? a.alpha[ch] : 1.f);
      }
      sc[i] = make_float2(t[0], t[1]);
      sh[i] = make_float2(t[2], t[3]);
      al[i] = make_float2(t[4], t[5]);
    }
    bf16* optr = a.out + ((long long)r + lane) * a.out_ld + cg * 8;
    const long long ostep = (long long)P * a.out_ld;
    for (int k = 0; k < nst; ++k) {
      mbar_wait_a(u.full + 8 * s, phase);
#pragma unroll
      for (int h = 0; h < PX; ++h) {
        const uint32_t addr = u.ring + s * stage_bytes + my_off[h];
        if (k * P + lane + h * lanes < seg) {
          const uint4 Y = lds128(addr);
          uint4 R;
          if (has_res) R = lds128(addr + kTile);
          uint4 O;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            float2 z = __ffma2_rn(up2(word(Y, i)), sc[i], sh[i]);
            if (has_res) z = __fadd2_rn(z, up2(word(R, i)));
            if (!(z.x > 0.f)) z.x *= al[i].x;
            if (!(z.y > 0.f)) z.y *= al[i].y;
            set_word(O, i, pk2(z));
          }
          st_stream(optr + (long long)h * lanes * a.out_ld, O);
        }
      }
      optr += ostep;
      __syncwarp();
      if ((threadIdx.x & 31) == 0) mbar_arrive_a(u.empty + 8 * s);
      if (++s == a.stages) { s = 0; phase ^= 1; }
    }
    r += seg;
  }
}

constexpr size_t kSmemBytes = 1024 /*align*/ + kRingBytes + kScratchBytes + 2 * kMaxStages * sizeof(uint64_t);

int encode_map(CUtensorMap* m, const void* ptr, int ld, int c, long long npix, int P, const char* what) {
  unsigned long long dims[2] = {(unsigned long long)c, (unsigned long long)npix};
  unsigned long long strides[1] = {(unsigned long long)ld * 2};
  unsigned int box[2] = {64, (unsigned int)P};
  return crfr_tmap_encode_bf16(m, ptr, 2, dims, strides, box, what);
}

int sm_count() { return crfr_sm_count(); }

// persistent grid: two CTAs per SM, at least 16 stages of work per CTA.  (A "slim" shape - 32 KB ring, four ranges per
// SM, so that one CTA fits beside a 181 KB row-streaming weight-gradient CTA of the helper stream - streams just as fast
// on its own (64 KB in flight per SM suffice) but did not shorten the step: 48.4 -> 48.8 ms, with or without a
// high-priority helper stream; the two kernels share the HBM and shared-memory pipes they are both bound by.)
int grid_for(long long total, int c) {
  const int P = kTileBytes / (2 * c);
  long long g = total / (16 * P);
  if (g < 1) g = 1;
  const int cap = 2 * sm_count();
  return (int)(g < cap ? g : cap);
}

int set_attrs() {
  static std::atomic<unsigned long long> d0{0}, d1{0}, d2{0};
  CRFR_CUDA((cudaError_t)crfr_smem_attr(norm_bwd_reduce_stream_kernel, (int)kSmemBytes, d0));
  CRFR_CUDA((cudaError_t)crfr_smem_attr(norm_bwd_apply_stream_kernel, (int)kSmemBytes, d1));
  CRFR_CUDA((cudaError_t)crfr_smem_attr(norm_fwd_stream_kernel, (int)kSmemBytes, d2));
  return CRFR_OK;
}

}  // namespace

// c a multiple of 64 (one TMA box = 64 channels = one 128-byte swizzle row), views 16-byte aligned
int crfr_norm_stream_supported(int c, long long npix, const void* const* ptrs, const int* lds, int count) {
  if (c < 64 || c > 512 || (c & 63) || npix >= (1ll << 31)) return 0;
  for (int i = 0; i < count; ++i)
    if (ptrs[i] && ((((uintptr_t)ptrs[i]) & 15) || (lds[i] & 7) || lds[i] < c)) return 0;
  return 1;
}

// partial slots per image: an image of hw pixels is covered by at most this many CTAs
int crfr_norm_stream_parts(int n, int hw, int c) {
  if (c < 64 || c > 512 || (c & 63)) return 0;
  const long long total = (long long)n * hw;
  const long long min_px = total / grid_for(total, c);   // every CTA owns at least floor(total / grid) >= 1 pixels
  return (int)((hw + min_px - 1) / min_px) + 1;
}

int crfr_norm_bwd_reduce_stream(const void* da, int da_ld, const void* db, int db_ld, const void* y, int y_ld,
                                const float* stats, const float* gamma, const float* beta, const float* alpha, int relu,
                                const void* res, int res_ld, void* dz, int dz_ld, int n, int hw, int c, float* partial,
                                cudaStream_t st) {
  const bool act = relu || alpha;
  Maps maps;
  StreamArgs a = {};
  const int ntensors = 2 + (db ? 1 : 0) + ((act && res) ? 1 : 0);
  a.tile_bytes = (ntensors <= 2 ? 2 : 1) * kTileBytes;
  const int P = a.tile_bytes / (2 * c);              // box height = pixels per stage
  const long long npix = (long long)n * hw;
  int t = 0;
  CRFR_TRY(encode_map(&maps.t[t++], da, da_ld, c, npix, P, "dout_a"));
  if (db) CRFR_TRY(encode_map(&maps.t[t++], db, db_ld, c, npix, P, "dout_b"));
  CRFR_TRY(encode_map(&maps.t[t++], y, y_ld, c, npix, P, "y"));
  if (act && res) CRFR_TRY(encode_map(&maps.t[t++], res, res_ld, c, npix, P, "residual"));
  for (int i = t; i < 4; ++i) maps.t[i] = maps.t[0];
  a.ntensors = t;
  a.ring_bytes = kRingBytes;
  a.stages = a.ring_bytes / (t * a.tile_bytes);
  if (a.stages > kMaxStages) a.stages = kMaxStages;
  a.hw = hw; a.c = c; a.nimg = n; a.parts = crfr_norm_stream_parts(n, hw, c); a.total = npix;
  a.relu = relu; a.has_b = db != nullptr; a.has_res = act && res != nullptr;
  a.stats = stats; a.gamma = gamma; a.beta = beta; a.alpha = alpha;
  a.out = (bf16*)dz; a.out_ld = dz_ld;
  a.partial = partial;
  CRFR_TRY(set_attrs());
  norm_bwd_reduce_stream_kernel<<<grid_for(npix, c), kThreads, kSmemBytes, st>>>(maps, a);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

int crfr_norm_bwd_apply_stream(const void* dsrc, int dsrc_ld, int recompute, const void* y, int y_ld, const float* stats,
                               const float* partial, int parts, const float* bstats, const float* tot,
                               const float* gamma, const float* beta,
                               const float* alpha, int relu, void* dy, int dy_ld, float* dgamma, float* dbeta,
                               float* dalpha, int n, int hw, int c, cudaStream_t st) {
  Maps maps;
  StreamArgs a = {};
  const int P = 2 * kTileBytes / (2 * c);            // two maps per stage: 8 KB tiles, two pixels per consumer
  const long long npix = (long long)n * hw;
  CRFR_TRY(encode_map(&maps.t[0], dsrc, dsrc_ld, c, npix, P, recompute ? "dout" : "dz"));
  CRFR_TRY(encode_map(&maps.t[1], y, y_ld, c, npix, P, "y"));
  maps.t[2] = maps.t[3] = maps.t[0];
  a.ntensors = 2;
  a.ring_bytes = kRingBytes;
  a.tile_bytes = 2 * kTileBytes;
  a.stages = a.ring_bytes / (2 * a.tile_bytes);
  if (a.stages > kMaxStages) a.stages = kMaxStages;
  a.hw = hw; a.c = c; a.nimg = n; a.total = npix;
  a.relu = relu; a.recompute = recompute;
  a.stats = stats; a.gamma = gamma; a.beta = beta; a.alpha = alpha;
  a.partial = const_cast<float*>(partial); a.parts = parts; a.inv_hw = 1.f / (float)hw;
  a.bstats = bstats; a.tot = tot;
  a.out = (bf16*)dy; a.out_ld = dy_ld;
  a.dgamma = dgamma; a.dbeta = dbeta; a.dalpha = dalpha;
  CRFR_TRY(set_attrs());
  norm_bwd_apply_stream_kernel<<<grid_for(npix, c), kThreads, kSmemBytes, st>>>(maps, a);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

int crfr_norm_fwd_stream(const void* y, int y_ld, const float* stats, const float* gamma, const float* beta,
                         const float* alpha, int relu, const void* res, int res_ld, void* out, int out_ld, int n, int hw,
                         int c, cudaStream_t st) {
  Maps maps;
  StreamArgs a = {};
  const int P = 2 * kTileBytes / (2 * c);
  const long long npix = (long long)n * hw;
  CRFR_TRY(encode_map(&maps.t[0], y, y_ld, c, npix, P, "y"));
  if (res) CRFR_TRY(encode_map(&maps.t[1], res, res_ld, c, npix, P, "residual"));
  else maps.t[1] = maps.t[0];
  maps.t[2] = maps.t[3] = maps.t[0];
  a.ntensors = res ? 2 : 1;
  a.ring_bytes = kRingBytes;
  a.tile_bytes = 2 * kTileBytes;
  a.stages = a.ring_bytes / (a.ntensors * a.tile_bytes);
  if (a.stages > kMaxStages) a.stages = kMaxStages;
  a.hw = hw; a.c = c; a.nimg = n; a.total = npix;
  a.relu = relu; a.has_res = res != nullptr;
  a.stats = stats; a.gamma = gamma; a.beta = beta; a.alpha = alpha;
  a.out = (bf16*)out; a.out_ld = out_ld;
  CRFR_TRY(set_attrs());
  norm_fwd_stream_kernel<<<grid_for(npix, c), kThreads, kSmemBytes, st>>>(maps, a);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}
