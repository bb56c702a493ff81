// CTA-pair (tcgen05 cta_group::2) version of the row-streaming 3x3 convolution of rowconv.cu (64 -> 64 channels,
// width 128: model/FSRnet.py:79,85 inside the coarse and decoder stacks, forward and dgrad).
//
// Why: the single-CTA kernel issues M = 128, N = 192 MMAs whose operands (4 KB of A + 6 KB of B per MMA) take most of
// the shared-memory bandwidth of the SM; measured, such an MMA costs 134 cycles in isolation (175 inside the kernel)
// against the 96 the tensor pipe needs.  A CTA pair issues ONE M = 256 MMA for two SMs: every CTA still supplies its
// own 128 rows of A, but only HALF of the B rows (the tensor cores of the pair exchange the halves), and the pair runs
// at exactly 96 cycles per K = 16 step (tools/micro/mma_bench.cu 2, profiles/r1_mma_microbench.txt).
//
// Work split: the two CTAs of a cluster walk the SAME rows of two DIFFERENT images (rank r -> image 2 * pair + r), so
// that one issuing thread can drive both with one descriptor set: identical ring positions, identical TMEM slots,
// identical (first tap, tap count) sequences at image and range edges.  The flattened (image pair, row) space is cut
// into one contiguous range per cluster exactly as rowconv.cu cuts (image, row) per CTA.
//
// B operand: with cta_group::2 rank 0 holds rows [0, N/2) and rank 1 rows [N/2, N) of the N x K matrix the MMA names
// with ONE shared-memory address.  The ky-stacked B of rowconv.cu is addressed as a sub-range (first tap j0, count cnt)
// of 192 rows, so every combination that occurs - (0,3) interior rows, (0,2) (1,2) image / range edges, (0,1) (1,1)
// (2,1) where the TMEM ring wraps - has its own per-rank half in shared memory: 320 rows x 128 B per kx, 120 KB.
//
// Protocol (everything else is rowconv.cu): own TMA producer and epilogue per CTA; rank 1's otherwise idle MMA warp
// forwards its "row landed" barrier to rank 0 (remote mbarrier arrive); rank 0 issues tcgen05.mma.cta_group::2 and
// commits with .multicast::cluster, which releases ring slots and publishes accumulator slots in BOTH CTAs; the
// epilogue warps of both CTAs return drained TMEM slots on rank 0's barrier (8 arrivals).
#include <cudaTypedefs.h>
#include <stdlib.h>

#include <atomic>

#include "common.cuh"
#include "crfr.h"
#include "internal.h"
#include "sm100.cuh"

using namespace sm100;

namespace {

constexpr int kW = 128;
constexpr int kC = 64;
constexpr int kRowBytes = 130 * 128;       // one input row with halo, 128 B per pixel
constexpr int kSlotBytes = 17 * 1024;      // ring slot stride (1024-aligned)
constexpr int kSlots = 5;
constexpr int kCaseRows = 320;             // per kx: 96 + 64 + 64 + 32 + 32 + 32 rows (see case_row)
constexpr int kKxBytes = kCaseRows * 128;
constexpr int kWeightBytes = 3 * kKxBytes;
// Epilogue layouts.  A row is a serial chain per epilogue warp (tcgen05.ld, pack, shuffle stages, stores, statistics / the
// fused normalisation-backward pass), so what bounds the epilogue is how many such chains are in flight per scheduler and
// that NOTHING spills: with ~217 KB of the SM carved out as shared memory the L1 is a few KB and a local-memory reload
// costs an L2 round trip (ncu: long-scoreboard stalls on the spilled loop counters and coefficients were 51 % of all
// samples of the first fused version).  The register file is 4 partitions of 16 K registers, warp w lives in partition
// w % 4, and setmaxnreg moves what warpgroup 0 (producer warp, MMA warp, 2 idle warps) does not need to the epilogue:
//   FUSE = 0: 2 groups of 8 warps; warp (quadrant q, half hf) owns 32 pixels x 32 channels: 104 registers, 113 us
//   FUSE = 1: 3 groups of 4 warps; warp q owns 32 pixels x 64 channels: 152 registers for the extra maps and sums
// Group g takes the output rows with orow % kGroups == g.
// Kernel variants V: 0 = plain, 1 = fused dgrad epilogue (FUSE above; 3 = the same for a normalisation without residual and
// without a second gradient, whose epilogue fits the 16-warp half-row layout).
template <int V>
struct Cfg {
  static constexpr int kGroups = V == 1 ? 3 : 2;
  static constexpr int kRowWarps = V == 1 ? 4 : 8;                    // warps that share one output row
  static constexpr int kEpiThreads = 32 * kRowWarps * kGroups;
  static constexpr int kThreads = 128 + kEpiThreads;                  // V = 0, 1, 3: 640 / 512 / 640
  // the CTA's register pool is what the launch allocates; the epilogue's share once warpgroup 0 keeps its own
  static constexpr int kRegsLaunch = (65536 / kThreads) & ~7;
  static constexpr int kRegsLean = V == 1 ? 56 : 64;
  static constexpr int kRegsEpi = ((kThreads * kRegsLaunch - 128 * kRegsLean) / kEpiThreads) & ~7;
};
constexpr int kMaxGroups = 3;
constexpr int kAccSlots = 8;
constexpr int kDone = 8;                   // ring of "input row consumed" barriers (a power of two >= kAccSlots)
constexpr int kPrefetch = 8;               // rows pulled into L2 ahead of the shared-memory ring
constexpr int kSmemBytes = kWeightBytes + kSlots * kSlotBytes + kMaxGroups * 4 * 192 * 4 /*stats*/ + kC * 4 /*bias*/ +
                           1024 /*align*/ + 512 /*barriers*/;
static_assert(kSmemBytes <= 232448, "shared memory budget");

struct PairParams {
  int n, h;              // images (even), rows per image
  int total_rows;        // (n / 2) * h: rows of the flattened (image pair, row) space
  int flip;              // 1: dgrad
  const float* bias;
  float* partial;        // InstanceNorm partials [n][parts][2][64] or nullptr
  int parts;
  bf16* dst;             // output NHWC [n][h][128][dst_ld]
  int dst_ld;
  // FUSE = 1 (dgrad only): the first pass of the backward of the normalisation that produced this convolution's input,
  // out = act(gamma * (y - mean) * rstd + beta (+ res)), runs in the epilogue: D = dgrad output (+ db),
  // dz = D * act'(z) is stored INSTEAD of the dgrad output and its per-(image, channel) sums go to partial3
  const bf16* fy; int fy_ld;
  const bf16* fb; int fb_ld;          // nullable
  const bf16* fres; int fres_ld;      // nullable
  const float* fstats; const float* fgamma; const float* fbeta; const float* falpha; int frelu;
  float* partial3;                    // [n][parts][3][64]: sum dz, sum dz * xhat, sum D * min(z, 0)
};

// first row (of the 320 per kx) of the half that belongs to the sub-range (first tap j0, cnt taps) of the stacked B
__host__ __device__ __forceinline__ int case_row(int j0, int cnt) {
  return cnt == 3 ? 0 : (cnt == 2 ? 96 + 64 * j0 : 224 + 32 * j0);
}

__device__ __forceinline__ int first_cluster_of_row(long long x, int R, int G) {
  return (int)(((x + 1) * G + R - 1) / R) - 1;
}

// input rows (with the halo rows of every segment) of a cluster's range, in load order
struct RowWalk {
  long long r, r_end;
  int h, pr, iy, iy1;
  bool valid;
  __device__ RowWalk(long long r_begin, long long r_end_, int h_) : r(r_begin), r_end(r_end_), h(h_) { start_seg(); }
  __device__ void start_seg() {
    valid = r < r_end;
    if (!valid) return;
    pr = (int)(r / h);
    const int y0 = (int)(r % h);
    const int seg = (int)min((long long)(h - y0), r_end - r);
    iy = max(y0 - 1, 0);
    iy1 = min(y0 + seg, h - 1);
    r += seg;
  }
  __device__ void next() {
    if (++iy > iy1) start_seg();
  }
};

// ---- cluster / cta_group::2 primitives ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_rank(const void* local, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(local)), "r"(rank));
  return r;
}
// Remote arrive with the default (.release.cta) semantics, as CUTLASS' ClusterBarrier::arrive(cta_id) does.  What the
// arrivals of this kernel order is asynchronous-proxy work (TMA writes observed through complete_tx, tcgen05.ld / st
// completed by tcgen05.wait + fence::before_thread_sync), not generic-proxy stores, so no cluster-scope fence is needed;
// the .release.cluster / .acquire.cluster forms compile to MEMBAR.ALL.GPU + ERRBAR and CCTL.IVALL per arrive / wait and
// made the first version of this kernel 1.7x slower than the single-CTA one (profiles/r2_rowconv_pair_ncu.txt).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) { mbar_wait(bar, parity); }
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* slot_in_smem) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_in_smem)), "n"(512)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t addr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "n"(512) : "memory");
}
__device__ __forceinline__ void umma2_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, 1, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc)
      : "memory");
}
// arrives on the barrier at this shared-memory offset in BOTH CTAs once every MMA issued so far has completed
__device__ __forceinline__ void umma2_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((uint16_t)3)
               : "memory");
}

// bf16x2 word -> two fp32 (low half = even channel)
__device__ __forceinline__ float2 bf2(uint32_t u) { return make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xffff0000u)); }

// 16-byte read-only load that does not allocate in L1: with ~217 KB of the SM's 256 KB carved out as shared memory the L1
// is a few KB, and the epilogue's streaming reads (32 KB in flight per CTA) must not queue for lines in it
__device__ __forceinline__ uint4 ldg_stream(const bf16* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}

__device__ __forceinline__ uint32_t uw(const uint4& v, int i) { return i == 0 ? v.x : (i == 1 ? v.y : (i == 2 ? v.z : v.w)); }

// 12 pair MMAs of one input row into one destination window: 3 kx shifts x 4 K steps.  The descriptors differ only in
// their low word (start address), so the issue loop is two 32-bit adds and one UTCHMMA per MMA: the issuing warp is the
// one serial resource of the kernel (230 instructions per row in the first version = 1 300 of 2 200 cycles per row).
__device__ __forceinline__ void umma2_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %3};\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "setp.ne.b32 p, 1, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %4, p;\n\t}" ::"r"(d_tmem),
      "r"(a_lo), "r"(b_lo), "r"(desc_hi), "r"(idesc)
      : "memory");
}
__device__ __forceinline__ void issue_row(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi, uint32_t idesc) {
#pragma unroll
  for (int kx = 0; kx < 3; ++kx)
#pragma unroll
    for (int k = 0; k < 4; ++k)
      umma2_lo(d_tmem, a_lo + (uint32_t)(kx * 8 + 2 * k), b_lo + (uint32_t)(kx * (kKxBytes >> 4) + 2 * k), desc_hi, idesc);
}


// ---- epilogues ---------------------------------------------------------------------------------------------------
// The epilogue touches NO shared memory per row: the kernel is bound by shared-memory bandwidth (MMA operands 84 KB + TMA
// fill 17 KB per row).  Each warp transposes its pixels x channels in registers - a transpose of 16-byte chunks inside
// every group of 4 or 8 lanes (butterfly stages of shuffles) - after which lane j of a group holds chunk j (8 channels)
// of the group's pixels: its stores are coalesced and its per-channel sums accumulate locally.
struct EpiCtx {
  uint32_t tmem;
  uint64_t* done;
  uint64_t* acc_empty;
  float* sStat;
  const float* sBias;
  long long r_begin, r_end;
  int cid, ncl;
  uint32_t rank;
  int warp, lane;
};

// FUSE = 0: forward / dgrad, optional InstanceNorm statistics of the stored values.  2 groups of 8 warps; warp
// (quadrant q, half hf) owns the 32 pixels of TMEM lane quadrant q and 32 of the 64 channels.
template <bool FP>   // FP: fused first pass of the normalisation backward, plain form (no second gradient, no residual)
__device__ __forceinline__ void epilogue_half(const PairParams& p, const EpiCtx& cx) {
  constexpr int kGroups = Cfg<0>::kGroups;
  constexpr int NQ = FP ? 3 : 2;
  const int warp = cx.warp, lane = cx.lane, cid = cx.cid, ncl = cx.ncl;
  const uint32_t tmem = cx.tmem, rank = cx.rank;
  const int ew = warp - 4, gi = ew >> 3, hf = (ew >> 2) & 1;
  const int q = warp & 3;                   // TMEM lane quadrant this warp may read: pixels 32 q .. 32 q + 31
  const int et = (ew & 7) * 32 + lane;      // 0..255 within the group
  const int cg = lane & 3;                  // after the transpose: this lane's channel chunk (channels ch0 .. ch0 + 7) ...
  const int pg = lane >> 2;                 // ... of pixels 32 q + 4 pg + (0..3)
  const int ch0 = hf * 32 + cg * 8;
  const bool has_bias = p.bias != nullptr;
  const int bar_stat = 1 + gi;
  float* sSt = cx.sStat + gi * 768;         // [4 quadrants][NQ][64]
  const uint32_t remote_acc_empty0 = map_to_rank(&cx.acc_empty[0], 0);   // rank 0's barrier array (own one for rank 0)
  float2 as[4], aq[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) as[k] = aq[k] = make_float2(0.f, 0.f);
  // FP: coefficients of this lane's 8 channels for the current image (z = sc * y + sh, slope al for z <= 0), third sum
  float2 sc[4], sh[4], al[4], ad[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) sc[k] = sh[k] = al[k] = ad[k] = make_float2(0.f, 0.f);
  const bool f_act = FP && (p.frelu || p.falpha != nullptr);
  int orow = 0;
  int gbase = 0;              // input rows of the previous segments
  long long r = cx.r_begin;
  while (r < cx.r_end) {
    const int y0 = (int)(r % p.h), pr = (int)(r / p.h);
    const int seg = (int)min((long long)(p.h - y0), cx.r_end - r);
    const int iy0 = max(y0 - 1, 0), iy1 = min(y0 + seg, p.h - 1);
    const int n = 2 * pr + (int)rank;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (!FP) break;
      float t[6];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int ch = ch0 + 2 * k + e;
        const float mu = p.fstats[2 * (n * kC + ch)], rs = p.fstats[2 * (n * kC + ch) + 1];
        t[e] = (p.fgamma ? p.fgamma[ch] : 1.f) * rs;
        t[2 + e] = (p.fbeta ? p.fbeta[ch] : 0.f) - mu * t[e];
        t[4 + e] = p.frelu ? 0.f : (p.falpha ? p.falpha[ch] : 1.f);
      }
      sc[k] = make_float2(t[0], t[1]);
      sh[k] = make_float2(t[2], t[3]);
      al[k] = make_float2(t[4], t[5]);
    }
    for (int y = y0; y < y0 + seg; ++y, ++orow) {
      if (orow % kGroups != gi) continue;
      const int slot = orow & (kAccSlots - 1);
      const int g = gbase + (min(y + 1, iy1) - iy0);       // the input row whose MMAs complete this output row
      // this lane's 4 pixels of the row: pixel q * 32 + pg * 4 + i, channels ch0 .. ch0 + 7
      const long long pix0 = ((long long)n * p.h + y) * kW + (q * 32 + pg * 4);
      if (FP && hf == 0)   // pull the lines of y this row reads into L2 while the warp waits for the MMAs
        asm volatile("prefetch.global.L2 [%0];" ::"l"(p.fy + (((long long)n * p.h + y) * kW + (q * 32 + lane)) * p.fy_ld));
      mbar_wait(&cx.done[g & (kDone - 1)], (g / kDone) & 1);
      tc_fence_after();
      const uint32_t tcol = tmem + ((uint32_t)(q * 32) << 16) + slot * kC + hf * 32;
      uint32_t v[32];
      tmem_ld32(tcol, v);
      tmem_ld_wait();
      tmem_st32_zero(tcol);        // hand the slot back zeroed
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(remote_acc_empty0 + 8u * (uint32_t)slot);
      // + bias, round to bf16: w[4 c .. 4 c + 3] = chunk c (channels 32 hf + 8 c .. + 7) of this lane's pixel
      uint32_t w[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        const __nv_bfloat162 lo =
            __floats2bfloat162_rn(__uint_as_float(v[2 * k]) + (has_bias ? cx.sBias[hf * 32 + 2 * k] : 0.f),
                                  __uint_as_float(v[2 * k + 1]) + (has_bias ? cx.sBias[hf * 32 + 2 * k + 1] : 0.f));
        w[k] = *reinterpret_cast<const uint32_t*>(&lo);
      }
      uint4 Y[4];
      if (FP) {   // issued here (the accumulator registers are free again): the transpose below hides their L2 latency
        const bf16* yp = p.fy + pix0 * p.fy_ld + ch0;
#pragma unroll
        for (int i = 0; i < 4; ++i) Y[i] = ldg_stream(yp + (long long)i * p.fy_ld);
      }
      // 4 x 4 chunk transpose inside each group of 4 lanes: afterwards w[4 i .. 4 i + 3] = chunk cg of pixel 4 pg + i
#pragma unroll
      for (int s = 2; s >= 1; s >>= 1) {
        const bool up = (lane & s) != 0;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          if (c & s) continue;
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const uint32_t a = w[4 * c + e], b = w[4 * (c | s) + e];
            const uint32_t recv = __shfl_xor_sync(0xffffffffu, up ? a : b, s);
            w[4 * c + e] = up ? recv : a;
            w[4 * (c | s) + e] = up ? b : recv;
          }
        }
      }
      if (FP) {
        // first pass of the normalisation backward on the rounded gradient, exactly as norm_stream.cu's reduce pass:
        // z = sc * y + sh; z <= 0: ad += D * z, D *= al; dz = bf16(D) replaces the dgrad output; as += dz; aq += dz * y
#pragma unroll
        for (int i = 0; i < 4; ++i) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            float2 gd = bf2(w[4 * i + k]);
            const float2 f = bf2(uw(Y[i], k));
            if (f_act) {
              const float2 z = __ffma2_rn(f, sc[k], sh[k]);
              if (!(z.x > 0.f)) { ad[k].x = fmaf(gd.x, z.x, ad[k].x); gd.x *= al[k].x; }
              if (!(z.y > 0.f)) { ad[k].y = fmaf(gd.y, z.y, ad[k].y); gd.y *= al[k].y; }
            }
            const __nv_bfloat162 pb = __floats2bfloat162_rn(gd.x, gd.y);
            const uint32_t wd = *reinterpret_cast<const uint32_t*>(&pb);
            w[4 * i + k] = wd;
            const float2 d = bf2(wd);
            as[k] = __fadd2_rn(as[k], d);
            aq[k] = __ffma2_rn(d, f, aq[k]);
          }
        }
      }
      bf16* line = p.dst + pix0 * p.dst_ld + ch0;
#pragma unroll
      for (int i = 0; i < 4; ++i)
        *reinterpret_cast<uint4*>(line + (long long)i * p.dst_ld) = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
      if (!FP && p.partial) {
        // per-channel sums of the stored (rounded) values: this lane's 8 channels over its 4 pixels, packed fp32x2
#pragma unroll
        for (int i = 0; i < 4; ++i) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float2 f = bf2(w[4 * i + k]);
            as[k] = __fadd2_rn(as[k], f);
            aq[k] = __ffma2_rn(f, f, aq[k]);
          }
        }
      }
    }
    if (FP || p.partial) {
      // end of this CTA's rows of image n: fold the group's pixel lanes in fixed order (8 lanes by shuffle, the 4
      // quadrant warps through shared memory) and publish the group's partial in its own slot - also when it is all zero
#pragma unroll
      for (int o = 4; o <= 16; o <<= 1) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          as[k].x += __shfl_xor_sync(0xffffffffu, as[k].x, o);  as[k].y += __shfl_xor_sync(0xffffffffu, as[k].y, o);
          aq[k].x += __shfl_xor_sync(0xffffffffu, aq[k].x, o);  aq[k].y += __shfl_xor_sync(0xffffffffu, aq[k].y, o);
          if (FP) { ad[k].x += __shfl_xor_sync(0xffffffffu, ad[k].x, o);  ad[k].y += __shfl_xor_sync(0xffffffffu, ad[k].y, o); }
        }
      }
      named_bar_sync(bar_stat, 256);   // previous use of the scratch is over
      if (lane < 4) {
        float* d0 = sSt + (q * NQ + 0) * kC + ch0;
        float* d1 = sSt + (q * NQ + 1) * kC + ch0;
        float* d2 = sSt + (q * NQ + 2) * kC + ch0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          d0[2 * k] = as[k].x; d0[2 * k + 1] = as[k].y;
          d1[2 * k] = aq[k].x; d1[2 * k + 1] = aq[k].y;
          if (FP) { d2[2 * k] = ad[k].x; d2[2 * k + 1] = ad[k].y; }
        }
      }
      named_bar_sync(bar_stat, 256);
      const int b0 = first_cluster_of_row((long long)pr * p.h, p.total_rows, ncl);
      const int part = cid - b0;
      if (FP) {
        float* dst = p.partial3 + ((long long)n * p.parts + kGroups * part + gi) * 3 * kC;
        if (et < kC) {
          float t[3];
#pragma unroll
          for (int j = 0; j < 3; ++j)
            t[j] = (sSt[j * kC + et] + sSt[(3 + j) * kC + et]) + (sSt[(6 + j) * kC + et] + sSt[(9 + j) * kC + et]);
          // centre and scale: sum(dz * xhat) = rstd * (sum(dz * y) - mean * sum(dz))
          const float mu = p.fstats[2 * (n * kC + et)], rs = p.fstats[2 * (n * kC + et) + 1];
          dst[et] = t[0];
          dst[kC + et] = (t[1] - mu * t[0]) * rs;
          dst[2 * kC + et] = t[2];
        }
        if (y0 + seg == p.h && gi == 0)   // last cluster of this image: the unused slots must read as zero
          for (int z = kGroups * (part + 1); z < p.parts; ++z)
            for (int j = et; j < 3 * kC; j += 256) p.partial3[((long long)n * p.parts + z) * 3 * kC + j] = 0.f;
      } else {
        float* dst = p.partial + ((long long)n * p.parts + kGroups * part + gi) * 2 * kC;
        if (et < 2 * kC) dst[et] = (sSt[et] + sSt[128 + et]) + (sSt[256 + et] + sSt[384 + et]);
        if (y0 + seg == p.h && gi == 0)   // last cluster of this image: the unused slots must read as zero
          for (int z = kGroups * (part + 1); z < p.parts; ++z)
            if (et < 2 * kC) p.partial[((long long)n * p.parts + z) * 2 * kC + et] = 0.f;
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) as[k] = aq[k] = ad[k] = make_float2(0.f, 0.f);
    }
    gbase += iy1 - iy0 + 1;
    r += seg;
  }
}

// FUSE = 1 (dgrad): the first pass of the normalisation backward on the rounded dgrad output, exactly as norm_stream.cu's
// reduce pass: D = dgrad (+ db); z = sc * y + sh (+ res); z <= 0: ad += D * z, D *= al; dz = bf16(D) is stored in place of
// the dgrad output; as += dz; aq += dz * y.  3 groups of 4 warps; warp q owns 32 pixels x 64 channels.
__device__ __forceinline__ void epilogue_row(const PairParams& p, const EpiCtx& cx) {
  constexpr int kGroups = Cfg<1>::kGroups;
  constexpr int NQ = 3;
  const int warp = cx.warp, lane = cx.lane;
  const uint32_t tmem = cx.tmem;
  const int ew = warp - 4, gi = ew >> 2;
  const int q = warp & 3;                   // TMEM lane quadrant this warp may read: pixels 32 q .. 32 q + 31
  const int et = (ew & 3) * 32 + lane;      // 0..127 within the group
  const int cg = lane & 7;                  // after the transpose: this lane's channel chunk (channels 8 cg .. 8 cg + 7) ...
  const int pg = lane >> 3;                 // ... of pixels 32 q + 8 pg + (0..7)
  const int bar_stat = 1 + gi;
  float* sSt = cx.sStat + gi * 768;         // [4 warps][NQ][64]
  const uint32_t remote_acc_empty0 = map_to_rank(&cx.acc_empty[0], 0);
  const bool f_act = p.frelu || p.falpha != nullptr;
  const bool f_b = p.fb != nullptr, f_res = f_act && p.fres != nullptr;
  // coefficients of this lane's 8 channels for the current image (z = sc * y + sh, slope al for z <= 0); sums
  float2 sc[4], sh[4], al[4], as[4], aq[4], ad[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) sc[k] = sh[k] = al[k] = as[k] = aq[k] = ad[k] = make_float2(0.f, 0.f);
  int orow = 0, og = 0;       // og = orow % kGroups
  int gbase = 0;              // input rows of the previous segments
  long long r = cx.r_begin;
  while (r < cx.r_end) {
    const int y0 = (int)(r % p.h), pr = (int)(r / p.h);
    const int seg = (int)min((long long)(p.h - y0), cx.r_end - r);
    const int iy0 = max(y0 - 1, 0), iy1 = min(y0 + seg, p.h - 1);
    const int n = 2 * pr + (int)cx.rank;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float t[6];
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int ch = cg * 8 + 2 * k + e;
        const float mu = p.fstats[2 * (n * kC + ch)], rs = p.fstats[2 * (n * kC + ch) + 1];
        t[e] = (p.fgamma ? p.fgamma[ch] : 1.f) * rs;
        t[2 + e] = (p.fbeta ? p.fbeta[ch] : 0.f) - mu * t[e];
        t[4 + e] = p.frelu ? 0.f : (p.falpha ? p.falpha[ch] : 1.f);
      }
      sc[k] = make_float2(t[0], t[1]);
      sh[k] = make_float2(t[2], t[3]);
      al[k] = make_float2(t[4], t[5]);
    }
    for (int y = y0; y < y0 + seg; ++y, ++orow, og = (og + 1 == kGroups) ? 0 : og + 1) {
      if (og != gi) continue;
      const int slot = orow & (kAccSlots - 1);
      const int g = gbase + (min(y + 1, iy1) - iy0);       // the input row whose MMAs complete this output row
      // element offset of this lane's 8 pixels of the row (pixel q * 32 + pg * 8 + i), before the per-map ld
      const long long pix0 = ((long long)n * p.h + y) * kW + (q * 32 + pg * 8);
      // pull the lines the fused pass reads into L2 while this warp waits for the MMAs (lane cg: pixel cg of its 8)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(p.fy + (pix0 + cg) * p.fy_ld));
      if (f_b) asm volatile("prefetch.global.L2 [%0];" ::"l"(p.fb + (pix0 + cg) * p.fb_ld));
      if (f_res) asm volatile("prefetch.global.L2 [%0];" ::"l"(p.fres + (pix0 + cg) * p.fres_ld));
      mbar_wait(&cx.done[g & (kDone - 1)], (g / kDone) & 1);
      tc_fence_after();
      // two halves of 32 accumulator columns, each packed to bf16 before the next is read (bounds the live registers):
      // w[4 c .. 4 c + 3] = chunk c (channels 8 c .. 8 c + 7) of this lane's pixel
      uint32_t w[32];
      {
        uint32_t v[32];
        tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + slot * kC, v);
        tmem_ld_wait();
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const __nv_bfloat162 lo = __floats2bfloat162_rn(__uint_as_float(v[2 * k]), __uint_as_float(v[2 * k + 1]));
          w[k] = *reinterpret_cast<const uint32_t*>(&lo);
        }
        tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + slot * kC + 32, v);
        tmem_ld_wait();
        tmem_st32_zero(tmem + ((uint32_t)(q * 32) << 16) + slot * kC);        // hand the slot back zeroed
        tmem_st32_zero(tmem + ((uint32_t)(q * 32) << 16) + slot * kC + 32);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(remote_acc_empty0 + 8u * (uint32_t)slot);
#pragma unroll
        for (int k = 0; k < 16; ++k) {
          const __nv_bfloat162 hi = __floats2bfloat162_rn(__uint_as_float(v[2 * k]), __uint_as_float(v[2 * k + 1]));
          w[16 + k] = *reinterpret_cast<const uint32_t*>(&hi);
        }
      }
      // 8 x 8 chunk transpose inside each group of 8 lanes: afterwards w[4 i .. 4 i + 3] = chunk cg of pixel 8 pg + i
#pragma unroll
      for (int s = 4; s >= 1; s >>= 1) {
        const bool up = (lane & s) != 0;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          if (c & s) continue;
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const uint32_t a = w[4 * c + e], b = w[4 * (c | s) + e];
            const uint32_t recv = __shfl_xor_sync(0xffffffffu, up ? a : b, s);
            w[4 * c + e] = up ? recv : a;
            w[4 * (c | s) + e] = up ? b : recv;
          }
        }
      }
      const bf16* yp = p.fy + pix0 * p.fy_ld + cg * 8;
      const bf16* bp = p.fb + pix0 * p.fb_ld + cg * 8;
      const bf16* rp = p.fres + pix0 * p.fres_ld + cg * 8;
      bf16* line = p.dst + pix0 * p.dst_ld + cg * 8;
#pragma unroll
      for (int h2 = 0; h2 < 4; ++h2) {   // four quarters of 2 pixels: bounds the registers of the maps in flight
        uint4 Yv[2], Bv[2], Rv[2];
#pragma unroll
        for (int i = 0; i < 2; ++i) Yv[i] = ldg_stream(yp + (long long)(2 * h2 + i) * p.fy_ld);
        if (f_b) {
#pragma unroll
          for (int i = 0; i < 2; ++i) Bv[i] = ldg_stream(bp + (long long)(2 * h2 + i) * p.fb_ld);
        }
        if (f_res) {
#pragma unroll
          for (int i = 0; i < 2; ++i) Rv[i] = ldg_stream(rp + (long long)(2 * h2 + i) * p.fres_ld);
        }
#pragma unroll
        for (int i4 = 0; i4 < 2; ++i4) {
          const int i = 2 * h2 + i4;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            float2 gd = bf2(w[4 * i + k]);
            if (f_b) gd = __fadd2_rn(gd, bf2(uw(Bv[i4], k)));
            const float2 f = bf2(uw(Yv[i4], k));
            if (f_act) {
              float2 z = __ffma2_rn(f, sc[k], sh[k]);
              if (f_res) z = __fadd2_rn(z, bf2(uw(Rv[i4], k)));
              if (!(z.x > 0.f)) { ad[k].x = fmaf(gd.x, z.x, ad[k].x); gd.x *= al[k].x; }
              if (!(z.y > 0.f)) { ad[k].y = fmaf(gd.y, z.y, ad[k].y); gd.y *= al[k].y; }
            }
            const __nv_bfloat162 pb = __floats2bfloat162_rn(gd.x, gd.y);
            const uint32_t wd = *reinterpret_cast<const uint32_t*>(&pb);
            w[4 * i + k] = wd;
            const float2 d = bf2(wd);
            as[k] = __fadd2_rn(as[k], d);
            aq[k] = __ffma2_rn(d, f, aq[k]);
          }
          *reinterpret_cast<uint4*>(line + (long long)i * p.dst_ld) = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
        }
      }
    }
    // end of this CTA's rows of image n: fold the group's pixel lanes in fixed order (4 lanes by shuffle, the 4 warps
    // through shared memory) and publish the group's partial in its own slot - also when it is all zero
#pragma unroll
    for (int o = 8; o <= 16; o <<= 1) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        as[k].x += __shfl_xor_sync(0xffffffffu, as[k].x, o);  as[k].y += __shfl_xor_sync(0xffffffffu, as[k].y, o);
        aq[k].x += __shfl_xor_sync(0xffffffffu, aq[k].x, o);  aq[k].y += __shfl_xor_sync(0xffffffffu, aq[k].y, o);
        ad[k].x += __shfl_xor_sync(0xffffffffu, ad[k].x, o);  ad[k].y += __shfl_xor_sync(0xffffffffu, ad[k].y, o);
      }
    }
    named_bar_sync(bar_stat, 128);   // previous use of the scratch is over
    if (lane < 8) {
      float* d0 = sSt + ((ew & 3) * NQ + 0) * kC + cg * 8;
      float* d1 = sSt + ((ew & 3) * NQ + 1) * kC + cg * 8;
      float* d2 = sSt + ((ew & 3) * NQ + 2) * kC + cg * 8;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        d0[2 * k] = as[k].x; d0[2 * k + 1] = as[k].y;
        d1[2 * k] = aq[k].x; d1[2 * k + 1] = aq[k].y;
        d2[2 * k] = ad[k].x; d2[2 * k + 1] = ad[k].y;
      }
    }
    named_bar_sync(bar_stat, 128);
    const int b0 = first_cluster_of_row((long long)pr * p.h, p.total_rows, cx.ncl);
    const int part = cx.cid - b0;
    float* dst = p.partial3 + ((long long)n * p.parts + kGroups * part + gi) * 3 * kC;
    if (et < kC) {
      float t[3];
#pragma unroll
      for (int j = 0; j < 3; ++j)
        t[j] = (sSt[j * kC + et] + sSt[(3 + j) * kC + et]) + (sSt[(6 + j) * kC + et] + sSt[(9 + j) * kC + et]);
      // centre and scale: sum(dz * xhat) = rstd * (sum(dz * y) - mean * sum(dz))
      const float mu = p.fstats[2 * (n * kC + et)], rs = p.fstats[2 * (n * kC + et) + 1];
      dst[et] = t[0];
      dst[kC + et] = (t[1] - mu * t[0]) * rs;
      dst[2 * kC + et] = t[2];
    }
    if (y0 + seg == p.h && gi == 0)   // last cluster of this image: the unused slots must read as zero
      for (int z = kGroups * (part + 1); z < p.parts; ++z)
        for (int j = et; j < 3 * kC; j += 128) p.partial3[((long long)n * p.parts + z) * 3 * kC + j] = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) as[k] = aq[k] = ad[k] = make_float2(0.f, 0.f);
    gbase += iy1 - iy0 + 1;
    r += seg;
  }
}

template <int FUSE>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(Cfg<FUSE>::kThreads, 1)
rowconv_pair_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW, PairParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* sW = base;
  uint8_t* sRing = base + kWeightBytes;
  float* sStat = (float*)(sRing + kSlots * kSlotBytes);   // [kGroups][4 warps][2 or 3][64]
  float* sBias = sStat + kMaxGroups * 4 * 192;
  uint64_t* full = (uint64_t*)(sBias + kC);        // [kSlots] this CTA's input row has landed
  uint64_t* peer_full = full + kSlots;             // [kSlots] rank 0 only: rank 1's row has landed
  uint64_t* done = peer_full + kSlots;             // [kDone] the pair's MMAs of input row g are complete (multicast commit):
                                                   //         frees ring slot g % kSlots AND completes an output row
  uint64_t* w_full = done + kDone;
  uint64_t* peer_w_full = w_full + 1;
  uint64_t* acc_empty = peer_w_full + 1;           // [kAccSlots] rank 0 only: the epilogue warps of a row in both CTAs
  uint32_t* tmem_slot = (uint32_t*)(acc_empty + kAccSlots);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_rank();
  const int cid = blockIdx.x >> 1, ncl = gridDim.x >> 1;
  if (threadIdx.x == 0) {
    for (int s = 0; s < kSlots; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&peer_full[s], 1);
    }
    for (int b = 0; b < kDone; ++b) mbar_init(&done[b], 1);
    mbar_init(w_full, 1);
    mbar_init(peer_w_full, 1);
    for (int b = 0; b < kAccSlots; ++b) mbar_init(&acc_empty[b], 2 * Cfg<FUSE>::kRowWarps);
    fence_barrier_init();
    prefetch_tmap(&tmX);
    prefetch_tmap(&tmW);
  }
  if (threadIdx.x >= 64 && threadIdx.x < 64 + kC) sBias[threadIdx.x - 64] = p.bias ? p.bias[threadIdx.x - 64] : 0.f;
  if (warp == 1) tmem_alloc_pair(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  if (warp >= 4 && warp < 8) {   // all accumulators start at zero: every MMA of this kernel accumulates
    for (int c = 0; c < 512; c += 32) tmem_st32_zero(tmem + ((uint32_t)((warp & 3) * 32) << 16) + c);
    tmem_st_wait();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // barriers initialised and TMEM zeroed in BOTH CTAs before any remote arrive / pair MMA
  tc_fence_after();

  // contiguous range of flattened (image pair, row) rows for this cluster; this CTA works on image 2 * pair + rank.
  // (Computed after setmaxnreg in each branch: what is live across it is spilled to local memory and reloaded in the loops.)
  if (warp < 4) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(Cfg<FUSE>::kRegsLean));
  const long long r_begin = (long long)p.total_rows * cid / ncl;
  const long long r_end = (long long)p.total_rows * (cid + 1) / ncl;
  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (both CTAs)
    const bool leader = elect_one();
    if (leader) {
      mbar_expect_tx(w_full, kWeightBytes);
      const int hi = (int)rank;                        // 0: lower half of the stacked rows, 1: upper half
      for (int kx = 0; kx < 3; ++kx)
        for (int cnt = 1; cnt <= 3; ++cnt)
          for (int j0 = 0; j0 + cnt <= 3; ++j0) {
            const int half = 32 * cnt;                         // rows this CTA holds of the 64 * cnt stacked rows
            const int start = 64 * j0 + hi * half;
            for (int i = 0; i < half; i += 32) {
              const int R = start + i, j = R >> 6, co0 = R & 63;
              const int tap = (2 - j) * 3 + kx;                // stacked block j maps input row r to output row r-1+j
              tma_load_2d(sW + kx * kKxBytes + (case_row(j0, cnt) + i) * 128, &tmW, w_full, 0,
                          (p.flip ? 8 - tap : tap) * kC + co0);
            }
          }
    }
    // (An L2 prefetch cursor running 8-12 rows ahead of the ring - cp.async.bulk.prefetch.tensor or prefetch.global.L2 from
    // this warp's lanes - made the kernel 3-6 us SLOWER once the issuing warp was no longer the bottleneck: the launch moves
    // 537 MB in ~120 us, i.e. the memory system is already at 4.4 TB/s of mixed read / write traffic.)
    RowWalk ld(r_begin, r_end, p.h);
    for (int g = 0; ld.valid; ++g, ld.next()) {
      const int s = g % kSlots;
      if (g >= kSlots) mbar_wait(&done[(g - kSlots) % kDone], ((g - kSlots) / kDone) & 1);   // row g - kSlots consumed
      if (leader) {
        mbar_expect_tx(&full[s], kRowBytes);
        tma_load_4d(sRing + s * kSlotBytes, &tmX, &full[s], 0, -1, ld.iy, 2 * ld.pr + (int)rank);
      }
    }
  } else if (warp == 1 && rank != 0) {
    // ------------------------------------------------------------------ rank 1: forward "landed" to the issuing CTA
    const uint32_t remote_w = map_to_rank(peer_w_full, 0);
    const uint32_t remote_full0 = map_to_rank(&peer_full[0], 0);
    mbar_wait(w_full, 0);
    if (lane == 0) mbar_arrive_cluster(remote_w);
    RowWalk ld(r_begin, r_end, p.h);
    for (int g = 0; ld.valid; ++g, ld.next()) {
      const int s = g % kSlots;
      mbar_wait(&full[s], (g / kSlots) & 1);
      if (lane == 0) mbar_arrive_cluster(remote_full0 + 8u * (uint32_t)s);
      __syncwarp();
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ rank 0: MMA issuer for the pair
    // One warp issues every MMA of two SMs; whatever it executes between two rows is time the tensor pipes may idle,
    // so all per-row state is kept incrementally (no divisions), the descriptors are built from precomputed low words,
    // and ONE commit per input row serves both the producers (ring slot free) and the epilogues (output row complete).
    const bool leader = elect_one();
    const uint64_t wdesc0 = make_smem_desc_sw128(smem_u32(sW), 16, 1024);
    const uint64_t rdesc0 = make_smem_desc_sw128(smem_u32(sRing), 16, 1024);
    const uint32_t desc_hi = (uint32_t)(wdesc0 >> 32), w_lo = (uint32_t)wdesc0, ring_lo = (uint32_t)rdesc0;
    const uint32_t idesc1 = make_idesc_bf16(256, kC, 0, 0), idesc2 = make_idesc_bf16(256, 2 * kC, 0, 0),
                   idesc3 = make_idesc_bf16(256, 3 * kC, 0, 0);
    mbar_wait(w_full, 0);
    mbar_wait_cluster(peer_w_full, 0);
    int sg = 0;                 // ring slot of the current input row, and its parity
    uint32_t sph = 0;
    int dg = 0;                 // done barrier of the current input row (g % kDone)
    int o_touched = 0;          // output rows [0, o_touched) of this cluster have been claimed (their slot waited for)
    int obase = 0;
    long long r = r_begin;
    while (r < r_end) {
      const int y0 = (int)(r % p.h);
      const int seg = (int)min((long long)(p.h - y0), r_end - r);
      const int iy0 = max(y0 - 1, 0), iy1 = min(y0 + seg, p.h - 1);
      for (int iy = iy0; iy <= iy1; ++iy) {
        // output rows fed by this input row, clipped to the segment
        const int t_lo = max(iy - 1, y0), t_hi = min(iy + 1, y0 + seg - 1);
        const int o_lo = obase + (t_lo - y0), o_hi = obase + (t_hi - y0);
        while (o_touched <= o_hi) {   // first touch: both epilogues have drained (and zeroed) the slot
          mbar_wait_cluster(&acc_empty[o_touched & (kAccSlots - 1)], ((o_touched >> 3) & 1) ^ 1);
          ++o_touched;
        }
        const int slot = o_lo & (kAccSlots - 1);
        const int cnt = o_hi - o_lo + 1;
        const int j0 = t_lo - (iy - 1);
        mbar_wait(&full[sg], sph);
        mbar_wait_cluster(&peer_full[sg], sph);
        tc_fence_after();
        const uint32_t a_lo = ring_lo + (uint32_t)(sg * (kSlotBytes >> 4));
        if (leader) {
          if (slot + cnt <= kAccSlots) {
            issue_row(tmem + slot * kC, a_lo, w_lo + (uint32_t)(case_row(j0, cnt) * 8), desc_hi,
                      cnt == 3 ? idesc3 : (cnt == 2 ? idesc2 : idesc1));
          } else {   // the window wraps around the TMEM ring: the part up to the end, then the remainder from column 0
            const int ca = kAccSlots - slot, cb = cnt - ca;
            issue_row(tmem + slot * kC, a_lo, w_lo + (uint32_t)(case_row(j0, ca) * 8), desc_hi, ca == 2 ? idesc2 : idesc1);
            issue_row(tmem, a_lo, w_lo + (uint32_t)(case_row(j0 + ca, cb) * 8), desc_hi, cb == 2 ? idesc2 : idesc1);
          }
        }
        if (leader) umma2_commit(&done[dg]);
        __syncwarp();
        if (++sg == kSlots) { sg = 0; sph ^= 1; }
        dg = (dg + 1) & (kDone - 1);
      }
      obase += seg;
      r += seg;
    }
  }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(Cfg<FUSE>::kRegsEpi));
    const long long r_begin = (long long)p.total_rows * cid / ncl;
    const long long r_end = (long long)p.total_rows * (cid + 1) / ncl;
    const EpiCtx cx = {tmem, done, acc_empty, sStat, sBias, r_begin, r_end, cid, ncl, rank, warp, lane};
    if (FUSE == 0 || FUSE == 3) epilogue_half<FUSE == 3>(p, cx);
    else epilogue_row(p, cx);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // nobody frees TMEM or leaves while the peer may still issue MMAs / remote arrives
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair(*tmem_slot);   // read again: a register held across the setmaxnreg above may be spilled
  }
}

int clusters_for(int total_rows) {
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int cl = sms / 2;
  return cl < total_rows ? cl : total_rows;
}

// partial slots per image: clusters that can share an image x 2 epilogue groups
int parts_for(int pairs, int h, int groups) {
  const int total = pairs * h, grid = clusters_for(total);
  const int min_rows = total / grid;
  return groups * ((h + min_rows - 1) / min_rows + 1);
}

}  // namespace

int crfr_rowconv_pair_supported(int n, int h) { return n >= 2 && (n & 1) == 0 && h >= 1; }

size_t crfr_rowconv_pair_ws_bytes(int n, int h) {
  if (!crfr_rowconv_pair_supported(n, h)) return 0;
  return sizeof(float) * (size_t)n * parts_for(n / 2, h, Cfg<0>::kGroups) * 2 * kC + 256;
}

int crfr_rowconv_pair_parts(int n, int h, int plain) {
  return crfr_rowconv_pair_supported(n, h) ? parts_for(n / 2, h, plain ? Cfg<3>::kGroups : Cfg<1>::kGroups) : 0;
}

// Same contract as crfr_rowconv (rowconv.cu); n must be even.  fuse (dgrad only, see PairParams): the epilogue stores
// dz = (dgrad (+ db)) * act'(z) instead of the dgrad output and writes the partial sums of the normalisation backward's
// first pass to fuse->partial ([n][crfr_rowconv_pair_parts(n, h)][3][64] floats, to be folded by bwd_fold_kernel).
int crfr_rowconv_pair(const void* src, int src_ld, int n, int h, const void* w_packed, int flip, const float* bias,
                      void* dst, int dst_ld, float* stats, float eps, void* ws, size_t ws_bytes, cudaStream_t st,
                      const crfr_rowconv_fuse* fuse) {
  CRFR_CHECK_ARG(crfr_rowconv_pair_supported(n, h), "rowconv_pair: needs an even number of images");
  CRFR_CHECK_ARG(((uintptr_t)src & 15) == 0 && ((uintptr_t)dst & 15) == 0 && ((uintptr_t)w_packed & 15) == 0 &&
                     (src_ld & 7) == 0 && (dst_ld & 7) == 0,
                 "rowconv_pair: pointers must be 16B aligned and ld a multiple of 8");
  if (fuse) {
    CRFR_CHECK_ARG(flip && !stats && fuse->y && fuse->stats && fuse->partial, "rowconv_pair: fused pass needs dgrad, y, stats");
    CRFR_CHECK_ARG(((uintptr_t)fuse->y & 15) == 0 && ((uintptr_t)fuse->db & 15) == 0 && ((uintptr_t)fuse->res & 15) == 0 &&
                       ((fuse->y_ld | fuse->db_ld | fuse->res_ld) & 7) == 0,
                   "rowconv_pair: fused maps must be 16B aligned and ld a multiple of 8");
  }
  CUtensorMap tmX, tmW;
  {
    unsigned long long dims[4] = {(unsigned long long)kC, (unsigned long long)kW, (unsigned long long)h, (unsigned long long)n};
    unsigned long long strides[3] = {(unsigned long long)src_ld * 2, (unsigned long long)kW * src_ld * 2, (unsigned long long)h * kW * src_ld * 2};
    unsigned int box[4] = {64, 130, 1, 1};
    CRFR_TRY(crfr_tmap_encode_bf16(&tmX, src, 4, dims, strides, box, "activation"));
  }
  {
    unsigned long long dims[2] = {64, 9 * 64};
    unsigned long long strides[1] = {128};
    unsigned int box[2] = {64, 32};
    CRFR_TRY(crfr_tmap_encode_bf16(&tmW, w_packed, 2, dims, strides, box, "weights"));
  }
  static std::atomic<unsigned long long> attr0{0}, attr1{0}, attr3{0};
  CRFR_CUDA((cudaError_t)crfr_smem_attr(rowconv_pair_kernel<3>, kSmemBytes, attr3));
  CRFR_CUDA((cudaError_t)crfr_smem_attr(rowconv_pair_kernel<0>, kSmemBytes, attr0));
  CRFR_CUDA((cudaError_t)crfr_smem_attr(rowconv_pair_kernel<1>, kSmemBytes, attr1));
  PairParams p = {};
  p.n = n; p.h = h; p.total_rows = (n / 2) * h; p.flip = flip;
  p.bias = bias;
  p.partial = nullptr;
  p.parts = 0;
  p.dst = (bf16*)dst;
  p.dst_ld = dst_ld;

  if (stats) {
    const size_t need = crfr_rowconv_pair_ws_bytes(n, h);
    if (!ws || ws_bytes < need) {
      crfr_set_error("rowconv_pair: workspace %zu < %zu", ws_bytes, need);
      return CRFR_EWORKSPACE;
    }
    p.partial = (float*)ws;
    p.parts = parts_for(n / 2, h, Cfg<0>::kGroups);
  }
  if (fuse) {
    p.fy = (const bf16*)fuse->y; p.fy_ld = fuse->y_ld;
    p.fb = (const bf16*)fuse->db; p.fb_ld = fuse->db_ld;
    p.fres = (const bf16*)fuse->res; p.fres_ld = fuse->res_ld;
    p.fstats = fuse->stats; p.fgamma = fuse->gamma; p.fbeta = fuse->beta; p.falpha = fuse->alpha; p.frelu = fuse->relu;
    p.partial3 = fuse->partial;
    if (!fuse->db && !fuse->res) {   // plain form: 16-warp half-row epilogue
      p.parts = parts_for(n / 2, h, Cfg<3>::kGroups);
      rowconv_pair_kernel<3><<<2 * clusters_for(p.total_rows), Cfg<3>::kThreads, kSmemBytes, st>>>(tmX, tmW, p);
    } else {
      p.parts = parts_for(n / 2, h, Cfg<1>::kGroups);
      rowconv_pair_kernel<1><<<2 * clusters_for(p.total_rows), Cfg<1>::kThreads, kSmemBytes, st>>>(tmX, tmW, p);
    }
  } else {
    rowconv_pair_kernel<0><<<2 * clusters_for(p.total_rows), Cfg<0>::kThreads, kSmemBytes, st>>>(tmX, tmW, p);
  }
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  if (stats) CRFR_TRY(crfr_norm_finalize(p.partial, n, p.parts, h * kW, kC, eps, stats, st));
  return CRFR_OK;
}
