// tcgen05 / TMEM implicit-GEMM convolution engine for sm_100a, fed by TMA.
//
// Forward / dgrad (3x3, stride 1, pad 1, channels in multiples of 64), NHWC bf16:
//   one CTA computes a tile of 128 output pixels x N output channels.  The 128 pixels are a TMA box
//   (64 channels x bw x bh x bn) of the NHWC activation tensor, so the im2col gather of tap (ky,kx) is just the
//   same box shifted by (kx-1, ky-1); out-of-bounds elements are zero-filled by the TMA unit (= the padding).
//   K loop = taps x (Cin/64): per step one 16 KB activation tile (A, K-major, SWIZZLE_128B) and one N x 64 weight
//   tile (B, K-major) land in a 3-4 stage smem ring (mbarrier full/empty), one elected thread issues 4
//   tcgen05.mma (M=128, N, K=16) per step into a TMEM accumulator, and 4 epilogue warps drain TMEM with
//   tcgen05.ld, add the bias, round to bf16 and store NHWC rows.
//   dgrad is the same kernel on dY with flipped tap offsets and [tap][cin][cout] weights.
// Wgrad: D[(kx,ci)][co] = sum_pixels X[p + tap][ci] * dY[p][co]: both operands are MN-major views of the same
//   NHWC tiles (pixels are the K dimension); two kx taps are stacked in M=128 through the leading-byte-offset of
//   the smem descriptor; each pixel split stores its fp32 partial result to its own [tap][cin][cout] slice and one
//   pass sums the slices in split order (no float atomics: the weight gradient is the same bits on every run).
//
// ref: the nn.Conv2d sites of model/FSRnet.py (:79,85,110,114,351,387,411,432) that carry 99 % of the FLOPs.
#include <cudaTypedefs.h>
#include <stdlib.h>

#include "common.cuh"
#include "crfr.h"
#include "internal.h"
#include "sm100.cuh"

using namespace sm100;

namespace {

// ------------------------------------------------------------------------------------------------
// host: tensor maps (tmap.cu)
// ------------------------------------------------------------------------------------------------
// NHWC bf16 activation view [n][h][w][c] with per-pixel stride ld; box = (64, bw, bh, bn), SWIZZLE_128B
int make_act_map(CUtensorMap* m, const void* ptr, int n, int h, int w, int c, int ld, int bw, int bh, int bn) {
  const unsigned long long dims[4] = {(unsigned long long)c, (unsigned long long)w, (unsigned long long)h,
                                      (unsigned long long)n};
  const unsigned long long strides[3] = {(unsigned long long)ld * 2, (unsigned long long)w * ld * 2,
                                         (unsigned long long)h * w * ld * 2};
  const unsigned int box[4] = {64, (unsigned int)bw, (unsigned int)bh, (unsigned int)bn};
  return crfr_tmap_encode_bf16(m, ptr, 4, dims, strides, box, "activation");
}

// packed weights [rows][kdim] bf16 (kdim contiguous); box = (64, box_rows)
int make_weight_map(CUtensorMap* m, const void* ptr, long long rows, int kdim, int box_rows) {
  const unsigned long long dims[2] = {(unsigned long long)kdim, (unsigned long long)rows};
  const unsigned long long strides[1] = {(unsigned long long)kdim * 2};
  const unsigned int box[2] = {64, (unsigned int)box_rows};
  return crfr_tmap_encode_bf16(m, ptr, 2, dims, strides, box, "weights");
}

struct Tiling {
  int bw, bh, bn, tiles_x, tiles_y, tiles_n, rows;  // rows = bw*bh*bn <= 128
};

bool make_tiling(int n, int h, int w, Tiling* t) {
  if (w >= 128) {
    t->bw = 128; t->bh = 1; t->bn = 1;
  } else {
    t->bw = w;
    t->bh = 128 / w;
    if (t->bh > h) t->bh = h;
    if (t->bh < 1) return false;
    t->bn = 128 / (t->bw * t->bh);
    if (t->bn < 1) t->bn = 1;
    if (t->bn > 256) return false;
  }
  t->rows = t->bw * t->bh * t->bn;
  t->tiles_x = (w + t->bw - 1) / t->bw;
  t->tiles_y = (h + t->bh - 1) / t->bh;
  t->tiles_n = (n + t->bn - 1) / t->bn;
  return t->rows <= 128 && t->rows >= 1;
}

// ------------------------------------------------------------------------------------------------
// forward / dgrad kernel
// ------------------------------------------------------------------------------------------------
struct ConvParams {
  int n, h, w;
  int kchunks, ksize, ntaps, pad, sign;
  int bw, bh, bn, tiles_x, tiles_y, rows;
  int total_tiles; // pixel tiles (a CTA walks several)
  int n_total;     // all output channels; this CTA computes columns [blockIdx.y * N, +N)
  int out_ld;
  int out_f32;     // 0: bf16 NHWC rows, 1: fp32 NHWC rows
  void* out;
  const float* bias;
  float* partial;  // InstanceNorm partials [n][slots][2][n_total] of the stored (bf16) output, or nullptr
  int slots, gpt;  // partial slots per image; 32-row groups of a tile that belong to one image (4, 2 or 1)
};

constexpr int kConvThreads = 192;  // warp 0: TMA, warp 1: MMA + TMEM alloc, warps 2-5: epilogue
constexpr int kATileBytes = 128 * 128;

// R (3x3, 64 input channels, N <= 64): the TMA unit issues one request per 128-byte pixel row of a box, and the generic
// form asks for 128 rows per (tap, K chunk) step - 1 152 rows and 72 KB of re-streamed weights per pixel tile, which bounds
// the 64 -> 64 layers at 766 cycles per K step with the tensor pipe 17 % active (ncu: nothing else above 25 % of its peak).
// R keeps all nine weight tiles resident in shared memory and loads ONE box per kx shift that also holds the two halo
// rows, (bh + 2) x bw pixels: the three ky taps of a kx are row offsets into the same box (the launcher asks for bw % 8 == 0, which every
// shape that reaches this form has; the swizzle is a function of the address, so any 128-byte row offset would do - see the
// weight-gradient form).  576 rows per tile instead of 1 152, 3 ring steps of 12 MMAs instead of 9 of 4.
constexpr int kResidentIters = 9;
// MODE 0: generic; 1: R (above); 2: T2 - TWO pixel tiles per weight tile: a ring step loads the activation tiles of two
// consecutive pixel tiles of the CTA and ONE weight tile, and issues the MMAs of both (four TMEM accumulators: the pair being
// computed and the pair in the epilogue): 384 instead of 512 TMA rows per two (tap, K chunk) steps at N = 128.
template <int N, int MODE = 0>
struct ConvCfg {
  static constexpr bool R = MODE == 1, T2 = MODE == 2;
  static constexpr int kBTileBytes = N * 128;
  static constexpr int kStageBytes = R ? 2 * kATileBytes : (T2 ? 2 : 1) * kATileBytes + kBTileBytes;   // R: up to 256 pixel rows (box + halo)
  // stages: the K loops are short (9-72 steps per tile) and every step is a TMA round trip to L2 (~1 us): the ring is as deep
  // as the 227 KB of shared memory allow beside the staging tile (24 / 32 / 48 KB per stage)
  static constexpr int kStages = (R || T2) ? 4 : (N <= 64) ? 8 : (N <= 128) ? 6 : 3;
  static constexpr int kAccBufs = T2 ? 4 : 2;
  static constexpr int kResidentBytes = R ? kResidentIters * kBTileBytes : 0;
  static constexpr int kTmemCols = (N <= 32) ? 32 : (N <= 64) ? 64 : (N <= 128) ? 128 : 256;
  static constexpr int kOutTiles = (N + 63) / 64;               // 64-channel sub-tiles staged for the TMA store
  static constexpr int kOutBytes = kOutTiles * kATileBytes;
  static constexpr int kSmemBytes = kStages * kStageBytes + kResidentBytes + kOutBytes + 1024 /*align slack*/ + 256 /*barriers*/;
  static_assert(N % 32 == 0 && N <= 256 && kAccBufs * kTmemCols <= 512, "tile width");
  static_assert(kSmemBytes <= 232448, "shared memory budget");
};

// Persistent: the grid is (CTAs, column tiles); a CTA walks pixel tiles blockIdx.x, blockIdx.x + gridDim.x, ... so
// that barrier setup / TMEM allocation are paid once and - with two TMEM accumulators - the epilogue of tile i
// overlaps the TMA + MMA work of tile i+1 (the layers on this kernel have short K loops: 9-72 steps per tile).
template <int N, int MODE>
__global__ void __launch_bounds__(kConvThreads, 1)
tc_conv_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmY, ConvParams p) {   // R: tmA has the box with the halo rows
  using Cfg = ConvCfg<N, MODE>;
  constexpr bool R = Cfg::R, T2 = Cfg::T2;
  constexpr int kAB = Cfg::kAccBufs;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* sB = base + Cfg::kStages * Cfg::kStageBytes;          // R: resident weight tiles [iters][N][64]
  uint8_t* sOut = sB + Cfg::kResidentBytes;
  uint64_t* full = (uint64_t*)(sOut + Cfg::kOutBytes);
  uint64_t* empty = full + Cfg::kStages;
  uint64_t* tmem_full = empty + Cfg::kStages;   // [kAB]
  uint64_t* tmem_empty = tmem_full + kAB;       // [kAB]
  uint64_t* w_full = tmem_empty + kAB;          // R: the resident weights have landed
  uint32_t* tmem_slot = (uint32_t*)(w_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < Cfg::kStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < kAB; ++b) {
      mbar_init(&tmem_full[b], 1);
      mbar_init(&tmem_empty[b], 4);
    }
    mbar_init(w_full, 1);
    fence_barrier_init();
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    prefetch_tmap(&tmY);
  }
  if (warp == 1) tmem_alloc<kAB * Cfg::kTmemCols>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  const int iters = R ? 3 : p.ntaps * p.kchunks;   // ring steps per pixel tile
  const uint32_t a_bytes = (uint32_t)p.rows * 128u;
  const int ncol0 = blockIdx.y * N;
  const int my_tiles = (int)blockIdx.x < p.total_tiles ? (p.total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;

  if (warp == 0) {
    const bool leader = elect_one();
    if (R && leader && my_tiles > 0) {
      mbar_expect_tx(w_full, (uint32_t)kResidentIters * Cfg::kBTileBytes);
      for (int tap = 0; tap < kResidentIters; ++tap)
        tma_load_2d(sB + tap * Cfg::kBTileBytes, &tmB, w_full, 0, tap * p.n_total + ncol0);
    }
    int g = 0;   // running stage index across tiles
    for (int i = 0; i < my_tiles; i += T2 ? 2 : 1) {
      int t = blockIdx.x + i * gridDim.x;
      const int tx = t % p.tiles_x; t /= p.tiles_x;
      const int ty = t % p.tiles_y; t /= p.tiles_y;
      const int x0 = tx * p.bw, y0 = ty * p.bh, n0 = t * p.bn;
      // T2: the second pixel tile of the pair (absent where the CTA's tile count is odd: that step loads and computes one tile)
      const bool has2 = T2 && i + 1 < my_tiles;
      int t1 = blockIdx.x + (has2 ? i + 1 : i) * gridDim.x;
      const int tx1 = t1 % p.tiles_x; t1 /= p.tiles_x;
      const int ty1 = t1 % p.tiles_y; t1 /= p.tiles_y;
      const int x1 = tx1 * p.bw, y1 = ty1 * p.bh, n1 = t1 * p.bn;
      for (int it = 0; it < iters; ++it, ++g) {
        const int s = g % Cfg::kStages;
        mbar_wait(&empty[s], ((g / Cfg::kStages) & 1) ^ 1);
        uint8_t* sa = base + s * Cfg::kStageBytes;
        if (R) {   // step = kx: the box of rows y0 - 1 .. y0 + bh at the x shift of this kx
          if (leader) {
            mbar_expect_tx(&full[s], (uint32_t)((p.bh + 2) * p.bw) * 128u);
            tma_load_4d(sa, &tmA, &full[s], 0, x0 + p.sign * (it - 1), y0 - 1, n0);
          }
          continue;
        }
        const int tap = it / p.kchunks, kc = it - tap * p.kchunks;
        const int ky = tap / p.ksize, kx = tap - ky * p.ksize;
        if (leader) {
          mbar_expect_tx(&full[s], (has2 ? 2u : 1u) * a_bytes + (uint32_t)Cfg::kBTileBytes);
          tma_load_4d(sa, &tmA, &full[s], kc * 64, x0 + p.sign * (kx - p.pad), y0 + p.sign * (ky - p.pad), n0);
          if (has2) tma_load_4d(sa + kATileBytes, &tmA, &full[s], kc * 64, x1 + p.sign * (kx - p.pad), y1 + p.sign * (ky - p.pad), n1);
          tma_load_2d(sa + (T2 ? 2 : 1) * kATileBytes, &tmB, &full[s], kc * 64, tap * p.n_total + ncol0);
        }
      }
    }
  } else if (warp == 1) {
    const bool leader = elect_one();
    const uint32_t idesc = make_idesc_bf16(128, N, 0, 0);
    const uint64_t desc0 = make_smem_desc_sw128(smem_u32(base), 16, 1024);
    const uint64_t descB = make_smem_desc_sw128(smem_u32(sB), 16, 1024);
    if (R && my_tiles > 0) mbar_wait(w_full, 0);
    int g = 0;
    for (int i = 0; i < my_tiles; i += T2 ? 2 : 1) {
      // accumulator of tile i: generic i & 1 (use i >> 1); T2: pair j = i / 2 owns buffers 2 (j & 1) + {0, 1} (use j >> 1)
      const int buf = T2 ? ((i >> 1) & 1) * 2 : (i & 1);
      const uint32_t use = T2 ? (uint32_t)(i >> 2) : (uint32_t)(i >> 1);
      mbar_wait(&tmem_empty[buf], (use & 1) ^ 1);   // the epilogue has drained this accumulator
      if (T2) mbar_wait(&tmem_empty[buf + 1], (use & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem + buf * Cfg::kTmemCols;
      for (int it = 0; it < iters; ++it, ++g) {
        const int s = g % Cfg::kStages;
        mbar_wait(&full[s], (g / Cfg::kStages) & 1);
        tc_fence_after();
        const uint64_t da = desc0 + (uint64_t)((s * Cfg::kStageBytes) >> 4);
        if (R) {   // step = kx; tap (ky, kx) reads the box from row (forward: ky, dgrad: 2 - ky) on
          if (leader) {
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
              const int row = p.sign > 0 ? ky : 2 - ky;
              const uint64_t dak = da + (uint64_t)((row * p.bw * 128) >> 4);
              const uint64_t dbk = descB + (uint64_t)(((ky * 3 + it) * Cfg::kBTileBytes) >> 4);
#pragma unroll
              for (int k = 0; k < 4; ++k) umma_bf16(d_tmem, dak + 2 * k, dbk + 2 * k, idesc, (uint32_t)((it | ky | k) != 0));
            }
            umma_commit(&empty[s]);
          }
          __syncwarp();
          continue;
        }
        const uint64_t db = da + (uint64_t)(((T2 ? 2 : 1) * kATileBytes) >> 4);
        if (leader) {
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_bf16(d_tmem, da + 2 * k, db + 2 * k, idesc, (uint32_t)((it | k) != 0));
          if (T2 && i + 1 < my_tiles) {
            const uint64_t da1 = da + (uint64_t)(kATileBytes >> 4);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16(d_tmem + Cfg::kTmemCols, da1 + 2 * k, db + 2 * k, idesc, (uint32_t)((it | k) != 0));
          }
          umma_commit(&empty[s]);
        }
        __syncwarp();
      }
      if (leader) {
        umma_commit(&tmem_full[buf]);
        if (T2) umma_commit(&tmem_full[buf + 1]);
      }
      __syncwarp();
    }
  } else {
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const int iw = r % p.bw;
    const int rr = r / p.bw;
    const int ih = rr % p.bh, in = rr / p.bh;
    const float* bias = p.bias ? p.bias + ncol0 : nullptr;
    const bool issuer = warp == 2 && lane == 0;
    float bsum[Cfg::kOutTiles][4];   // batch statistics (BatchNorm): running sums of this thread's channel pair and row group
#pragma unroll
    for (int t2 = 0; t2 < Cfg::kOutTiles; ++t2) bsum[t2][0] = bsum[t2][1] = bsum[t2][2] = bsum[t2][3] = 0.f;
    for (int i = 0; i < my_tiles; ++i) {
      const int buf = T2 ? ((i >> 1) & 1) * 2 + (i & 1) : (i & 1);
      const uint32_t use = T2 ? (uint32_t)(i >> 2) : (uint32_t)(i >> 1);
      int t = blockIdx.x + i * gridDim.x;
      const int tx = t % p.tiles_x; t /= p.tiles_x;
      const int ty = t % p.tiles_y; t /= p.tiles_y;
      const int x0 = tx * p.bw, y0 = ty * p.bh, n0 = t * p.bn;
      const int x = x0 + iw, y = y0 + ih, n = n0 + in;
      const bool valid = r < p.rows && x < p.w && y < p.h && n < p.n;
      const long long pix = ((long long)n * p.h + y) * p.w + x;
      float* dstf = (float*)p.out + pix * p.out_ld + ncol0;
      mbar_wait(&tmem_full[buf], use & 1);
      tc_fence_after();
      if (!p.out_f32) {
        // the TMA store of the previous tile must have finished reading the staging buffer
        if (issuer) tma_store_wait_read<0>();
        named_bar_sync(1, 128);
      }
#pragma unroll
      for (int c0 = 0; c0 < N; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + buf * Cfg::kTmemCols + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          float f[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) f[e] = __uint_as_float(v[j + e]) + (bias ? bias[c0 + j + e] : 0.f);
          if (p.out_f32) {
            if (valid) {
              *reinterpret_cast<float4*>(dstf + c0 + j) = make_float4(f[0], f[1], f[2], f[3]);
              *reinterpret_cast<float4*>(dstf + c0 + j + 4) = make_float4(f[4], f[5], f[6], f[7]);
            }
          } else {
            // stage the bf16 tile in the SWIZZLE_128B layout of the output tensor map: sub-tile (c / 64), row r
            const int c = c0 + j;
            uint8_t* srow = sOut + (c >> 6) * kATileBytes + r * 128;
            *reinterpret_cast<bf16x8*>(srow + ((((c & 63) >> 3) ^ (r & 7)) << 4)) = pack8(f);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[buf]);   // accumulator free for tile i + 2
      if (!p.out_f32) {
        fence_proxy_async();
        named_bar_sync(1, 128);
        if (issuer) {   // one TMA store per 64-channel sub-tile; out-of-range pixels are clipped
#pragma unroll
          for (int t2 = 0; t2 < Cfg::kOutTiles; ++t2)
            tma_store_4d(&tmY, sOut + t2 * kATileBytes, ncol0 + t2 * 64, x0, y0, n0);
          tma_store_commit();
        }
        if (p.partial) {
          // InstanceNorm statistics of the stored (rounded) values, from the staged tile: thread = (channel pair,
          // 32-row group); a warp reads one 128-byte row per step (conflict free).  Every group lies inside one image;
          // its sums go to a fixed (image, tile, group) slot and are folded in fixed order by crfr_norm_finalize.
          // Batch mode (gpt < 0, BatchNorm: one group over the whole batch): slot = (pixel tile, group), any tiling; the
          // rows of the tile that lie outside the tensor hold values that are never stored and are masked out.
          const int et = (warp - 2) * 32 + lane, cp = et & 31, pg = et >> 5;
          const bool batch = p.gpt < 0;
          uint32_t vmask = 0xffffffffu;   // bit k: row pg * 32 + k of the tile lies inside the tensor (pg is NOT this warp's
          if (batch) {                    // TMEM quadrant q: the statistics walk the staged tile, not the accumulator)
            const int r2 = pg * 32 + lane, rr2 = r2 / p.bw;
            vmask = __ballot_sync(0xffffffffu, r2 < p.rows && x0 + r2 % p.bw < p.w && y0 + rr2 % p.bh < p.h && n0 + rr2 / p.bh < p.n);
          }
          const int img = batch ? 0 : n0 + (pg * 32) / (p.bw * p.bh);
          const int slot = batch ? 0 : (ty * p.tiles_x + tx) * p.gpt + pg % p.gpt;
          float* dst = p.partial + ((long long)img * p.slots + slot) * 2 * p.n_total + ncol0 + 2 * cp;
          if (img < p.n)
#pragma unroll
          for (int t2 = 0; t2 < Cfg::kOutTiles; ++t2) {
            float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
#pragma unroll 8
            for (int k = 0; k < 32; ++k) {
              const int px = pg * 32 + k;
              float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(
                  sOut + t2 * kATileBytes + px * 128 + ((((cp >> 2) ^ (px & 7)) << 4) | ((cp & 3) << 2))));
              if (!((vmask >> k) & 1u)) f = make_float2(0.f, 0.f);
              s0 += f.x; q0 = fmaf(f.x, f.x, q0);
              s1 += f.y; q1 = fmaf(f.y, f.y, q1);
            }
            if (batch) {   // one running sum per (CTA, row group) over all of the CTA's tiles, written once at the end
              bsum[t2][0] += s0; bsum[t2][1] += s1; bsum[t2][2] += q0; bsum[t2][3] += q1;
            } else {
              *reinterpret_cast<float2*>(dst + t2 * 64) = make_float2(s0, s1);
              *reinterpret_cast<float2*>(dst + p.n_total + t2 * 64) = make_float2(q0, q1);
            }
          }
        }
      }
    }
    if (p.partial && p.gpt < 0) {   // batch statistics: slot = (CTA, row group)
      const int et = (warp - 2) * 32 + lane, cp = et & 31, pg = et >> 5;
      float* dst = p.partial + ((long long)(blockIdx.x * 4 + pg)) * 2 * p.n_total + ncol0 + 2 * cp;
#pragma unroll
      for (int t2 = 0; t2 < Cfg::kOutTiles; ++t2) {
        *reinterpret_cast<float2*>(dst + t2 * 64) = make_float2(bsum[t2][0], bsum[t2][1]);
        *reinterpret_cast<float2*>(dst + p.n_total + t2 * 64) = make_float2(bsum[t2][2], bsum[t2][3]);
      }
    }
    if (issuer) tma_store_wait_read<0>();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<kAB * Cfg::kTmemCols>(tmem);
  }
}

int conv_sm_count() { return crfr_sm_count(); }

template <int N, int MODE = 0>
int launch_conv(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmY, const ConvParams& p, int tiles,
                cudaStream_t st) {
  using Cfg = ConvCfg<N, MODE>;
  static std::atomic<unsigned long long> attr_done{0};
  CRFR_CUDA((cudaError_t)crfr_smem_attr(tc_conv_kernel<N, MODE>, Cfg::kSmemBytes, attr_done));
  // persistent over pixel tiles: about one CTA per SM in total (column tiles share the pixel-tile walk)
  const int ncol = p.n_total / N;
  int ctas = conv_sm_count() / ncol;   // rounded down: more CTAs than SMs would be a second, nearly empty wave
  if (ctas > tiles) ctas = tiles;
  if (ctas < 1) ctas = 1;
  tc_conv_kernel<N, MODE><<<dim3(ctas, ncol), kConvThreads, Cfg::kSmemBytes, st>>>(tmA, tmB, tmY, p);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

// ------------------------------------------------------------------------------------------------
// wgrad kernel
// ------------------------------------------------------------------------------------------------
struct WgradParams {
  int n, h, w;
  int bw, bh, bn, tiles_x, tiles_y, total_tiles;
  int cin, cout;   // cout = all dY channels; a CTA handles columns [ntile * N, +N)
  int rows;        // pixels per tile (bw*bh*bn <= 128); rows beyond it are kept zero in shared memory
  float* G;        // [gridDim.x][taps][cin][cout] fp32: one slice per split, every element stored once
};

constexpr int kTile16K = 128 * 128;

// TAPS = 3: one kernel row (ky) of a 3x3 conv per CTA, the three kx taps share the dY tile.  TAPS = 1: plain
// [cin x cout] = X^T dY product (1x1 convs and the im2col-lowered edge layers).
// H (TAPS = 3, haloed box): one kernel COLUMN (kx) per CTA instead, from ONE X box that also holds the two halo rows,
// (bh + 2) x bw pixels - the three ky taps are row offsets into it (the second M atom of the first MMA is simply bw pixel
// rows further, LBO = bw x 128 B).  (bh + 2) x bw + 128 N / 64 TMA rows per step instead of 384 + 128 N / 64: the TMA request
// rate bounds these kernels as it does the forward engine, and the smaller stage buys a deeper ring.
template <int N, int TAPS, bool H = false>
struct WgCfg {
  static constexpr int kDyTiles = N / 64;
  static constexpr int kXBytes = H ? 2 * kTile16K : TAPS * kTile16K;
  static constexpr int kStageBytes = kXBytes + kDyTiles * kTile16K;
  static constexpr int kStages = (kStageBytes <= 32 * 1024) ? 6 : (kStageBytes <= 48 * 1024) ? 4 : (kStageBytes <= 64 * 1024) ? 3 : 2;
  static constexpr bool kSwap = TAPS == 3 && (N == 128 || N == 64);   // dY as the M operand, the three tap views along N
  static constexpr int kAccs = (TAPS + 1) / 2;                     // accumulators of M = 128 (two taps each)
  static constexpr int kTmemCols = kSwap ? 256 : (kAccs * N <= 64) ? 64 : (kAccs * N <= 128) ? 128 : 256;   // kSwap: 192 columns
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 + 256;
};

__device__ __forceinline__ void st_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("st.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

template <int N, int TAPS, bool H>
__global__ void __launch_bounds__(kConvThreads, 1)
tc_wgrad_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmDY, WgradParams p) {
  using Cfg = WgCfg<N, TAPS, H>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full = (uint64_t*)(base + Cfg::kStages * Cfg::kStageBytes);
  uint64_t* empty = full + Cfg::kStages;
  uint64_t* tmem_full = empty + Cfg::kStages;
  uint32_t* tmem_slot = (uint32_t*)(tmem_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < Cfg::kStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(tmem_full, 1);
    fence_barrier_init();
    prefetch_tmap(&tmX);
    prefetch_tmap(&tmDY);
  }
  if (warp == 1) tmem_alloc<Cfg::kTmemCols>(tmem_slot);
  if (p.rows < 128 || H) {
    // pixels are the K dimension: the rows of a 128-row tile that the (smaller) TMA box never writes must read as
    // zero, so clear the whole ring once
    for (int i = threadIdx.x; i < Cfg::kStages * Cfg::kStageBytes / 16; i += kConvThreads)
      reinterpret_cast<uint4*>(base)[i] = make_uint4(0u, 0u, 0u, 0u);
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  // TAPS == 3: blockIdx.y = ky (H: kx) + 3 * column tile;  TAPS == 1: blockIdx.y = column tile of dY
  const int ky = TAPS == 3 ? blockIdx.y % 3 : 0, kc = blockIdx.z;
  float* const G = p.G + (long long)blockIdx.x * (TAPS == 3 ? 9 : 1) * p.cin * p.cout;   // this split's slice
  const int ncol0 = (TAPS == 3 ? blockIdx.y / 3 : blockIdx.y) * N;
  const uint32_t stage_tx = H ? (uint32_t)((p.bh + 2) * p.bw + Cfg::kDyTiles * p.rows) * 128u
                              : (uint32_t)(TAPS + Cfg::kDyTiles) * (uint32_t)p.rows * 128u;
  const int first = blockIdx.x, step = gridDim.x;
  const int my_tiles = first < p.total_tiles ? (p.total_tiles - first + step - 1) / step : 0;

  if (warp == 0) {
    const bool leader = elect_one();
    for (int i = 0; i < my_tiles; ++i) {
      const int s = i % Cfg::kStages;
      mbar_wait(&empty[s], ((i / Cfg::kStages) & 1) ^ 1);
      int t = first + i * step;
      const int tx = t % p.tiles_x; t /= p.tiles_x;
      const int ty = t % p.tiles_y; t /= p.tiles_y;
      const int x0 = tx * p.bw, y0 = ty * p.bh, n0 = t * p.bn;
      uint8_t* sb = base + s * Cfg::kStageBytes;
      if (leader) {
        mbar_expect_tx(&full[s], stage_tx);
        if (H) {   // `ky` is this CTA's kx: the box of rows y0 - 1 .. y0 + bh at its x shift
          tma_load_4d(sb, &tmX, &full[s], kc * 64, x0 + ky - 1, y0 - 1, n0);
        } else if (TAPS == 3) {
#pragma unroll
          for (int kx = 0; kx < 3; ++kx)
            tma_load_4d(sb + kx * kTile16K, &tmX, &full[s], kc * 64, x0 + kx - 1, y0 + ky - 1, n0);
        } else {
          tma_load_4d(sb, &tmX, &full[s], kc * 64, x0, y0, n0);
        }
#pragma unroll
        for (int j = 0; j < Cfg::kDyTiles; ++j)
          tma_load_4d(sb + Cfg::kXBytes + j * kTile16K, &tmDY, &full[s], ncol0 + j * 64, x0, y0, n0);
      }
    }
  } else if (warp == 1) {
    const bool leader = elect_one();
    const uint32_t idesc = Cfg::kSwap ? make_idesc_bf16(N, 192, 1, 1) : make_idesc_bf16(128, N, 1, 1);
    // kSwap (three taps, 128 dY channels): the dY tile is the M operand (128 channels: a full M) and the three tap views of X are
    // stacked along N - ONE M = 128, N = 192 MMA per K step, every block of it wanted, instead of two M = 128, N = 128 MMAs of
    // which the second uses half its rows (an M = 64 MMA costs the pipe as much as M = 128): 96 instead of 128 cycles.
    // Otherwise:
    // M = 128 = two 64-channel atoms LBO (= one 16 KB tile) apart: taps (0,1) in the first MMA; the second atom of
    // the last MMA is whatever tile follows (rows 64..127 of that accumulator are never read)
    // (H: the atoms are the ky = 0 / 1 / 2 views of one box, bw pixel rows apart; dY keeps its 16 KB tiles)
    const uint32_t x_lbo = H ? (uint32_t)p.bw * 128u : (uint32_t)kTile16K;
    const uint64_t desc0 = make_smem_desc_sw128(smem_u32(base), x_lbo, 1024);
    const uint64_t descB = make_smem_desc_sw128(smem_u32(base), kTile16K, 1024);
    for (int i = 0; i < my_tiles; ++i) {
      const int s = i % Cfg::kStages;
      mbar_wait(&full[s], (i / Cfg::kStages) & 1);
      tc_fence_after();
      const uint64_t a01 = desc0 + (uint64_t)((s * Cfg::kStageBytes) >> 4);
      const uint64_t a2x = a01 + (uint64_t)((2 * x_lbo) >> 4);
      const uint64_t db = descB + (uint64_t)((s * Cfg::kStageBytes + Cfg::kXBytes) >> 4);
#pragma unroll
      for (int k = 0; k < 8; ++k) {  // 8 x 16 pixels
        const uint32_t acc = (uint32_t)((i | k) != 0);
        if (Cfg::kSwap) {
          if (leader) umma_bf16(tmem, db + k * (2048 >> 4), a01 + k * (2048 >> 4), idesc, acc);
          continue;
        }
        if (leader) umma_bf16(tmem, a01 + k * (2048 >> 4), db + k * (2048 >> 4), idesc, acc);
        if (TAPS == 3)
          if (leader) umma_bf16(tmem + N, a2x + k * (2048 >> 4), db + k * (2048 >> 4), idesc, acc);
      }
      if (leader) umma_commit(&empty[s]);
      __syncwarp();
    }
    if (leader) umma_commit(tmem_full);
    __syncwarp();
  } else if (my_tiles > 0) {
    const int q = warp & 3;
    const int r = q * 32 + lane;
    mbar_wait(tmem_full, 0);
    tc_fence_after();
    const int ci = kc * 64 + (r & 63);
    if (Cfg::kSwap) {
      // D[co = lane][(tap view a) x 64 ci]: a warp's 32 lanes hold 32 consecutive co of one (tap, ci) -> one coalesced
      // 128-byte reduction per column
#pragma unroll
      // (64 dY channels: an M = 64 accumulator keeps row i in lane 32 * (i / 16) + i % 16 - the upper half of every warp's
      // lanes holds nothing)
      const int co = N == 64 ? q * 16 + lane : r;
      const bool live = N != 64 || lane < 16;
#pragma unroll
      for (int c0 = 0; c0 < 192; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + c0, v);
        tmem_ld_wait();
        const int a = c0 / 64;
        const int tap = H ? a * 3 + ky : ky * 3 + a;
        float* dst = G + ((long long)tap * p.cin + kc * 64 + (c0 & 63)) * p.cout + ncol0 + co;
        if (live) {
#pragma unroll
          for (int j = 0; j < 32; ++j) dst[(long long)j * p.cout] = __uint_as_float(v[j]);
        }
      }
    } else
#pragma unroll
    for (int half = 0; half < Cfg::kAccs; ++half) {
      const int kx = half == 0 ? (r >> 6) : 2;                          // (H: this is the tap's ky, and `ky` its kx)
      const bool live = TAPS == 3 ? (half == 0 || r < 64) : (r < 64);   // warp-uniform (32-row granularity)
      const int tap = TAPS == 3 ? (H ? kx * 3 + ky : ky * 3 + kx) : 0;
      float* dst = G + ((long long)tap * p.cin + ci) * p.cout + ncol0;
#pragma unroll
      for (int c0 = 0; c0 < N; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + half * N + c0, v);
        tmem_ld_wait();
        if (live) {
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            st_v4(dst + c0 + j, __uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]),
                  __uint_as_float(v[j + 3]));
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<Cfg::kTmemCols>(tmem);
  }
}

// G[i] = sum of the `splits` partial slices in split order (a fixed order: the same bits on every run)
__global__ void wgrad_split_sum_kernel(const float4* __restrict__ part, int splits, long long slice4, float4* __restrict__ G) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= slice4) return;
  float4 s = part[i];
  for (int k = 1; k < splits; ++k) {
    const float4 v = part[k * slice4 + i];
    s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
  }
  G[i] = s;
}

// dW[co][ci][t] += G[t][ci][co]
__global__ void wgrad_unpack_kernel(const float* __restrict__ G, float* __restrict__ dw, int cin, int cout, int T) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = (long long)cout * cin * T;
  if (i >= total) return;
  int t = (int)(i % T);
  long long q = i / T;
  int ci = (int)(q % cin);
  int co = (int)(q / cin);
  dw[i] += G[((long long)t * cin + ci) * cout + co];
}

template <int N, int TAPS, bool H = false>
int launch_wgrad(const CUtensorMap& tmX, const CUtensorMap& tmDY, const WgradParams& p, int splits, cudaStream_t st) {
  using Cfg = WgCfg<N, TAPS, H>;
  static std::atomic<unsigned long long> attr_done{0};
  CRFR_CUDA((cudaError_t)crfr_smem_attr(tc_wgrad_kernel<N, TAPS, H>, Cfg::kSmemBytes, attr_done));
  const int gy = (TAPS == 3 ? 3 : 1) * (p.cout / N);
  tc_wgrad_kernel<N, TAPS, H><<<dim3(splits, gy, p.cin / 64), kConvThreads, Cfg::kSmemBytes, st>>>(tmX, tmDY, p);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

bool spatial_ok(int h, int w, bool exact128) {
  Tiling t;
  if (!make_tiling(1, h, w, &t)) return false;
  if (w > 128 && (w % 128) != 0 && exact128) return false;
  return true;
}

int pick_tile_n(int n_total) {
  const int cands[] = {256, 224, 192, 128, 96, 64, 32};
  for (int c : cands)
    if (n_total % c == 0) return c;
  return 0;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// generic launchers (internal.h)
// ------------------------------------------------------------------------------------------------
int crfr_tc_gemm(const TcGemm& g, cudaStream_t st) {
  CRFR_CHECK_ARG(((uintptr_t)g.src & 15) == 0 && ((uintptr_t)g.out & 15) == 0 && ((uintptr_t)g.wt & 15) == 0 &&
                     (g.src_ld & 7) == 0 && (g.out_ld & 3) == 0,
                 "tc_gemm: pointers must be 16B aligned and ld a multiple of 8");
  CRFR_CHECK_ARG(g.k_total % 64 == 0 && g.k_total > 0, "tc_gemm: K %d must be a multiple of 64", g.k_total);
  const int tile_n = g.tile_n ? g.tile_n : pick_tile_n(g.n_total);
  CRFR_CHECK_ARG(tile_n && g.n_total % tile_n == 0, "tc_gemm: N %d has no supported tile width", g.n_total);
  Tiling t;
  if (!make_tiling(g.n, g.h, g.w, &t)) {
    crfr_set_error("tc_gemm: unsupported spatial size %dx%d", g.h, g.w);
    return CRFR_EUNSUPPORTED;
  }
  CUtensorMap tmA, tmB, tmY;
  CRFR_TRY(make_act_map(&tmA, g.src, g.n, g.h, g.w, g.k_total, g.src_ld, t.bw, t.bh, t.bn));
  if (!g.out_f32) {
    CRFR_CHECK_ARG(tile_n % 64 == 0 && (g.out_ld & 7) == 0, "tc_gemm: bf16 output needs a tile width multiple of 64");
    CRFR_TRY(make_act_map(&tmY, g.out, g.n, g.h, g.w, g.n_total, g.out_ld, t.bw, t.bh, t.bn));
  } else {
    tmY = tmA;   // unused by the fp32 epilogue
  }
  const int T = g.ksize * g.ksize;
  CRFR_TRY(make_weight_map(&tmB, g.wt, (long long)T * g.n_total, g.k_total, tile_n));
  ConvParams p;
  p.n = g.n; p.h = g.h; p.w = g.w;
  p.kchunks = g.k_total / 64; p.ksize = g.ksize; p.ntaps = T; p.pad = g.pad; p.sign = g.sign;
  p.bw = t.bw; p.bh = t.bh; p.bn = t.bn; p.tiles_x = t.tiles_x; p.tiles_y = t.tiles_y; p.rows = t.rows;
  p.n_total = g.n_total; p.out_ld = g.out_ld; p.out_f32 = g.out_f32; p.out = g.out; p.bias = g.bias;
  const int tiles = t.tiles_x * t.tiles_y * t.tiles_n;
  p.total_tiles = tiles;
  p.partial = nullptr; p.slots = 0; p.gpt = 0;
  if (g.stat_slots) *g.stat_slots = 0;
  int batch_ctas = conv_sm_count() / (g.n_total / tile_n);   // = launch_conv's grid.x
  if (batch_ctas > tiles) batch_ctas = tiles;
  if (batch_ctas < 1) batch_ctas = 1;
  if (g.stat_batch && g.stat_ws && g.stat_slots && !g.out_f32 && tile_n % 64 == 0 && !g.bias &&
      sizeof(float) * (size_t)batch_ctas * 4 * 2 * g.n_total <= g.stat_ws_bytes) {
    p.partial = g.stat_ws;
    p.slots = batch_ctas * 4;
    p.gpt = -1;
    *g.stat_slots = p.slots;
  } else if (g.stat_ws && g.stat_slots && !g.out_f32 && tile_n % 64 == 0 && t.rows == 128 && g.h % t.bh == 0 && g.w % t.bw == 0 &&
      (t.bw * t.bh) % 32 == 0) {
    // fused statistics: 128-row tiles of whole image rows whose 32-row groups never straddle an image.  Eligibility
    // must not depend on the batch size (a ragged last tile just skips the images that do not exist): the statistics
    // of an image on this engine are then the same bits however the batch is chunked or sharded, which keeps chunked /
    // data-parallel runs within rounding of the single-call result (tests/test_fsrnet_gpu.py: 1e-4 on the losses)
    const int area = t.bw * t.bh;
    p.gpt = area >= 128 ? 4 : area / 32;
    p.slots = t.tiles_x * t.tiles_y * p.gpt;
    if (sizeof(float) * (size_t)g.n * p.slots * 2 * g.n_total <= g.stat_ws_bytes) {
      p.partial = g.stat_ws;
      *g.stat_slots = p.slots;
    }
  }
  switch (tile_n) {
    case 32: return launch_conv<32>(tmA, tmB, tmY, p, tiles, st);
    case 64:
      if (p.ksize == 3 && p.pad == 1 && p.kchunks == 1 && p.bn == 1 && (p.bw & 7) == 0 && (p.bh + 2) * p.bw <= 256) {
        CUtensorMap tmA2;   // the box with its two halo rows
        CRFR_TRY(make_act_map(&tmA2, g.src, g.n, g.h, g.w, g.k_total, g.src_ld, t.bw, t.bh + 2, 1));
        return launch_conv<64, 1>(tmA2, tmB, tmY, p, tiles, st);
      }
      return launch_conv<64>(tmA, tmB, tmY, p, tiles, st);
    case 96: return launch_conv<96>(tmA, tmB, tmY, p, tiles, st);
    case 128:
      if (tiles >= 4 * conv_sm_count()) return launch_conv<128, 2>(tmA, tmB, tmY, p, tiles, st);
      return launch_conv<128>(tmA, tmB, tmY, p, tiles, st);
    case 192: return launch_conv<192>(tmA, tmB, tmY, p, tiles, st);
    case 224: return launch_conv<224>(tmA, tmB, tmY, p, tiles, st);
    case 256: return launch_conv<256>(tmA, tmB, tmY, p, tiles, st);
  }
  crfr_set_error("tc_gemm: unsupported tile width %d", tile_n);
  return CRFR_EUNSUPPORTED;
}

namespace {
int launch_wgrad_any(const TcWgrad& g, const Tiling& t, const CUtensorMap& tmX, const CUtensorMap& tmDY, const WgradParams& p,
                     int splits, cudaStream_t st) {
  if (g.taps3x3) {
    if (t.bn == 1 && (t.bh + 2) * t.bw <= 256 && (g.cout == 64 || g.cout % 128 == 0)) {
      CUtensorMap tmXh;   // the X box with its two halo rows
      CRFR_TRY(make_act_map(&tmXh, g.x, g.n, g.h, g.w, g.cin, g.x_ld, t.bw, t.bh + 2, 1));
      if (g.cout == 64) return launch_wgrad<64, 3, true>(tmXh, tmDY, p, splits, st);
      return launch_wgrad<128, 3, true>(tmXh, tmDY, p, splits, st);
    }
    if (g.cout == 64) return launch_wgrad<64, 3>(tmX, tmDY, p, splits, st);
    if (g.cout % 128 == 0) return launch_wgrad<128, 3>(tmX, tmDY, p, splits, st);
    crfr_set_error("tc_wgrad: 3x3 needs cout 64 or a multiple of 128, got %d", g.cout);
    return CRFR_EUNSUPPORTED;
  }
  if (g.cout % 128 == 0) return launch_wgrad<128, 1>(tmX, tmDY, p, splits, st);
  return launch_wgrad<64, 1>(tmX, tmDY, p, splits, st);
}
}  // namespace

int crfr_tc_wgrad_raw(const TcWgrad& g, cudaStream_t st) {
  CRFR_CHECK_ARG(((uintptr_t)g.x & 15) == 0 && ((uintptr_t)g.dy & 15) == 0 && (g.x_ld & 7) == 0 && (g.dy_ld & 7) == 0,
                 "tc_wgrad: pointers must be 16B aligned and ld a multiple of 8");
  CRFR_CHECK_ARG(g.cin % 64 == 0 && g.cout % 64 == 0, "tc_wgrad: channels must be multiples of 64");
  Tiling t;
  if (!make_tiling(g.n, g.h, g.w, &t)) {
    crfr_set_error("tc_wgrad: unsupported spatial size %dx%d", g.h, g.w);
    return CRFR_EUNSUPPORTED;
  }
  CUtensorMap tmX, tmDY;
  CRFR_TRY(make_act_map(&tmX, g.x, g.n, g.h, g.w, g.cin, g.x_ld, t.bw, t.bh, t.bn));
  CRFR_TRY(make_act_map(&tmDY, g.dy, g.n, g.h, g.w, g.cout, g.dy_ld, t.bw, t.bh, t.bn));
  WgradParams p;
  p.n = g.n; p.h = g.h; p.w = g.w;
  p.bw = t.bw; p.bh = t.bh; p.bn = t.bn; p.tiles_x = t.tiles_x; p.tiles_y = t.tiles_y;
  p.total_tiles = t.tiles_x * t.tiles_y * t.tiles_n;
  p.cin = g.cin; p.cout = g.cout;
  p.rows = t.rows;
  const int tile_n = (g.cout % 128 == 0) ? 128 : 64;
  const int ctas_per_split = (g.taps3x3 ? 3 : 1) * (g.cout / tile_n) * (g.cin / 64);
  // One CTA per SM at a time (160-192 KB of shared memory): the grid runs in waves of `sms` CTAs, so it must not exceed a whole
  // number of them - 50 splits x 6 CTAs = 300 CTAs on 148 SMs were THREE waves for 2.03 waves of work.  Two waves, rounded DOWN.
  const int sms = conv_sm_count();
  int splits = (2 * sms) / ctas_per_split;
  if (splits < 1) splits = ctas_per_split <= sms ? sms / ctas_per_split : 1;
  if (splits > p.total_tiles) splits = p.total_tiles;
  if (splits < 1) splits = 1;
  // several splits store their partials into g.part and are summed into G afterwards; as many as fit (one: straight into G)
  const long long slice = (long long)(g.taps3x3 ? 9 : 1) * g.cin * g.cout;
  const long long fit = g.part ? (long long)(g.part_bytes / (sizeof(float) * (size_t)slice)) : 0;
  if (splits > fit) splits = fit > 1 ? (int)fit : 1;
  CRFR_CHECK_ARG(splits == 1 || ((uintptr_t)g.part & 15) == 0, "tc_wgrad: partial buffer must be 16B aligned");
  p.G = splits > 1 ? g.part : g.G;
  CRFR_TRY(launch_wgrad_any(g, t, tmX, tmDY, p, splits, st));
  if (splits > 1) {
    wgrad_split_sum_kernel<<<crfr_cdiv(slice / 4, 256), 256, 0, st>>>((const float4*)g.part, splits, slice / 4, (float4*)g.G);
    CRFR_COUNT_LAUNCH();
    CRFR_LAUNCH_CHECK();
  }
  return CRFR_OK;
}

size_t crfr_tc_wgrad_part_bytes() {
  // splits x slice <= 2 * SMs x (3 tap rows x 64 cin x 128 cout per CTA) floats whatever the shape (see crfr_tc_wgrad_raw)
  return sizeof(float) * (size_t)2 * conv_sm_count() * 3 * 64 * 128 + 256;
}

int crfr_tc_supported(int op, int h, int w, int cin, int cout, int k, int stride, int pad) {
  if (k != 3 || stride != 1 || pad != 1) return 0;
  if (cin % 64 || cout % 64) return 0;
  const int nout = (op == 1) ? cin : cout;  // GEMM N
  if (op == 2) {
    if (cout != 64 && cout % 128 != 0) return 0;
    return spatial_ok(h, w, true) ? 1 : 0;
  }
  if (pick_tile_n(nout) == 0) return 0;
  return spatial_ok(h, w, false) ? 1 : 0;
}

size_t crfr_tc_workspace_bytes(const crfr_conv_desc* d) {
  // wgrad: the [tap][cin][cout] result + the per-split partial sums
  size_t wg = sizeof(float) * (size_t)d->k * d->k * d->cin * d->cout + 256 + crfr_tc_wgrad_part_bytes();
  {   // statistics partials of the fused epilogue: [n][tiles per image x 4][2][cout]
    Tiling t;
    if (make_tiling(d->n, d->oh, d->ow, &t)) {
      const size_t sp = sizeof(float) * (size_t)d->n * t.tiles_x * t.tiles_y * 4 * 2 * d->cout + 256;
      if (sp > wg) wg = sp;
    }
  }
  if (crfr_rowconv_supported(d->h, d->w, d->cin, d->cout, d->k, d->stride, d->pad)) {
    const size_t rc = crfr_rowconv_ws_bytes(d->n, d->h);
    if (rc > wg) wg = rc;
    const size_t rw = crfr_rowwgrad_ws_bytes(d->n, d->h);
    if (rw > wg) wg = rw;
  }
  return wg;
}

int crfr_tc_conv(const crfr_conv_desc* d, int dgrad, const void* src, const void* w_packed, const float* bias,
                 void* dst, float* stats, float eps, void* ws, size_t ws_bytes, cudaStream_t st, int batch_stats) {
  if (!batch_stats && crfr_rowconv_supported(d->h, d->w, d->cin, d->cout, d->k, d->stride, d->pad)) {
    return crfr_rowconv(src, dgrad ? d->out_ld : d->in_ld, d->n, d->h, w_packed, dgrad, bias, dst,
                        dgrad ? d->in_ld : d->out_ld, dgrad ? nullptr : stats, eps, ws, ws_bytes, st);
  }
  TcGemm g;
  g.src = src; g.n = d->n; g.h = d->h; g.w = d->w;
  g.k_total = dgrad ? d->cout : d->cin;
  g.src_ld = dgrad ? d->out_ld : d->in_ld;
  g.wt = w_packed; g.ksize = d->k; g.pad = d->pad; g.sign = dgrad ? -1 : 1;
  g.n_total = dgrad ? d->cin : d->cout;
  g.tile_n = g.n_total <= 256 ? g.n_total : 0;   // wider layers: several column tiles per pixel tile
  g.out = dst; g.out_ld = dgrad ? d->in_ld : d->out_ld; g.out_f32 = 0; g.bias = bias;
  // InstanceNorm statistics: in the epilogue where the tiling allows it (partials in the workspace, folded by
  // crfr_norm_finalize), otherwise by a separate pass over the stored output
  int slots = 0;
  const bool want_stats = stats && !dgrad;
  g.stat_ws = want_stats ? (float*)ws : nullptr;
  g.stat_ws_bytes = want_stats ? ws_bytes : 0;
  g.stat_slots = &slots;
  g.stat_batch = batch_stats;
  CRFR_TRY(crfr_tc_gemm(g, st));
  if (want_stats && batch_stats) {   // one group over the whole batch
    const long long count = (long long)d->n * d->oh * d->ow;
    if (slots) CRFR_TRY(crfr_norm_finalize((const float*)ws, 1, slots, (int)count, d->cout, eps, stats, st));
    else CRFR_TRY(crfr_norm_stats(dst, 1, (int)count, d->cout, d->out_ld, eps, stats, ws, ws_bytes, (void*)st));
  } else if (want_stats) {
    if (slots) CRFR_TRY(crfr_norm_finalize((const float*)ws, d->n, slots, d->oh * d->ow, d->cout, eps, stats, st));
    else CRFR_TRY(crfr_norm_stats(dst, d->n, d->oh * d->ow, d->cout, d->out_ld, eps, stats, ws, ws_bytes, (void*)st));
  }
  return CRFR_OK;
}

int crfr_tc_wgrad(const crfr_conv_desc* d, const void* x, const void* dy, float* dw, void* ws, size_t ws_bytes,
                  cudaStream_t st) {
  if (crfr_rowwgrad_supported(d->h, d->w, d->cin, d->cout, d->k, d->stride, d->pad))
    return crfr_rowwgrad(x, d->in_ld, dy, d->out_ld, d->n, d->h, dw, ws, ws_bytes, st);
  const size_t need = sizeof(float) * (size_t)9 * d->cin * d->cout;
  if (!ws || ws_bytes < need) {
    crfr_set_error("tc_wgrad: workspace %zu < %zu", ws_bytes, need);
    return CRFR_EWORKSPACE;
  }
  CRFR_CUDA(cudaMemsetAsync(ws, 0, need, st));
  TcWgrad g;
  g.x = x; g.n = d->n; g.h = d->h; g.w = d->w; g.cin = d->cin; g.x_ld = d->in_ld;
  g.dy = dy; g.cout = d->cout; g.dy_ld = d->out_ld; g.taps3x3 = 1; g.G = (float*)ws;
  const size_t part_off = (need + 255) & ~(size_t)255;
  g.part = ws_bytes > part_off ? (float*)((uint8_t*)ws + part_off) : nullptr;
  g.part_bytes = ws_bytes > part_off ? ws_bytes - part_off : 0;
  CRFR_TRY(crfr_tc_wgrad_raw(g, st));
  long long total = (long long)d->cout * d->cin * 9;
  wgrad_unpack_kernel<<<crfr_cdiv(total, 256), 256, 0, st>>>((const float*)ws, dw, d->cin, d->cout, 9);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}
