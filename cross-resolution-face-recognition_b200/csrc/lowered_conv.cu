// Edge layers lowered onto the tcgen05 GEMM engine.
//
// The layers whose channel counts cannot fill a UMMA tile (3-channel images) or that are strided / transposed are
// rewritten as [cheap HBM-bound gather kernel] + [plain tcgen05 GEMM over 64-channel K chunks]:
//   R1  Conv2d 3x3 s1 p1, cin = 3 (coarse conv_input, FSRnet.py:312)   fwd, wgrad : im2col(27 -> 64 ch) . W
//   R2  Conv2d 3x3 s1 p1, cout = 3 (conv_mid :318, conv_out :439)      fwd : x . W(27 -> 32 cols, fp32) then col2im
//                                                                     dgrad, wgrad : im2col(dY) as the GEMM operand
//   R3  Conv2d 7x7 s4|s2 p3, cin = 3 (encoder / prior stems :345, :384; ResNet stem model/resnet.py:158)   fwd, wgrad : im2col(147 -> 192 ch) . W
//                                                                     dgrad : dY . W (192 cols, fp32) then col2im
//   R4  ConvTranspose2d 7x7 s4 p2 op1, 64 -> 64 (decoder :436): sub-pixel decomposition.  Output pixel (4a+py, 4b+px)
//       only sees the taps ky = (py+2) mod 4 (+4), kx likewise, i.e. every one of the 16 output phases is a <= 2x2-tap
//       convolution of the 32x32 input with offsets in {-1,0,1}.  All phases together are ONE 3x3 pad-1 convolution
//       64 -> 16*64 channels with a block-sparse weight (49 of 144 blocks non-zero), run on the implicit-GEMM kernel,
//       followed by a pixel shuffle; dgrad / wgrad are that convolution's dgrad / wgrad on the un-shuffled dOut.
//       (The earlier x . W -> 1.6 GB fp32 -> col2im formulation moved 12x more bytes.)
//   R5  Conv2d 3x3 s2 p1|p0 / 1x1 s2 p0, channels % 64 == 0 (ResNet stage transitions and downsample branches,
//       model/resnet.py:9-16, 193-200; p0: the reflection-padded stride-2 stages of SUPER_RESOLUTION/model/FSRnet.py)
//                                                                     fwd, wgrad : im2col(T*cin) . W
//                                                                     dgrad : dY . W (T*cin cols, fp32) then col2im
//   R6  Conv2d 1x1 s1 p0, channels % 64 == 0 (the pre-activation Bottlenecks of SUPER_RESOLUTION/model/FSRnet.py:75-114)
//                                                                     fwd, dgrad : one GEMM;  wgrad : X^T . dY
//   R7  ConvTranspose2d 3x3 s2 p1 op1, channels % 64 == 0 (the up stages of SUPER_RESOLUTION/model/FSRnet.py): the
//       transpose of R5's convolution, so R5's three forms with the roles exchanged
//                                                                     fwd : X . W (9*cout cols, fp32) then col2im
//                                                                     dgrad : im2col(dY) . W
//                                                                     wgrad : im2col(dY)^T . X
// R1 - R3 also take the padding-0 ("valid") 3x3 / 7x7 stride-1 forms of the variant's reflection-padded stems and heads
// (R2 with 64 or 128 input channels).
// Partial products that are summed by a col2im kernel stay fp32 until the single final rounding, so the arithmetic
// contract is the same as the direct kernels': fp32 accumulation over all taps and channels, one bf16 rounding.
#include "common.cuh"
#include "crfr.h"
#include "internal.h"

namespace {

// ---------------------------------------------------------------------------------------------------------
// gather kernels
// ---------------------------------------------------------------------------------------------------------
// P[o][tap*3 + c] = x[o*stride + sign*(tap - pad)][c] for 3-channel images stored 4 bf16 per pixel (zero outside the
// image and for k >= T*3); kpad % 8 == 0.  One thread writes one 16-byte group of a row, so a warp writes whole
// 128-byte lines; the 8 values of a group come from at most 4 taps, each fetched as one 8-byte pixel.  The grid is
// (groups of an output row, n * oh) and KS is a template parameter so that no per-thread runtime division is left
// (the first version spent most of its time in them).
template <int KS>
__global__ void im2col_small_kernel(const bf16* __restrict__ x, int h, int w, int oh, int ow, int stride, int pad, int sign,
                                    bf16* __restrict__ P, int kpad, int rows) {
  const int groups = kpad >> 3;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;   // (ox, g) within the output row
  if (idx >= ow * groups) return;
  const int ox = idx / groups, g = idx - ox * groups;
  const int k0 = g * 8, kmax = KS * KS * 3;
  for (int row = blockIdx.y; row < rows; row += gridDim.y) {   // row = n * oh + oy
  const int n = row / oh, oy = row - n * oh;
  uint32_t out[4] = {0u, 0u, 0u, 0u};
  if (k0 < kmax) {
    // the 8 values of this group come from taps t0 .. t0+3: fetch those (up to) four pixels, then pick per value with
    // selects - every array below is indexed statically, so nothing is demoted to local memory
    const int t0 = k0 / 3;
    uint2 pv[4];
#pragma unroll
    for (int ti = 0; ti < 4; ++ti) {
      const int tap = t0 + ti;
      const int ky = tap / KS, kx = tap - ky * KS;
      const int y = oy * stride + sign * (ky - pad), xx = ox * stride + sign * (kx - pad);
      pv[ti] = make_uint2(0u, 0u);
      if (tap < KS * KS && y >= 0 && y < h && xx >= 0 && xx < w)
        pv[ti] = *reinterpret_cast<const uint2*>(x + (((long long)n * h + y) * w + xx) * 4);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = k0 + j;
      const int tap = k / 3, c = k - tap * 3, ti = tap - t0;
      const uint2 v = ti == 0 ? pv[0] : (ti == 1 ? pv[1] : (ti == 2 ? pv[2] : pv[3]));
      uint32_t val = c == 0 ? (v.x & 0xffffu) : (c == 1 ? (v.x >> 16) : (v.y & 0xffffu));
      if (k >= kmax) val = 0u;
      out[j >> 1] |= val << ((j & 1) * 16);
    }
  }
  *reinterpret_cast<uint4*>(P + ((long long)row * ow + ox) * kpad + g * 8) = make_uint4(out[0], out[1], out[2], out[3]);
  }
}

// The 3x3 / stride 1 / pad 1 case with the 27 values padded to one 64-wide K block (coarse conv_input, conv_mid,
// conv_out and their gradients: six launches per FSRNet step at 128 x 128): one thread per pixel gathers its nine
// neighbours (8-byte loads, L1-resident overlap with the neighbouring threads), assembles the values with statically
// indexed selects, and the block writes its 128 x 128 bytes through a swizzled shared-memory transpose as fully
// coalesced 16-byte stores.  The generic kernel above (one thread per 16 output bytes, four dependent-address loads
// each) ran at 0.7-1.4 TB/s of output; this one is bound by the 268 MB it writes.
__global__ void __launch_bounds__(128)
im2col3_s1_kernel(const bf16* __restrict__ x, int h, int w, int sign, bf16* __restrict__ P, long long total) {
  __shared__ uint4 tile[128 * 8];
  const long long p = (long long)blockIdx.x * 128 + threadIdx.x;
  uint32_t out[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) out[i] = 0u;
  if (p < total) {
    const int xx = (int)(p % w);
    const long long q = p / w;
    const int y = (int)(q % h);
    const long long n = q / h;
    uint2 pv[9];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int yy = y + sign * (ky - 1), x2 = xx + sign * (kx - 1);
        pv[ky * 3 + kx] = make_uint2(0u, 0u);
        if (yy >= 0 && yy < h && x2 >= 0 && x2 < w)
          pv[ky * 3 + kx] = *reinterpret_cast<const uint2*>(x + ((n * h + yy) * w + x2) * 4);
      }
#pragma unroll
    for (int k = 0; k < 27; ++k) {
      const int tap = k / 3, c = k - tap * 3;
      const uint32_t val = c == 0 ? (pv[tap].x & 0xffffu) : (c == 1 ? (pv[tap].x >> 16) : (pv[tap].y & 0xffffu));
      out[k >> 1] |= val << ((k & 1) * 16);
    }
  }
  const int t = threadIdx.x, sw = t & 7;
#pragma unroll
  for (int j = 0; j < 8; ++j)   // chunks 4..7 are the zero padding of K = 27 -> 64
    tile[t * 8 + (j ^ sw)] = j < 4 ? make_uint4(out[4 * j], out[4 * j + 1], out[4 * j + 2], out[4 * j + 3]) : make_uint4(0u, 0u, 0u, 0u);
  __syncthreads();
  uint4* dst = reinterpret_cast<uint4*>(P) + (long long)blockIdx.x * 1024;
  const long long limit = (total - (long long)blockIdx.x * 128) * 8;   // 16-byte chunks of this block inside the matrix
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int i = j * 128 + t, tp = i >> 3, jj = i & 7;
    if (i < limit) dst[i] = tile[tp * 8 + (jj ^ (tp & 7))];
  }
}

// The 7x7 case (the stems: stride 4 at FSRnet.py:110, stride 2 at model/resnet.py:166) with the 147 values padded to K = 192:
// one thread per output pixel fetches its 49 input pixels (8-byte loads, 16 or 32 bytes apart across a warp) and assembles
// the row's 96 words in order - a tap is three halves, so taps alternately start on a word boundary and in the middle of a
// word, all resolved statically - into a shared-memory row of 97 words (conflict-free), and the block writes its rows as
// fully coalesced stores.  The generic kernel (one thread per 16 output bytes, four scattered loads each) wrote 1.2 TB/s:
// 248 us for the 308 MB of ResNet_34's stem at batch 256, five times per KD step.
constexpr int kI7Pix = 64;
__global__ void __launch_bounds__(kI7Pix)
im2col7_kernel(const bf16* __restrict__ x, int h, int w, int oh, int ow, int stride, int pad, bf16* __restrict__ P,
               long long total) {
  __shared__ uint32_t tile[kI7Pix * 97];
  const long long p0 = (long long)blockIdx.x * kI7Pix;
  const long long p = p0 + threadIdx.x;
  if (p < total) {
    const int ox = (int)(p % ow);
    const long long q = p / ow;
    const int oy = (int)(q % oh);
    const long long n = q / oh;
    uint32_t* row = tile + threadIdx.x * 97;
    const int y0 = oy * stride - pad, x0 = ox * stride - pad;
    const uint2* img = reinterpret_cast<const uint2*>(x) + n * h * w;
    uint32_t carry = 0u;
#pragma unroll
    for (int ky = 0; ky < 7; ++ky) {
      const int y = y0 + ky;
      const bool yin = y >= 0 && y < h;
      const uint2* rp = img + (long long)y * w;
#pragma unroll
      for (int kx = 0; kx < 7; ++kx) {
        const int xx = x0 + kx;
        uint2 v = make_uint2(0u, 0u);
        if (yin && xx >= 0 && xx < w) v = __ldg(rp + xx);
        const int k = (ky * 7 + kx) * 3;   // first of the tap's three values
        if ((k & 1) == 0) {
          row[k >> 1] = v.x;               // c0 | c1 << 16
          carry = v.y & 0xffffu;           // c2: the low half of the next word
        } else {
          row[k >> 1] = carry | (v.x << 16);
          row[(k >> 1) + 1] = (v.x >> 16) | (v.y << 16);
        }
      }
    }
    row[73] = carry;                       // value 146, then the zero padding 147 .. 191
#pragma unroll
    for (int i = 74; i < 96; ++i) row[i] = 0u;
  }
  __syncthreads();
  const long long left = total - p0;
  const int words = (int)(left < kI7Pix ? left : kI7Pix) * 96;
  uint32_t* dst = reinterpret_cast<uint32_t*>(P) + p0 * 96;
  for (int i = threadIdx.x; i < words; i += kI7Pix) {
    const int pix = i / 96;
    dst[i] = tile[pix * 97 + (i - pix * 96)];
  }
}

int launch_im2col_small(const bf16* x, int n, int h, int w, int oh, int ow, int ks, int stride, int pad, int sign, bf16* P,
                        int kpad, cudaStream_t st) {
  if (ks == 7 && sign == 1 && kpad == 192) {
    const long long total = (long long)n * oh * ow;
    im2col7_kernel<<<(unsigned)crfr_cdiv(total, kI7Pix), kI7Pix, 0, st>>>(x, h, w, oh, ow, stride, pad, P, total);
    CRFR_COUNT_LAUNCH();
    CRFR_LAUNCH_CHECK();
    return CRFR_OK;
  }
  if (ks == 3 && stride == 1 && pad == 1 && kpad == 64 && oh == h && ow == w) {
    const long long total = (long long)n * h * w;
    im2col3_s1_kernel<<<(unsigned)crfr_cdiv(total, 128), 128, 0, st>>>(x, h, w, sign, P, total);
    CRFR_COUNT_LAUNCH();
    CRFR_LAUNCH_CHECK();
    return CRFR_OK;
  }
  const int rows = n * oh;
  // a block per (row slice) would be 65 k one-store blocks at 128x128: block launch rate, not bandwidth, bounds that.
  // ~16 blocks per SM, each walking rows with the grid stride
  const unsigned gx = (unsigned)crfr_cdiv((long long)ow * (kpad >> 3), 256);
  unsigned gy = (148u * 16u + gx - 1) / gx;
  if (gy > (unsigned)rows) gy = (unsigned)rows;
  const dim3 grid(gx, gy);
  if (ks == 3) im2col_small_kernel<3><<<grid, 256, 0, st>>>(x, h, w, oh, ow, stride, pad, sign, P, kpad, rows);
  else if (ks == 7) im2col_small_kernel<7><<<grid, 256, 0, st>>>(x, h, w, oh, ow, stride, pad, sign, P, kpad, rows);
  else {
    crfr_set_error("im2col_small: kernel size %d not instantiated", ks);
    return CRFR_EUNSUPPORTED;
  }
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

// dst[P][c] = bias[c] + sum_{tap : t = P + sgn*(pad - tap), t % stride == 0, t/stride inside} src[t/stride][tap*C + c]
// src fp32 [.., src_ld]; outputs: fp32 NCHW and/or bf16 NHWC (ld, zero channel padding)
__global__ void col2im_small_kernel(const float* __restrict__ src, int src_ld, int C, int sh, int sw, int bh, int bw,
                                    int ks, int stride, int pad, int sgn, const float* __restrict__ bias,
                                    float* __restrict__ y_nchw, bf16* __restrict__ y, int y_ld, long long total) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int X = (int)(i % bw);
  long long q = i / bw;
  const int Y = (int)(q % bh);
  const long long n = q / bh;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int c = 0; c < 4; ++c) acc[c] = (bias && c < C) ? bias[c] : 0.f;   // (C <= 4; static indices keep acc in registers)
  // only every stride-th tap can hit a source pixel: start at the first one and step by the stride (the 7x7 stride-4 stems
  // walked all 49 taps with a modulo each to find their 1-4 contributions: 133 us per launch at 128 images)
  const int ky0 = sgn > 0 ? (Y + pad) % stride : ((pad - Y) % stride + stride) % stride;
  const int kx0 = sgn > 0 ? (X + pad) % stride : ((pad - X) % stride + stride) % stride;
  for (int ky = ky0; ky < ks; ky += stride) {
    const int ty = Y + sgn * (pad - ky);
    if (ty < 0) continue;
    const int sy = ty / stride;
    if (sy >= sh) continue;
    for (int kx = kx0; kx < ks; kx += stride) {
      const int tx = X + sgn * (pad - kx);
      if (tx < 0) continue;
      const int sx = tx / stride;
      if (sx >= sw) continue;
      const float* s = src + ((n * sh + sy) * sw + sx) * src_ld + (ky * ks + kx) * C;
#pragma unroll
      for (int c = 0; c < 4; ++c)
        if (c < C) acc[c] += s[c];
    }
  }
  if (y_nchw) {
#pragma unroll
    for (int c = 0; c < 4; ++c)
      if (c < C) y_nchw[(n * C + c) * ((long long)bh * bw) + (long long)Y * bw + X] = acc[c];
  }
  if (y) {
#pragma unroll
    for (int c = 0; c < 4; ++c)
      if (c < y_ld) y[i * y_ld + c] = __float2bfloat16_rn(c < C ? acc[c] : 0.f);
    for (int c = 4; c < y_ld; ++c) y[i * y_ld + c] = __float2bfloat16_rn(0.f);
  }
}

// The 3x3 / stride 1 / pad 1, three-channel case of col2im (forward of conv_mid / conv_out, FSRnet.py:318,439): a block
// stages the [10 x 34 source pixels][27 partial products] halo tile of an 8 x 32 output tile in shared memory with
// coalesced 16-byte loads (row stride 33 floats: the nine-neighbour reads below are then conflict free) and every
// thread sums its 27 terms from there.  The generic kernel issues 27 scalar loads per pixel whose addresses are 128
// bytes apart across a warp - 32 L1 wavefronts per instruction - and is bound by exactly that (195 us for 128 images).
__global__ void __launch_bounds__(256)
col2im3_s1_kernel(const float* __restrict__ src, int h, int w, int sgn, const float* __restrict__ bias,
                  float* __restrict__ y_nchw, bf16* __restrict__ y, int y_ld) {
  constexpr int TH = 8, TW = 32, SH = TH + 2, SW = TW + 2, LD = 33;
  __shared__ float tile[SH * SW * LD];
  const int tiles_x = (w + TW - 1) / TW, tiles_y = h / TH;   // a last partial column tile when w % 32 != 0
  int b = blockIdx.x;
  const int tx0 = (b % tiles_x) * TW;
  b /= tiles_x;
  const int ty0 = (b % tiles_y) * TH;
  const long long n = b / tiles_y;
  const float* img = src + n * h * w * 32;
  for (int i = threadIdx.x; i < SH * SW * 8; i += 256) {   // one 16-byte quarter-line of a source pixel per iteration
    const int px = i >> 3, q = i & 7;
    const int sy = ty0 - 1 + px / SW, sx = tx0 - 1 + px % SW;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (sy >= 0 && sy < h && sx >= 0 && sx < w) v = *reinterpret_cast<const float4*>(img + ((long long)sy * w + sx) * 32 + q * 4);
    float* t = tile + px * LD + q * 4;
    t[0] = v.x; t[1] = v.y; t[2] = v.z; t[3] = v.w;
  }
  __syncthreads();
  const int ly = threadIdx.x >> 5, lx = threadIdx.x & 31;
  float acc[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) acc[c] = bias ? bias[c] : 0.f;
#pragma unroll
  for (int ky = 0; ky < 3; ++ky)
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
      const float* t = tile + ((ly + 1 + sgn * (1 - ky)) * SW + (lx + 1 + sgn * (1 - kx))) * LD + (ky * 3 + kx) * 3;
#pragma unroll
      for (int c = 0; c < 3; ++c) acc[c] += t[c];
    }
  const int Y = ty0 + ly, X = tx0 + lx;
  if (X >= w) return;
  if (y_nchw)
#pragma unroll
    for (int c = 0; c < 3; ++c) y_nchw[((n * 3 + c) * h + Y) * w + X] = acc[c];
  if (y) {
    const long long i = (n * h + Y) * w + X;
    for (int c = 0; c < y_ld; ++c) y[i * y_ld + c] = __float2bfloat16_rn(c < 3 ? acc[c] : 0.f);
  }
}

// ---- sub-pixel (phase) decomposition of the 7x7 s4 p2 transposed convolution --------------------------------
// tap k (0..6) -> output phase p = (k + 2) mod 4 and input offset d = (p + 2 - k) / 4 in {-1, 0, 1}
__device__ __forceinline__ void subpixel_of_tap(int k, int* phase, int* off) {
  const int p = (k + 2) & 3;
  *phase = p;
  *off = (p + 2 - k) / 4;   // exact: -4, 0 or 4 in the numerator
}

// mode 0 (forward):  src [49][co][ci] -> dst [9][(py*4+px)*64 + co][ci]
// mode 1 (dgrad):    src [49][ci][co] -> dst [9][ci][(py*4+px)*64 + co]            (dst pre-zeroed)
__global__ void deconv_subpixel_pack_kernel(const bf16* __restrict__ src, bf16* __restrict__ dst, int mode) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 49 * 64 * 64) return;
  const int s_ = i & 63, r = (i >> 6) & 63, tap = i >> 12;
  int py, dy, px, dx;
  subpixel_of_tap(tap / 7, &py, &dy);
  subpixel_of_tap(tap % 7, &px, &dx);
  const int t9 = (dy + 1) * 3 + (dx + 1), ph = py * 4 + px;
  if (mode == 0) dst[((size_t)t9 * 1024 + ph * 64 + r) * 64 + s_] = src[i];       // r = co, s = ci
  else dst[((size_t)t9 * 64 + r) * 1024 + ph * 64 + s_] = src[i];                 // r = ci, s = co
}

__global__ void deconv_bias_kernel(const float* __restrict__ bias, float* __restrict__ big) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 1024) big[i] = bias ? bias[i & 63] : 0.f;
}

// to_all == 0: y[n][4a+py][4b+px][co] = all[n][a][b][(py*4+px)*64 + co]   (pixel shuffle; y has per-pixel stride y_ld)
// to_all == 1: the inverse (un-shuffle of dOut).  One thread per 16 bytes.
__global__ void deconv_shuffle_kernel(bf16* __restrict__ y, int y_ld, bf16* __restrict__ all, int sh, int sw, int to_all,
                                      long long total) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int g = (int)(i & 7);
  long long p = i >> 3;                     // output pixel (n, Y, X)
  const int X = (int)(p % (4 * sw));
  long long q = p / (4 * sw);
  const int Y = (int)(q % (4 * sh));
  const long long n = q / (4 * sh);
  const long long ai = ((n * sh + (Y >> 2)) * sw + (X >> 2)) * 1024 + ((Y & 3) * 4 + (X & 3)) * 64 + g * 8;
  uint4* py_ = reinterpret_cast<uint4*>(y + p * y_ld + g * 8);
  uint4* pa = reinterpret_cast<uint4*>(all + ai);
  if (to_all) *pa = *py_;
  else *py_ = *pa;
}

// dW[ci][co][ky][kx] += G[t9][ci][(py*4+px)*64 + co]
__global__ void deconv_subpixel_unpack_kernel(const float* __restrict__ G, float* __restrict__ dw) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;   // over [ci][co][49]
  if (i >= 64 * 64 * 49) return;
  const int tap = i % 49, co = (i / 49) & 63, ci = i / (49 * 64);
  int py, dy, px, dx;
  subpixel_of_tap(tap / 7, &py, &dy);
  subpixel_of_tap(tap % 7, &px, &dx);
  const int t9 = (dy + 1) * 3 + (dx + 1), ph = py * 4 + px;
  dw[i] += G[((size_t)t9 * 64 + ci) * 1024 + ph * 64 + co];
}

// Generic im2col for channel counts that are multiples of 8 (16-byte vectors):
// P[o][tap*C + c] = x[o*stride + tap - pad][c], zero outside the image
__global__ void im2col_vec_kernel(const bf16* __restrict__ x, int x_ld, int C, int h, int w, int oh, int ow, int ks,
                                  int stride, int pad, bf16* __restrict__ P, long long total) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int groups = C >> 3, T = ks * ks;
  const int g = (int)(i % groups);
  long long r = i / groups;
  const int tap = (int)(r % T);
  long long o = r / T;
  const int ox = (int)(o % ow);
  long long q = o / ow;
  const int oy = (int)(q % oh);
  const long long n = q / oh;
  const int ky = tap / ks, kx = tap - ky * ks;
  const int y = oy * stride + ky - pad, xx = ox * stride + kx - pad;
  uint4 v = make_uint4(0u, 0u, 0u, 0u);
  if (y >= 0 && y < h && xx >= 0 && xx < w)
    v = *reinterpret_cast<const uint4*>(x + ((n * h + y) * w + xx) * x_ld + g * 8);
  *reinterpret_cast<uint4*>(P + o * ((long long)T * C) + (long long)tap * C + g * 8) = v;
}

// Its transpose: dx[p][c] = bias[c] + sum over the taps that reach input pixel p of dP[o][tap*C + c] (fp32 in, one
// rounding; bias may be NULL)
__global__ void col2im_vec_kernel(const float* __restrict__ dP, int C, int oh, int ow, int h, int w, int ks, int stride,
                                  int pad, const float* __restrict__ bias, bf16* __restrict__ dx, int dx_ld, long long total) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int groups = C >> 3;
  const int g = (int)(i % groups);
  long long p = i / groups;
  const int X = (int)(p % w);
  long long q = p / w;
  const int Y = (int)(q % h);
  const long long n = q / h;
  const long long ld = (long long)ks * ks * C;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (bias)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = bias[g * 8 + j];
  for (int ky = 0; ky < ks; ++ky) {
    const int ty = Y + pad - ky;
    if (ty < 0 || ty % stride) continue;
    const int oy = ty / stride;
    if (oy >= oh) continue;
    for (int kx = 0; kx < ks; ++kx) {
      const int tx = X + pad - kx;
      if (tx < 0 || tx % stride) continue;
      const int ox = tx / stride;
      if (ox >= ow) continue;
      const float4* s = reinterpret_cast<const float4*>(dP + ((n * oh + oy) * ow + ox) * ld + (ky * ks + kx) * C + g * 8);
      const float4 a = s[0], b = s[1];
      acc[0] += a.x; acc[1] += a.y; acc[2] += a.z; acc[3] += a.w;
      acc[4] += b.x; acc[5] += b.y; acc[6] += b.z; acc[7] += b.w;
    }
  }
  *reinterpret_cast<bf16x8*>(dx + p * dx_ld + g * 8) = pack8(acc);
}

// dst[r][tap*S + s] = src[tap][r][s] for s < S (src: [T][R][s_pad] bf16), zero elsewhere; dst is [rows_pad][kpad]
__global__ void repack_tapmajor_kernel(const bf16* __restrict__ src, int T, int R, int S, int s_pad, bf16* __restrict__ dst,
                                       int rows_pad, int kpad) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows_pad * kpad) return;
  const int k = i % kpad, r = i / kpad;
  bf16 v = __float2bfloat16_rn(0.f);
  if (r < R && k < T * S) {
    const int tap = k / S, s = k - tap * S;
    v = src[((long long)tap * R + r) * s_pad + s];
  }
  dst[i] = v;
}

// dw[(d0*D1 + d1)*T + tap] += G[k][n]
//   mode 0: k = tap*D1 + d1, n = d0            (R1 / R3: d0 = co, d1 = c)
//   mode 1: k = d1,          n = tap*D0 + d0   (R2: d0 = co, d1 = ci)
//   mode 2: k = d0,          n = tap*D1 + d1   (R4: d0 = ci, d1 = co)
__global__ void unpack_lowered_kernel(const float* __restrict__ G, int g_ld, float* __restrict__ dw, int D0, int D1, int T,
                                      int mode) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)D0 * D1 * T) return;
  const int tap = (int)(i % T);
  long long r = i / T;
  const int d1 = (int)(r % D1), d0 = (int)(r / D1);
  int k, n;
  if (mode == 0) { k = tap * D1 + d1; n = d0; }
  else if (mode == 1) { k = d1; n = tap * D0 + d0; }
  else { k = d0; n = tap * D1 + d1; }
  dw[i] += G[(long long)k * g_ld + n];
}

struct Arena {
  uint8_t* base;
  size_t cap, off;
  void* take(size_t bytes) {
    size_t a = (off + 1023) & ~(size_t)1023;
    if (a + bytes > cap) return nullptr;
    off = a + bytes;
    return base + a;
  }
  void rest(float** p, size_t* bytes) {   // everything not taken yet (the wgrad's partial sums)
    const size_t a = (off + 1023) & ~(size_t)1023;
    *p = a < cap ? (float*)(base + a) : nullptr;
    *bytes = a < cap ? cap - a : 0;
  }
};

#define TAKE(ptr, type, arena, bytes)                                              \
  type* ptr = (type*)(arena).take(bytes);                                          \
  if (!ptr) {                                                                      \
    crfr_set_error("lowered conv: workspace too small (%zu bytes given)", (arena).cap); \
    return CRFR_EWORKSPACE;                                                        \
  }

#define LAUNCH(kernel, total, st, ...)                                              \
  do {                                                                              \
    kernel<<<crfr_cdiv((total), 256), 256, 0, (st)>>>(__VA_ARGS__);                 \
    CRFR_COUNT_LAUNCH();                                                            \
    CRFR_LAUNCH_CHECK();                                                            \
  } while (0)

inline int kpad_of(const crfr_conv_desc* d) { return ((d->k * d->k * 3 + 63) / 64) * 64; }   // 27 -> 64, 147 -> 192

// Recipe 2's GEMMs are per-pixel products (no taps): at pad 0 they run over the n * h * w input pixels as one flat row of
// the tile engine, which keeps every 128-pixel tile full at the variant's 130-wide padded maps (as images, the second
// column tile of each 130-pixel row would hold 2 pixels).
struct PixGrid { int n, h, w; };
inline PixGrid valid_flat(const crfr_conv_desc* d) {
  if (d->pad == 1) return {d->n, d->h, d->w};
  return {1, 1, d->n * d->h * d->w};
}

int tcgen05_spatial_ok(int h, int w) { return crfr_tc_supported(2, h, w, 64, 64, 3, 1, 1); }

}  // namespace

// ---------------------------------------------------------------------------------------------------------
// recipe selection
// ---------------------------------------------------------------------------------------------------------
int crfr_lowered_recipe(const crfr_conv_desc* d) {
  const bool ld8 = (d->in_ld & 7) == 0 && (d->out_ld & 7) == 0, c64 = d->cin % 64 == 0 && d->cout % 64 == 0;
  if (!d->transposed) {
    if (d->k == 3 && d->stride == 1 && (d->pad == 1 || d->pad == 0) && d->cin == 3 && d->in_ld == 4 && d->cout % 64 == 0 &&
        d->cout <= 256 && tcgen05_spatial_ok(d->oh, d->ow))
      return 1;
    // pad 1 keeps its image-shaped GEMMs (tiled over h x w); pad 0 runs them over the flat pixel list (valid_flat below)
    if (d->k == 3 && d->stride == 1 && d->cout == 3 && d->out_ld == 4 &&
        ((d->pad == 1 && d->cin == 64 && tcgen05_spatial_ok(d->h, d->w)) ||
         (d->pad == 0 && (d->cin == 64 || d->cin == 128) && (d->in_ld & 7) == 0 && d->h > 2 && d->w > 2)))
      return 2;
    if (d->k == 7 && (((d->stride == 4 || d->stride == 2) && d->pad == 3) || (d->stride == 1 && d->pad == 0)) && d->cin == 3 &&
        d->in_ld == 4 && (d->cout == 64 || d->cout == 128) && tcgen05_spatial_ok(d->oh, d->ow))
      return 3;
    if (d->stride == 2 && ((d->k == 3 && (d->pad == 1 || d->pad == 0)) || (d->k == 1 && d->pad == 0)) && c64 && ld8 &&
        tcgen05_spatial_ok(d->oh, d->ow))
      return 5;
    if (d->k == 1 && d->stride == 1 && d->pad == 0 && c64 && ld8 && tcgen05_spatial_ok(d->h, d->w)) return 6;
    return 0;
  }
  if (d->k == 7 && d->stride == 4 && d->pad == 2 && d->cin == 64 && d->cout == 64 && d->oh == 4 * d->h && d->ow == 4 * d->w &&
      tcgen05_spatial_ok(d->h, d->w))
    return 4;
  if (d->k == 3 && d->stride == 2 && d->pad == 1 && d->oh == 2 * d->h && d->ow == 2 * d->w && c64 && ld8 &&
      tcgen05_spatial_ok(d->h, d->w))
    return 7;
  return 0;
}

// partial sums of the fused statistics: [n][slots][2][cout] fp32 with at most one slot per 32 output pixels of an image
static size_t stat_partial_bytes(const crfr_conv_desc* d) {
  return sizeof(float) * (size_t)d->n * (size_t)((d->oh * d->ow + 31) / 32) * 2 * (size_t)d->cout;
}

size_t crfr_lowered_ws_bytes(const crfr_conv_desc* d) {
  const int r = crfr_lowered_recipe(d);
  const size_t big = (size_t)d->n * d->h * d->w, small = (size_t)d->n * d->oh * d->ow;
  size_t b = 0;
  switch (r) {
    case 1: b = big * 64 * 2 + (size_t)256 * 64 * 2 + (size_t)64 * 256 * 4; break;
    case 2: b = big * 64 * 2 + big * 32 * 4 + (size_t)64 * 64 * 2 * 2 + (size_t)64 * 64 * 4; break;
    case 3: b = small * 192 * 2 + small * 192 * 4 + (size_t)192 * 128 * 2 * 2 + (size_t)192 * 128 * 4; break;
    case 4:   // big = input (small) grid here: [ipix][16 phases * 64] bf16 + block-sparse weights + wgrad accumulator
      b = big * 1024 * 2 + (size_t)9 * 1024 * 64 * 2 + (size_t)9 * 64 * 1024 * 4 + 1024 * 4 + 8192;
      break;
    case 5: {
      const size_t kc = (size_t)d->k * d->k * d->cin;
      b = small * kc * 2 + small * kc * 4 + (size_t)d->cout * kc * 2 + kc * d->cout * 4;
      break;
    }
    case 6: b = (size_t)d->cin * d->cout * 4; break;
    case 7: {   // big = the input grid here: [ipix][9 * cout] fp32 (forward) or bf16 (dgrad / wgrad) + weights / G
      const size_t kc = (size_t)9 * d->cout;
      b = big * kc * 4 + (size_t)d->cin * kc * 4 + 1024;
      break;
    }
    default: return 0;
  }
  if (r == 2 && d->pad == 0) b += (size_t)d->cin * 64 * 2 * 2 + (size_t)d->cin * 64 * 4;   // up to 128 input channels
  if (r == 1 || r == 3 || r == 5 || r == 6) b += stat_partial_bytes(d) + 1024;
  return b + 16 * 1024 + crfr_tc_wgrad_part_bytes() + 1024;   // + the wgrad's per-split partial sums
}

// ---------------------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------------------
// the GEMM of recipes 1 / 3 / 5 writes the layer's output: let its epilogue produce the InstanceNorm statistics too
static int gemm_with_stats(TcGemm& g, const crfr_conv_desc* d, Arena& A, float* stats, float eps, int* stats_done,
                           cudaStream_t st) {
  int slots = 0;
  if (stats && stats_done) {
    const size_t bytes = stat_partial_bytes(d);
    if (void* part = A.take(bytes)) {
      g.stat_ws = (float*)part;
      g.stat_ws_bytes = bytes;
      g.stat_slots = &slots;
    }
  }
  CRFR_TRY(crfr_tc_gemm(g, st));
  if (slots) {
    CRFR_TRY(crfr_norm_finalize(g.stat_ws, d->n, slots, d->oh * d->ow, d->cout, eps, stats, st));
    *stats_done = 1;
  }
  return CRFR_OK;
}

int crfr_lowered_fwd(const crfr_conv_desc* d, const void* x, const void* w_packed, int cin_pad, const float* bias,
                     void* y, float* y_nchw, void* ws, size_t ws_bytes, cudaStream_t st, float* stats, float eps,
                     int* stats_done) {
  const int recipe = crfr_lowered_recipe(d);
  Arena A{(uint8_t*)ws, ws_bytes, 0};
  const int T = d->k * d->k;
  if (stats_done) *stats_done = 0;
  if (recipe == 1 || recipe == 3) {
    if (!y || y_nchw) {
      crfr_set_error("lowered conv: recipe %d produces the bf16 NHWC output only", recipe);
      return CRFR_EUNSUPPORTED;
    }
    const int kp = kpad_of(d);
    const long long opix = (long long)d->n * d->oh * d->ow;
    TAKE(P, bf16, A, (size_t)opix * kp * 2);
    TAKE(Wg, bf16, A, (size_t)d->cout * kp * 2);
    CRFR_TRY(launch_im2col_small((const bf16*)x, d->n, d->h, d->w, d->oh, d->ow, d->k, d->stride, d->pad, 1, P, kp, st));
    LAUNCH(repack_tapmajor_kernel, d->cout * kp, st, (const bf16*)w_packed, T, d->cout, 3, cin_pad, Wg, d->cout, kp);
    TcGemm g{P, d->n, d->oh, d->ow, kp, kp, Wg, 1, 0, 1, d->cout, 0, y, d->out_ld, 0, bias};
    return gemm_with_stats(g, d, A, stats, eps, stats_done, st);
  }
  if (recipe == 5) {
    if (!y || y_nchw) {
      crfr_set_error("lowered conv: recipe 5 produces the bf16 NHWC output only");
      return CRFR_EUNSUPPORTED;
    }
    CRFR_CHECK_ARG(cin_pad == d->cin, "lowered conv: cin_pad %d != cin %d", cin_pad, d->cin);
    const int kc = T * d->cin;
    const long long opix = (long long)d->n * d->oh * d->ow;
    TAKE(P, bf16, A, (size_t)opix * kc * 2);
    LAUNCH(im2col_vec_kernel, opix * T * (d->cin / 8), st, (const bf16*)x, d->in_ld, d->cin, d->h, d->w, d->oh, d->ow, d->k,
           d->stride, d->pad, P, opix * T * (d->cin / 8));
    const void* wg = w_packed;   // [1][cout][cin] is already the GEMM weight for 1x1
    if (T > 1) {
      TAKE(Wg, bf16, A, (size_t)d->cout * kc * 2);
      LAUNCH(repack_tapmajor_kernel, d->cout * kc, st, (const bf16*)w_packed, T, d->cout, d->cin, cin_pad, Wg, d->cout, kc);
      wg = Wg;
    }
    TcGemm g{P, d->n, d->oh, d->ow, kc, kc, wg, 1, 0, 1, d->cout, 0, y, d->out_ld, 0, bias};
    return gemm_with_stats(g, d, A, stats, eps, stats_done, st);
  }
  if (recipe == 6 || recipe == 7) {
    if (!y || y_nchw) {
      crfr_set_error("lowered conv: recipe %d produces the bf16 NHWC output only", recipe);
      return CRFR_EUNSUPPORTED;
    }
    CRFR_CHECK_ARG(cin_pad == d->cin, "lowered conv: cin_pad %d != cin %d", cin_pad, d->cin);
    if (recipe == 6) {   // [1][cout][cin] is the GEMM weight
      TcGemm g{x, d->n, d->h, d->w, d->cin, d->in_ld, w_packed, 1, 0, 1, d->cout, 0, y, d->out_ld, 0, bias};
      return gemm_with_stats(g, d, A, stats, eps, stats_done, st);
    }
    // R7: dP[i][tap*cout + co] = sum_ci X[i][ci] W[ci][co][tap] (fp32; w_packed [tap][cout][cin] is that GEMM weight), then
    // y[P][co] = bias + sum over the (input pixel, tap) pairs that reach P, exactly R5's dgrad col2im
    const int kc = 9 * d->cout;
    const long long ipix = (long long)d->n * d->h * d->w, opix = (long long)d->n * d->oh * d->ow;
    TAKE(dP, float, A, (size_t)ipix * kc * 4);
    TcGemm g{x, d->n, d->h, d->w, d->cin, d->in_ld, w_packed, 1, 0, 1, kc, 0, dP, kc, 1, nullptr};
    CRFR_TRY(crfr_tc_gemm(g, st));
    LAUNCH(col2im_vec_kernel, opix * (d->cout / 8), st, dP, d->cout, d->h, d->w, d->oh, d->ow, 3, 2, 1, bias, (bf16*)y,
           d->out_ld, opix * (d->cout / 8));
    return CRFR_OK;
  }
  if (recipe == 2) {
    CRFR_CHECK_ARG(cin_pad == d->cin, "lowered conv: cin_pad %d != cin %d", cin_pad, d->cin);
    const long long pix = (long long)d->n * d->h * d->w;
    const PixGrid pg = valid_flat(d);
    TAKE(Q, float, A, (size_t)pix * 32 * 4);
    TAKE(Wq, bf16, A, (size_t)32 * d->cin * 2);
    CRFR_CUDA(cudaMemsetAsync(Wq, 0, (size_t)32 * d->cin * 2, st));
    CRFR_CUDA(cudaMemcpyAsync(Wq, w_packed, (size_t)27 * d->cin * 2, cudaMemcpyDeviceToDevice, st));   // rows (tap, co)
    TcGemm g{x, pg.n, pg.h, pg.w, d->cin, d->in_ld, Wq, 1, 0, 1, 32, 32, Q, 32, 1, nullptr};
    CRFR_TRY(crfr_tc_gemm(g, st));
    // y[p] = bias + sum_tap Q[p + (tap - pad)][tap*3 + co]
    if (d->pad == 0) {
      const long long opix = (long long)d->n * d->oh * d->ow;
      LAUNCH(col2im_small_kernel, opix, st, Q, 32, 3, d->h, d->w, d->oh, d->ow, 3, 1, 0, -1, bias, y_nchw, (bf16*)y,
             y ? d->out_ld : 0, opix);
      return CRFR_OK;
    }
    if (d->h % 8 == 0 && d->w % 32 == 0) {
      col2im3_s1_kernel<<<(unsigned)(d->n * (d->h / 8) * (d->w / 32)), 256, 0, st>>>(Q, d->h, d->w, -1, bias, y_nchw, (bf16*)y,
                                                                                   y ? d->out_ld : 0);
      CRFR_COUNT_LAUNCH();
      CRFR_LAUNCH_CHECK();
      return CRFR_OK;
    }
    LAUNCH(col2im_small_kernel, pix, st, Q, 32, 3, d->h, d->w, d->h, d->w, 3, 1, 1, -1, bias, y_nchw, (bf16*)y,
           y ? d->out_ld : 0, pix);
    return CRFR_OK;
  }
  if (recipe == 4) {
    if (!y || y_nchw) {
      crfr_set_error("lowered conv: the transposed recipe produces the bf16 NHWC output only");
      return CRFR_EUNSUPPORTED;
    }
    const long long ipix = (long long)d->n * d->h * d->w, opix = (long long)d->n * d->oh * d->ow;
    TAKE(All, bf16, A, (size_t)ipix * 1024 * 2);
    TAKE(Wbig, bf16, A, (size_t)9 * 1024 * 64 * 2);
    TAKE(bbig, float, A, 1024 * 4);
    CRFR_CUDA(cudaMemsetAsync(Wbig, 0, (size_t)9 * 1024 * 64 * 2, st));
    LAUNCH(deconv_subpixel_pack_kernel, 49 * 64 * 64, st, (const bf16*)w_packed, Wbig, 0);
    LAUNCH(deconv_bias_kernel, 1024, st, bias, bbig);
    TcGemm g{x, d->n, d->h, d->w, 64, d->in_ld, Wbig, 3, 1, 1, 1024, 256, All, 1024, 0, bbig};
    CRFR_TRY(crfr_tc_gemm(g, st));
    LAUNCH(deconv_shuffle_kernel, opix * 8, st, (bf16*)y, d->out_ld, All, d->h, d->w, 0, opix * 8);
    return CRFR_OK;
  }
  crfr_set_error("lowered conv: no recipe for this shape");
  return CRFR_EUNSUPPORTED;
}

// ---------------------------------------------------------------------------------------------------------
// dgrad (recipes 2, 3, 4)
// ---------------------------------------------------------------------------------------------------------
int crfr_lowered_dgrad(const crfr_conv_desc* d, const void* dy, const void* w_packed_t, int cout_pad, void* dx, void* ws,
                       size_t ws_bytes, cudaStream_t st) {
  const int recipe = crfr_lowered_recipe(d);
  Arena A{(uint8_t*)ws, ws_bytes, 0};
  const int T = d->k * d->k;
  if (recipe == 2) {
    // dX[q][ci] = sum_k R[q][k] Wd[ci][k],  R[q][tap*3+co] = dY[q - (tap - pad)][co],  Wd[ci][tap*3+co] = W[co][ci][tap]
    const long long pix = (long long)d->n * d->h * d->w;
    const PixGrid pg = valid_flat(d);
    TAKE(R, bf16, A, (size_t)pix * 64 * 2);
    TAKE(Wd, bf16, A, (size_t)d->cin * 64 * 2);
    CRFR_TRY(launch_im2col_small((const bf16*)dy, d->n, d->oh, d->ow, d->h, d->w, 3, 1, d->pad, -1, R, 64, st));
    LAUNCH(repack_tapmajor_kernel, d->cin * 64, st, (const bf16*)w_packed_t, T, d->cin, 3, cout_pad, Wd, d->cin, 64);
    TcGemm g{R, pg.n, pg.h, pg.w, 64, 64, Wd, 1, 0, 1, d->cin, d->cin, dx, d->in_ld, 0, nullptr};
    return crfr_tc_gemm(g, st);
  }
  if (recipe == 6) {   // dX = dY . W, w_packed_t [1][cin][cout]
    CRFR_CHECK_ARG(cout_pad == d->cout, "lowered dgrad: cout_pad %d != cout %d", cout_pad, d->cout);
    TcGemm g{dy, d->n, d->h, d->w, d->cout, d->out_ld, w_packed_t, 1, 0, 1, d->cin, 0, dx, d->in_ld, 0, nullptr};
    return crfr_tc_gemm(g, st);
  }
  if (recipe == 7) {
    // dX[i][ci] = sum_{tap, co} P[i][tap*cout + co] Wd[ci][tap*cout + co],  P = im2col(dY) with R5's geometry (3x3 s2 p1 from
    // the output grid to the input grid),  Wd[ci][tap*cout + co] = W[ci][co][tap] (w_packed_t [tap][cin][cout])
    CRFR_CHECK_ARG(cout_pad == d->cout, "lowered dgrad: cout_pad %d != cout %d", cout_pad, d->cout);
    const int kc = 9 * d->cout;
    const long long ipix = (long long)d->n * d->h * d->w;
    TAKE(P, bf16, A, (size_t)ipix * kc * 2);
    TAKE(Wd, bf16, A, (size_t)d->cin * kc * 2);
    LAUNCH(im2col_vec_kernel, ipix * 9 * (d->cout / 8), st, (const bf16*)dy, d->out_ld, d->cout, d->oh, d->ow, d->h, d->w, 3,
           2, 1, P, ipix * 9 * (d->cout / 8));
    LAUNCH(repack_tapmajor_kernel, d->cin * kc, st, (const bf16*)w_packed_t, T, d->cin, d->cout, cout_pad, Wd, d->cin, kc);
    TcGemm g{P, d->n, d->h, d->w, kc, kc, Wd, 1, 0, 1, d->cin, 0, dx, d->in_ld, 0, nullptr};
    return crfr_tc_gemm(g, st);
  }
  if (recipe == 3) {
    // dP[o][tap*3+c] = sum_co dY[o][co] W[co][c][tap] (fp32), then dx[P][c] = sum over the taps that hit P
    const int kp = kpad_of(d);   // 192
    const long long opix = (long long)d->n * d->oh * d->ow, ipix = (long long)d->n * d->h * d->w;
    TAKE(dP, float, A, (size_t)opix * kp * 4);
    TAKE(Wd, bf16, A, (size_t)kp * d->cout * 2);
    // w_packed_t is [tap][c(3)][cout_pad]: rows (tap, c) are the GEMM weight rows; pad to kp rows of cout
    CRFR_CUDA(cudaMemsetAsync(Wd, 0, (size_t)kp * d->cout * 2, st));
    CRFR_CHECK_ARG(cout_pad == d->cout, "lowered dgrad: cout_pad %d != cout %d", cout_pad, d->cout);
    CRFR_CUDA(cudaMemcpyAsync(Wd, w_packed_t, (size_t)T * 3 * d->cout * 2, cudaMemcpyDeviceToDevice, st));
    TcGemm g{dy, d->n, d->oh, d->ow, d->cout, d->out_ld, Wd, 1, 0, 1, kp, kp == 192 ? 192 : 0, dP, kp, 1, nullptr};
    CRFR_TRY(crfr_tc_gemm(g, st));
    LAUNCH(col2im_small_kernel, ipix, st, dP, kp, 3, d->oh, d->ow, d->h, d->w, d->k, d->stride, d->pad, 1, nullptr, nullptr,
           (bf16*)dx, d->in_ld, ipix);
    return CRFR_OK;
  }
  if (recipe == 5) {
    // dP[o][tap*cin+ci] = sum_co dY[o][co] W[co][ci][tap] (fp32); w_packed_t [tap][ci][cout] is that GEMM weight
    CRFR_CHECK_ARG(cout_pad == d->cout, "lowered dgrad: cout_pad %d != cout %d", cout_pad, d->cout);
    const int kc = T * d->cin;
    const long long opix = (long long)d->n * d->oh * d->ow, ipix = (long long)d->n * d->h * d->w;
    TAKE(dP, float, A, (size_t)opix * kc * 4);
    TcGemm g{dy, d->n, d->oh, d->ow, d->cout, d->out_ld, w_packed_t, 1, 0, 1, kc, 0, dP, kc, 1, nullptr};
    CRFR_TRY(crfr_tc_gemm(g, st));
    LAUNCH(col2im_vec_kernel, ipix * (d->cin / 8), st, dP, d->cin, d->oh, d->ow, d->h, d->w, d->k, d->stride, d->pad,
           nullptr, (bf16*)dx, d->in_ld, ipix * (d->cin / 8));
    return CRFR_OK;
  }
  if (recipe == 4) {
    // dgrad of the sub-pixel convolution: un-shuffle dOut, then the 3x3 conv 1024 -> 64 with the transposed weight
    CRFR_CHECK_ARG(cout_pad == 64, "lowered dgrad: cout_pad %d != 64", cout_pad);
    const long long ipix = (long long)d->n * d->h * d->w, opix = (long long)d->n * d->oh * d->ow;
    TAKE(All, bf16, A, (size_t)ipix * 1024 * 2);
    TAKE(Wbig, bf16, A, (size_t)9 * 64 * 1024 * 2);
    LAUNCH(deconv_shuffle_kernel, opix * 8, st, (bf16*)const_cast<void*>(dy), d->out_ld, All, d->h, d->w, 1, opix * 8);
    CRFR_CUDA(cudaMemsetAsync(Wbig, 0, (size_t)9 * 64 * 1024 * 2, st));
    LAUNCH(deconv_subpixel_pack_kernel, 49 * 64 * 64, st, (const bf16*)w_packed_t, Wbig, 1);
    TcGemm g{All, d->n, d->h, d->w, 1024, 1024, Wbig, 3, 1, -1, 64, 64, dx, d->in_ld, 0, nullptr};
    return crfr_tc_gemm(g, st);
  }
  crfr_set_error("lowered dgrad: no recipe for this shape");
  return CRFR_EUNSUPPORTED;
}

// dgrad of recipe 1's shape (3x3 s1 p1, 3 -> cout channels), a 3x3 cout -> 3 convolution of dY: recipe 2's forward GEMM
// with the transposed pack [tap][ci(3)][cout] as its weight rows (tap*3 + ci), then the col2im over the taps in the
// opposite direction.  dX[q][ci] = sum_tap Q[q + (pad - tap)][tap*3 + ci],  Q[p][tap*3 + ci] = sum_co dY[p][co] W[co][ci][tap]
size_t crfr_lowered_dgrad_cin3_ws_bytes(const crfr_conv_desc* d) {
  return (size_t)d->n * d->h * d->w * 32 * 4 + (size_t)32 * 64 * 2 + 4096;
}

int crfr_lowered_dgrad_cin3(const crfr_conv_desc* d, const void* dy, const void* w_packed_t, void* dx, void* ws,
                            size_t ws_bytes, cudaStream_t st) {
  if (crfr_lowered_recipe(d) != 1 || d->cout != 64 || d->out_ld != 64 || d->h % 8) {
    crfr_set_error("lowered dgrad (3-channel input): unsupported shape");
    return CRFR_EUNSUPPORTED;
  }
  Arena A{(uint8_t*)ws, ws_bytes, 0};
  const long long pix = (long long)d->n * d->h * d->w;
  TAKE(Q, float, A, (size_t)pix * 32 * 4);
  TAKE(Wq, bf16, A, (size_t)32 * 64 * 2);
  CRFR_CUDA(cudaMemsetAsync(Wq, 0, (size_t)32 * 64 * 2, st));
  CRFR_CUDA(cudaMemcpyAsync(Wq, w_packed_t, (size_t)27 * 64 * 2, cudaMemcpyDeviceToDevice, st));
  TcGemm g{dy, d->n, d->h, d->w, 64, d->out_ld, Wq, 1, 0, 1, 32, 32, Q, 32, 1, nullptr};
  CRFR_TRY(crfr_tc_gemm(g, st));
  col2im3_s1_kernel<<<(unsigned)(d->n * (d->h / 8) * ((d->w + 31) / 32)), 256, 0, st>>>(Q, d->h, d->w, 1, nullptr, nullptr,
                                                                                       (bf16*)dx, d->in_ld);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  return CRFR_OK;
}

// ---------------------------------------------------------------------------------------------------------
// wgrad (all recipes); dw is accumulated (+=)
// ---------------------------------------------------------------------------------------------------------
int crfr_lowered_wgrad(const crfr_conv_desc* d, const void* x, const void* dy, float* dw, void* ws, size_t ws_bytes,
                       cudaStream_t st) {
  const int recipe = crfr_lowered_recipe(d);
  Arena A{(uint8_t*)ws, ws_bytes, 0};
  const int T = d->k * d->k;
  if (recipe == 1 || recipe == 3) {
    const int kp = kpad_of(d);
    const long long opix = (long long)d->n * d->oh * d->ow;
    TAKE(P, bf16, A, (size_t)opix * kp * 2);
    TAKE(G, float, A, (size_t)kp * d->cout * 4);
    CRFR_TRY(launch_im2col_small((const bf16*)x, d->n, d->h, d->w, d->oh, d->ow, d->k, d->stride, d->pad, 1, P, kp, st));
    CRFR_CUDA(cudaMemsetAsync(G, 0, (size_t)kp * d->cout * 4, st));
    TcWgrad g{P, d->n, d->oh, d->ow, kp, kp, dy, d->cout, d->out_ld, 0, G};
    A.rest(&g.part, &g.part_bytes);
    CRFR_TRY(crfr_tc_wgrad_raw(g, st));
    LAUNCH(unpack_lowered_kernel, (long long)d->cout * 3 * T, st, G, d->cout, dw, d->cout, 3, T, 0);
    return CRFR_OK;
  }
  if (recipe == 5) {
    const int kc = T * d->cin;
    const long long opix = (long long)d->n * d->oh * d->ow;
    TAKE(P, bf16, A, (size_t)opix * kc * 2);
    TAKE(G, float, A, (size_t)kc * d->cout * 4);
    LAUNCH(im2col_vec_kernel, opix * T * (d->cin / 8), st, (const bf16*)x, d->in_ld, d->cin, d->h, d->w, d->oh, d->ow, d->k,
           d->stride, d->pad, P, opix * T * (d->cin / 8));
    CRFR_CUDA(cudaMemsetAsync(G, 0, (size_t)kc * d->cout * 4, st));
    TcWgrad g{P, d->n, d->oh, d->ow, kc, kc, dy, d->cout, d->out_ld, 0, G};
    A.rest(&g.part, &g.part_bytes);
    CRFR_TRY(crfr_tc_wgrad_raw(g, st));
    LAUNCH(unpack_lowered_kernel, (long long)d->cout * d->cin * T, st, G, d->cout, dw, d->cout, d->cin, T, 0);
    return CRFR_OK;
  }
  if (recipe == 2) {
    const long long pix = (long long)d->n * d->h * d->w;
    const PixGrid pg = valid_flat(d);
    TAKE(R, bf16, A, (size_t)pix * 64 * 2);
    TAKE(G, float, A, (size_t)d->cin * 64 * 4);
    CRFR_TRY(launch_im2col_small((const bf16*)dy, d->n, d->oh, d->ow, d->h, d->w, 3, 1, d->pad, -1, R, 64, st));
    CRFR_CUDA(cudaMemsetAsync(G, 0, (size_t)d->cin * 64 * 4, st));
    TcWgrad g{x, pg.n, pg.h, pg.w, d->cin, d->in_ld, R, 64, 64, 0, G};
    A.rest(&g.part, &g.part_bytes);
    CRFR_TRY(crfr_tc_wgrad_raw(g, st));
    LAUNCH(unpack_lowered_kernel, (long long)3 * d->cin * T, st, G, 64, dw, 3, d->cin, T, 1);
    return CRFR_OK;
  }
  if (recipe == 6) {   // G[ci][co] = X^T dY
    TAKE(G, float, A, (size_t)d->cin * d->cout * 4);
    CRFR_CUDA(cudaMemsetAsync(G, 0, (size_t)d->cin * d->cout * 4, st));
    TcWgrad g{x, d->n, d->h, d->w, d->cin, d->in_ld, dy, d->cout, d->out_ld, 0, G};
    A.rest(&g.part, &g.part_bytes);
    CRFR_TRY(crfr_tc_wgrad_raw(g, st));
    LAUNCH(unpack_lowered_kernel, (long long)d->cout * d->cin, st, G, d->cout, dw, d->cout, d->cin, 1, 0);
    return CRFR_OK;
  }
  if (recipe == 7) {
    // G[tap*cout + co][ci] = sum_i P[i][tap*cout + co] X[i][ci] with P = im2col(dY) as in the dgrad; dW[ci][co][tap] += G
    const int kc = 9 * d->cout;
    const long long ipix = (long long)d->n * d->h * d->w;
    TAKE(P, bf16, A, (size_t)ipix * kc * 2);
    TAKE(G, float, A, (size_t)kc * d->cin * 4);
    CRFR_CUDA(cudaMemsetAsync(G, 0, (size_t)kc * d->cin * 4, st));
    LAUNCH(im2col_vec_kernel, ipix * 9 * (d->cout / 8), st, (const bf16*)dy, d->out_ld, d->cout, d->oh, d->ow, d->h, d->w, 3,
           2, 1, P, ipix * 9 * (d->cout / 8));
    TcWgrad g{P, d->n, d->h, d->w, kc, kc, x, d->cin, d->in_ld, 0, G};
    A.rest(&g.part, &g.part_bytes);
    CRFR_TRY(crfr_tc_wgrad_raw(g, st));
    LAUNCH(unpack_lowered_kernel, (long long)d->cin * d->cout * 9, st, G, d->cin, dw, d->cin, d->cout, 9, 0);
    return CRFR_OK;
  }
  if (recipe == 4) {
    const long long ipix = (long long)d->n * d->h * d->w, opix = (long long)d->n * d->oh * d->ow;
    TAKE(All, bf16, A, (size_t)ipix * 1024 * 2);
    TAKE(G, float, A, (size_t)9 * 64 * 1024 * 4);
    LAUNCH(deconv_shuffle_kernel, opix * 8, st, (bf16*)const_cast<void*>(dy), d->out_ld, All, d->h, d->w, 1, opix * 8);
    CRFR_CUDA(cudaMemsetAsync(G, 0, (size_t)9 * 64 * 1024 * 4, st));
    TcWgrad g{x, d->n, d->h, d->w, 64, d->in_ld, All, 1024, 1024, 1, G};
    A.rest(&g.part, &g.part_bytes);
    CRFR_TRY(crfr_tc_wgrad_raw(g, st));
    LAUNCH(deconv_subpixel_unpack_kernel, 64 * 64 * 49, st, G, dw);
    return CRFR_OK;
  }
  crfr_set_error("lowered wgrad: no recipe for this shape");
  return CRFR_EUNSUPPORTED;
}
