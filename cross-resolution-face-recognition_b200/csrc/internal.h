// Internal (non-ABI) entry points shared between translation units.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

#include "crfr.h"

#ifdef __cplusplus
#include <atomic>
#endif

// ---- process-wide implementation switches (conv_api.cu).  Every setting computes equivalent results: each switch selects
// a reference implementation that tests compare against, or a serial schedule for profiles.  Defaults come from the
// environment (CRFR_ROWCONV_PAIR, CRFR_WGRAD_STREAM, CRFR_NORM_BWD=regs|stream, CRFR_NORM_FWD_STREAM, CRFR_FUSE_NORM_BWD)
// once; crfr_set_option overrides atomically.
enum {
  CRFR_OPT_ROWCONV_PAIR = 0, // cta_group::2 form of the row-streaming forward / dgrad kernel (even image counts)
  CRFR_OPT_WGRAD_STREAM,     // FSRNet backward: weight gradients on a helper stream
  CRFR_OPT_NORM_BWD_STREAM,  // TMA-fed normalisation backward (else register-staged)
  CRFR_OPT_NORM_FWD_STREAM,  // TMA-fed normalisation forward
  CRFR_OPT_FUSE_NORM_BWD,    // crfr_conv_dgrad_norm_bwd: first pass of the normalisation backward in the dgrad epilogue
  CRFR_OPT_COUNT
};
int crfr_opt(int id);

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per DEVICE: remember which devices have it (one process may drive
// several GPUs), and cache the SM count per device likewise.
template <typename K>
inline int crfr_smem_attr(K kernel, int bytes, std::atomic<unsigned long long>& done) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) dev = -1;
  const unsigned long long bit = (dev >= 0 && dev < 64) ? 1ull << dev : 0ull;
  if (bit && (done.load(std::memory_order_acquire) & bit)) return 0;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) return (int)e;
  if (bit) done.fetch_or(bit, std::memory_order_release);
  return 0;
}
int crfr_sm_count();   // SMs of the current device (cached per device)

// tmap.cu: bf16 / SWIZZLE_128B / zero-fill tensor map of rank <= 5; strides_bytes has rank-1 entries (dimension 0 is
// contiguous).  CUtensorMap comes from <cuda.h> (included by every caller through sm100.cuh / cudaTypedefs.h).
struct CUtensorMap_st;
int crfr_tmap_encode_bf16(CUtensorMap_st* m, const void* ptr, int rank, const unsigned long long* dims,
                          const unsigned long long* strides_bytes, const unsigned int* box, const char* what);

// layout.cu: dst[t][r][s] (bf16, s padded to s_pad) = src[r * rs + s * ss + t] (* rscale[r]) (* sscale[s]) for a list of
// jobs, 64 per launch.  The optional fp32 scales fold a per-channel factor (an eval-mode BatchNorm's gamma * rstd) into the
// weights before the one rounding to bf16.
#define CRFR_PACK_BATCH 64
struct crfr_pack_job {
  const float* src; void* dst;
  int T, R, S, s_pad;
  long long rs, ss;
  int block0, reserved;   // filled by the launcher
  const float* rscale = nullptr;
  const float* sscale = nullptr;
};
struct crfr_pack_batch {
  crfr_pack_job job[CRFR_PACK_BATCH];
  int njobs;
};
int crfr_pack_weight_batch(const crfr_pack_job* jobs, int n, cudaStream_t st);

// norm_act.cu
size_t crfr_norm_ws_bytes(int n, int hw, int c);
int crfr_norm_finalize(const float* partial, int n, int chunks, int hw, int c, float eps, float* stats,
                       cudaStream_t st);
// second half of the normalisation backward (fold of the first pass' partials [n][chunks][3][c] + apply pass); bstats
// [n][c][2] and tot [n][3][c] are scratch.  dsrc = dz, or dout with recompute != 0.
int crfr_norm_bwd_finish(const float* partial, int chunks, const void* dsrc, int dsrc_ld, int recompute, const void* y,
                         int y_ld, const float* stats, const float* gamma, const float* beta, const float* alpha, int relu,
                         void* dy, int dy_ld, float* dgamma, float* dbeta, float* dalpha, int n, int hw, int c,
                         float* bstats, float* tot, int use_stream, cudaStream_t st);

// norm_stream.cu: TMA-fed reduce / apply passes of the normalisation backward (same contract as the kernels in
// norm_act.cu; views = the tensors the passes touch, checked for TMA alignment)
int crfr_norm_stream_supported(int c, long long npix, const void* const* views, const int* lds, int count);
int crfr_norm_stream_parts(int n, int hw, int c);   // partial slots per image ([n][parts][3][c] floats), 0 = unsupported
int crfr_norm_bwd_reduce_stream(const void* da, int da_ld, const void* db, int db_ld, const void* y, int y_ld,
                                const float* stats, const float* gamma, const float* beta, const float* alpha, int relu,
                                const void* res, int res_ld, void* dz, int dz_ld, int n, int hw, int c, float* partial,
                                cudaStream_t st);
// (bstats / tot NULL: the apply pass folds the first pass' partial sums [n][parts][3][c] itself, no separate fold launch)
int crfr_norm_bwd_apply_stream(const void* dsrc, int dsrc_ld, int recompute, const void* y, int y_ld, const float* stats,
                               const float* partial, int parts, const float* bstats, const float* tot,
                               const float* gamma, const float* beta,
                               const float* alpha, int relu, void* dy, int dy_ld, float* dgamma, float* dbeta,
                               float* dalpha, int n, int hw, int c, cudaStream_t st);

int crfr_norm_fwd_stream(const void* y, int y_ld, const float* stats, const float* gamma, const float* beta,
                         const float* alpha, int relu, const void* res, int res_ld, void* out, int out_ld, int n, int hw,
                         int c, cudaStream_t st);

// losses.cu: MSE*97 loss with the fp32 per-channel sums of its gradient (bias gradient of the producing convolution),
// and the same sums for an explicit fp32 NCHW gradient
int crfr_loss_mse97_chan(const float* x, const float* t, int n, int c, int hw, float gscale, float* loss, void* dx,
                         int dx_ld, float* dchan, void* ws, size_t ws_bytes, cudaStream_t st);
int crfr_nchw_chansum(const float* g, int n, int c, int hw, float* out, void* ws, size_t ws_bytes, cudaStream_t st);

// direct_conv.cu
int crfr_direct_gather(int down, int n, int bh, int bw, int sh, int sw, int k, int stride, int pad, const void* src,
                       int src_ld, const void* w, int R, int s_pad, const float* bias, void* y, int y_ld,
                       float* y_nchw, cudaStream_t st);
int crfr_direct_wgrad(int n, int bh, int bw, int sh, int sw, int k, int stride, int pad, const void* small,
                      int small_ld, int A, const void* big, int big_ld, int B, float* G, void* ws, size_t ws_bytes, cudaStream_t st);
// out[c] += sum over pixels of t[pix][c]; per-chunk partials in ws (at least c floats), summed in a fixed order
int crfr_colsum(const void* t, int ld, int c, long long npix, float* out, void* ws, size_t ws_bytes, cudaStream_t st);

// tc_conv.cu: generic tcgen05 launchers used by the lowered (im2col) edge layers
struct TcGemm {           // out[pixel][n] = bias[n] + sum_{tap,k} src[pixel + sign*(tap - pad)][k] * w[tap][n][k]
  const void* src; int n, h, w, k_total, src_ld;
  const void* wt;         // bf16 [ksize*ksize][n_total][k_total]
  int ksize, pad, sign;
  int n_total, tile_n;    // tile_n = 0: pick automatically
  void* out; int out_ld, out_f32;
  const float* bias;
  // optional fused InstanceNorm statistics of the stored bf16 output: partial sums [n][slots][2][n_total] are written
  // to stat_ws when the tiling allows it and *stat_slots is set to the slot count (0: not fused, caller runs a pass)
  float* stat_ws = nullptr; size_t stat_ws_bytes = 0; int* stat_slots = nullptr;
  // stat_batch: ONE statistic group over the whole batch (BatchNorm): partial sums [1][tiles x 4][2][n_total], any tiling (rows
  // of a tile that lie outside the tensor are masked out); needs bias == nullptr
  int stat_batch = 0;
};
int crfr_tc_gemm(const TcGemm& g, cudaStream_t st);
struct TcWgrad {          // G[tap][ci][co] = sum_pixel x[pixel + tap - 1][ci] * dy[pixel][co]   (fp32, G is overwritten)
  const void* x; int n, h, w, cin, x_ld;
  const void* dy; int cout, dy_ld;
  int taps3x3;            // 1: 3x3 pad 1 (9 taps), 0: single tap
  float* G;
  // per-split partial sums, added into G in a fixed order (no float atomics): the pixel dimension is split only as far
  // as this buffer holds; crfr_tc_wgrad_part_bytes() bytes always suffice for the full split
  float* part = nullptr;
  size_t part_bytes = 0;
};
int crfr_tc_wgrad_raw(const TcWgrad& g, cudaStream_t st);
size_t crfr_tc_wgrad_part_bytes();

// tc_conv.cu (tcgen05 engine).  op: 0 = forward, 1 = dgrad, 2 = wgrad
int crfr_tc_supported(int op, int h, int w, int cin, int cout, int k, int stride, int pad);
size_t crfr_tc_workspace_bytes(const crfr_conv_desc* d);
int crfr_tc_conv(const crfr_conv_desc* d, int dgrad, const void* src, const void* w_packed, const float* bias,
                 void* dst, float* stats, float eps, void* ws, size_t ws_bytes, cudaStream_t st, int batch_stats = 0);
// conv_api.cu: forward convolution (no bias, bf16 output) + train-mode BatchNorm statistics [cout][2] = (mean, rstd) over
// the whole batch, from the convolution's epilogue where the tile engine runs the layer (else a separate pass)
int crfr_conv_fwd_bnstats(int engine, const crfr_conv_desc* d, const void* x, const void* w_packed, int cin_pad, void* y,
                          float* bn_stats, float eps, void* ws, size_t ws_bytes, cudaStream_t st);
int crfr_tc_wgrad(const crfr_conv_desc* d, const void* x, const void* dy, float* dw, void* ws, size_t ws_bytes,
                  cudaStream_t st);

// lowered_conv.cu: edge layers as [gather kernel] + [tcgen05 GEMM]; recipe 0 = not applicable
int crfr_lowered_recipe(const crfr_conv_desc* d);
size_t crfr_lowered_ws_bytes(const crfr_conv_desc* d);
// stats != nullptr: InstanceNorm statistics of the stored output where the GEMM's tiling can produce them in its epilogue;
// *stats_done says whether it did (0: the caller runs crfr_norm_stats over y)
int crfr_lowered_fwd(const crfr_conv_desc* d, const void* x, const void* w_packed, int cin_pad, const float* bias,
                     void* y, float* y_nchw, void* ws, size_t ws_bytes, cudaStream_t st, float* stats = nullptr,
                     float eps = 0.f, int* stats_done = nullptr);
int crfr_lowered_dgrad(const crfr_conv_desc* d, const void* dy, const void* w_packed_t, int cout_pad, void* dx, void* ws,
                       size_t ws_bytes, cudaStream_t st);
int crfr_lowered_wgrad(const crfr_conv_desc* d, const void* x, const void* dy, float* dw, void* ws, size_t ws_bytes,
                       cudaStream_t st);
// dgrad of recipe 1's shape (3-channel input, 3x3 s1) on the tcgen05 GEMM; crfr_conv_dgrad keeps the direct kernel there
size_t crfr_lowered_dgrad_cin3_ws_bytes(const crfr_conv_desc* d);
int crfr_lowered_dgrad_cin3(const crfr_conv_desc* d, const void* dy, const void* w_packed_t, void* dx, void* ws,
                            size_t ws_bytes, cudaStream_t st);

// rowconv.cu: persistent row-streaming kernel for 3x3 64->64 convolutions at width 128
int crfr_rowconv_supported(int h, int w, int cin, int cout, int k, int stride, int pad);
size_t crfr_rowconv_ws_bytes(int n, int h);
// rowconv2.cu: cta_group::2 form of the same kernel (two CTAs walk the same rows of two images); n must be even
int crfr_rowconv_pair_supported(int n, int h);
size_t crfr_rowconv_pair_ws_bytes(int n, int h);
// optional fusion of the first pass of a normalisation backward into the dgrad epilogue: the convolution's input was
// out = act(gamma * (y - mean) * rstd + beta (+ res)); with D = dgrad output (+ db) the kernel stores dz = D * act'(z)
// instead of the dgrad output and the partial sums of (dz, dz * xhat, D * min(z, 0)) per (image, channel)
struct crfr_rowconv_fuse {
  const void* y; int y_ld;        // raw map the normalisation read (same pixels as the dgrad output)
  const void* db; int db_ld;      // second gradient of the normalised tensor, or NULL
  const void* res; int res_ld;    // residual input of the normalisation, or NULL
  const float* stats; const float* gamma; const float* beta; const float* alpha; int relu;
  float* partial;                 // out: [n][crfr_rowconv_pair_parts(n, h, !db && !res)][3][64]
};
int crfr_rowconv_pair_parts(int n, int h, int plain = 0);   // partial slots per image of the fused pass (plain: no db / res)
int crfr_rowconv_pair(const void* src, int src_ld, int n, int h, const void* w_packed, int flip, const float* bias,
                      void* dst, int dst_ld, float* stats, float eps, void* ws, size_t ws_bytes, cudaStream_t st,
                      const crfr_rowconv_fuse* fuse = nullptr);
// rowwgrad.cu: persistent row-streaming weight gradient of the same shape (deterministic slab reduction)
int crfr_rowwgrad_supported(int h, int w, int cin, int cout, int k, int stride, int pad);
size_t crfr_rowwgrad_ws_bytes(int n, int h);
int crfr_rowwgrad(const void* x, int x_ld, const void* dy, int dy_ld, int n, int h, float* dw, void* ws,
                  size_t ws_bytes, cudaStream_t st);
int crfr_rowconv(const void* src, int src_ld, int n, int h, const void* w_packed, int flip, const float* bias, void* dst,
                 int dst_ld, float* stats, float eps, void* ws, size_t ws_bytes, cudaStream_t st);
