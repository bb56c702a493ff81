/* crfr.h - C-ABI of the B200-native hot path of HyoKong/Cross-Resolution-Face-Recognition.
 *
 * The reference has no FFI: its operator API is torch.nn.Module.__call__ + state_dict (SURVEY.md 8b).  Every entry
 * point below replaces the ATen/cuDNN (or Pillow / numpy) call sequence behind one reference site, cited as
 * "ref:" (paths relative to the reference root).  The Python host mirror (package crfr_b200) binds these with
 * ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless named host_*;
 *   - the caller owns all memory (inputs, outputs, workspace); the library never allocates device memory and
 *     keeps no pointer past return;
 *   - every call only enqueues work on `stream` (a cudaStream_t passed as void*) and returns immediately;
 *   - return value: 0 = ok, non-zero = error code; message via crfr_last_error() (thread-local);
 *   - activations are NHWC bf16 with an explicit per-pixel stride `ld` (elements) so that a tensor can be a channel
 *     slice of a wider buffer (this is how torch.cat at model/FSRnet.py:505 is eliminated);
 *   - parameters and parameter gradients are fp32 in the reference's own layouts (OIHW etc.); gradients are
 *     ACCUMULATED (+=) because the reference shares one module across several call sites (FSRnet.py:331-333).
 */
#ifndef CRFR_H_
#define CRFR_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CRFR_ENGINE_AUTO 0
#define CRFR_ENGINE_DIRECT 1   /* CUDA-core direct kernels (edge shapes, cross-check) */
#define CRFR_ENGINE_TCGEN05 2  /* tcgen05/TMEM implicit GEMM fed by TMA */

const char* crfr_last_error(void);
int crfr_version(void);
/* number of kernel launches issued by this library in this process (bench.py reports it as gpu_launches) */
unsigned long long crfr_launch_count(void);
/* Implementation switches for tests and profiles (results are equivalent either way); any other name is CRFR_EINVAL:
 *   "rowconv_pair":  3x3 64 -> 64 convolutions at width 128 (forward and dgrad) with an even image count as 1 = the
 *                    cta_group::2 kernel that pairs two CTAs (default), 0 = the single-CTA kernel; identical bits.
 *   "wgrad_stream":  FSRNet backward, weight gradients as 1 = on a helper stream behind each layer's dgrad (default),
 *                    0 = serially on the caller's stream (for profiles whose kernel times add up).
 *   "norm_bwd_impl": crfr_norm_act_bwd as 0 = register-staged reduce + fold + apply kernels, 1 = persistent TMA-fed
 *                    reduce + fold + apply kernels (default where the views are TMA-addressable: channels a multiple
 *                    of 64, 16-byte aligned), -1 = default / environment CRFR_NORM_BWD=regs|stream.
 *   "norm_fwd_stream": crfr_norm_act_fwd as 0 = register-staged kernel, 1 = persistent TMA-fed kernel (default where the
 *                    views are TMA-addressable); identical results bit for bit.
 *   "fuse_norm_bwd": crfr_conv_dgrad_norm_bwd as 0 = dgrad + crfr_norm_act_bwd, 1 = first pass of the normalisation
 *                    backward inside the dgrad epilogue where the row-streaming pair kernel runs (default). */
int crfr_set_option(const char* name, int value);
/* 1 if the engine can run the shape (h,w,cin,cout,k,stride,pad), else 0 */
int crfr_conv_engine_supported(int engine, int op, int h, int w, int cin, int cout, int k, int stride, int pad);

/* ---------------------------------------------------------------- layout ---------------------------------- */
/* ref: the NCHW fp32 tensors at the nn.Module boundary (model/FSRnet.py:497, model/resnet.py:208) */
int crfr_nchw_f32_to_nhwc_bf16(const float* src, void* dst, int n, int c, int h, int w, int dst_ld, int c_zero_to,
                               void* stream);
int crfr_nhwc_bf16_to_nchw_f32(const void* src, float* dst, int n, int c, int h, int w, int src_ld, void* stream);
/* dst[t][r][s] (bf16, s padded with zeros up to s_pad) = src[r*r_stride + s*s_stride + t*t_stride] (fp32) */
int crfr_pack_weight(const float* src, void* dst, int T, int R, int S, int s_pad, long long r_stride,
                     long long s_stride, long long t_stride, void* stream);

/* ---------------------------------------------------------------- convolutions ---------------------------- */
typedef struct crfr_conv_desc {
  int n, h, w;        /* input batch / spatial size            */
  int cin, cout;      /* logical channel counts                */
  int k, stride, pad; /* square kernel                         */
  int oh, ow;         /* output spatial size                   */
  int in_ld, out_ld;  /* per-pixel strides of x and y (elems)  */
  int transposed;     /* 0: Conv2d, 1: ConvTranspose2d         */
} crfr_conv_desc;

/* ref: nn.Conv2d / nn.ConvTranspose2d forward at model/FSRnet.py:79,85,110,114,312,318,345,351,384,391,392,432,436,439
 *      and model/resnet.py:23-26,158,196; the SUPER_RESOLUTION variant's layers (SUPER_RESOLUTION/model/FSRnet.py:251-416).
 * Shapes on the tcgen05 engine (ENGINE_AUTO picks them, ENGINE_TCGEN05 rejects the others with CRFR_EUNSUPPORTED; the
 * same for crfr_conv_dgrad / crfr_conv_wgrad unless noted; ENGINE_DIRECT runs every shape on CUDA cores):
 *   3x3 s1 pad 1 or 0, cin / cout multiples of 64 (wgrad: cout 64 or a multiple of 128);
 *   3x3 s2 pad 1 or 0 and 1x1 s2 / 1x1 s1 pad 0, channels multiples of 64;
 *   ConvTranspose2d 3x3 s2 pad 1 output_padding 1 and 7x7 s4 pad 2 output_padding 1 (64 -> 64), channels multiples of 64;
 *   3-channel input: 3x3 s1 pad 1 or 0 (cout a multiple of 64 up to 256; dgrad on CUDA cores), 7x7 s4 / s2 pad 3 and
 *   7x7 s1 pad 0 (cout 64 or 128);  3-channel output: 3x3 s1 pad 1 (cin 64) or pad 0 (cin 64 or 128).
 * A 1x1 layer with an output channel count that is not a multiple of 64 (the 11 / 13 / 68-channel heads) runs on CUDA
 * cores.  crfr_conv_engine_supported reports the Conv2d shapes (it has no transposed flag).
 * x: NHWC bf16.  w_packed: bf16 [k*k][cout][cin_pad] made by crfr_pack_weight.  bias: fp32 [cout] or NULL.
 * y: NHWC bf16 or NULL.  y_nchw: fp32 NCHW [n][cout][oh][ow] or NULL.
 * stats: fp32 [n][cout][2] = (mean, rstd) of y over (oh,ow) per (n, channel) - the InstanceNorm statistics
 *        (FSRnet.py:81) computed from the stored (bf16-rounded) values; NULL to skip. */
int crfr_conv_fwd(int engine, const crfr_conv_desc* d, const void* x, const void* w_packed, int cin_pad,
                  const float* bias, void* y, float* y_nchw, float* stats, float eps, void* ws, size_t ws_bytes,
                  void* stream);
/* dx = gradient w.r.t. x.  w_packed_t: bf16 [k*k][cin][cout_pad].  dx: NHWC bf16 with stride d->in_ld. */
int crfr_conv_dgrad(int engine, const crfr_conv_desc* d, const void* dy, const void* w_packed_t, int cout_pad,
                    void* dx, void* ws, size_t ws_bytes, void* stream);
/* dw (fp32, reference layout: Conv2d [cout][cin][k][k], ConvTranspose2d [cin][cout][k][k]) += ...; dbias += sum dy.
 * Both are reduced in a fixed order (no float atomics): two calls give the same bits. */
int crfr_conv_wgrad(int engine, const crfr_conv_desc* d, const void* x, const void* dy, float* dw, float* dbias,
                    void* ws, size_t ws_bytes, void* stream);
/* scratch for any of the three calls on d; a smaller workspace is CRFR_EWORKSPACE where the path needs one */
size_t crfr_conv_workspace_bytes(const crfr_conv_desc* d);

/* ---------------------------------------------------------------- normalisation + activation -------------- */
/* ref: nn.InstanceNorm2d (FSRnet.py:81,87,112,115,319,347,385,434), nn.PReLU (:84,88,113,314,346,386,433),
 *      residual add (:96,132); with groups==1 over the whole batch it is train-mode nn.BatchNorm2d + ReLU
 *      (model/resnet.py:24-28).
 * stats[n][c][2] (mean, rstd) over hw pixels of image n.
 * crfr_norm_workspace_bytes: scratch needed by crfr_norm_stats / crfr_norm_act_bwd for this shape. */
size_t crfr_norm_workspace_bytes(int n, int hw, int c);
int crfr_norm_stats(const void* y, int n, int hw, int c, int ld, float eps, float* stats, void* ws, size_t ws_bytes,
                    void* stream);
/* out = act(gamma*(y-mean)*rstd + beta + res); gamma/beta NULL = non-affine; alpha NULL = no activation;
 * alpha_is_relu != 0 -> ReLU (alpha ignored). res NULL = no residual. */
int crfr_norm_act_fwd(const void* y, int y_ld, const float* stats, const float* gamma, const float* beta,
                      const float* alpha, int relu, const void* res, int res_ld, void* out, int out_ld, int n,
                      int hw, int c, void* stream);
/* dout = dout_a (+ dout_b).  Outputs: dz (grad wrt pre-activation, == grad wrt res; may be NULL when res and dout_b
 * are NULL: it is then neither stored nor re-read, which saves one full map of HBM traffic), dy (grad wrt conv
 * output), dgamma/dbeta/dalpha fp32 [c] accumulated (NULL to skip). */
int crfr_norm_act_bwd(const void* dout_a, int da_ld, const void* dout_b, int db_ld, const void* y, int y_ld,
                      const float* stats, const float* gamma, const float* beta, const float* alpha, int relu,
                      const void* res, int res_ld, void* dz, int dz_ld, void* dy, int dy_ld, float* dgamma,
                      float* dbeta, float* dalpha, int n, int hw, int c, void* ws, size_t ws_bytes, void* stream);

/* Backward of "conv(act(norm(y) (+ res)))" across the convolution's input, as one operation (ref: the
 * InstanceNorm2d -> PReLU -> Conv2d and InstanceNorm2d -> add -> PReLU -> Conv2d chains of _Residual_Block,
 * model/FSRnet.py:91-97):  D = dgrad(dout) (+ dx_b, a further gradient of the convolution's input from its other
 * consumers, or NULL); then exactly crfr_norm_act_bwd on D: dz = D * act'(z) (always written: it is the gradient of
 * `res`), dy, dgamma / dbeta / dalpha accumulated.  Same results as crfr_conv_dgrad followed by crfr_norm_act_bwd (the
 * fp32 sums may associate differently).  For the row-streaming shapes (3x3 s1 64 -> 64 at width 128, even image
 * count) the first pass of the normalisation backward runs inside the dgrad epilogue (option "fuse_norm_bwd", default
 * 1): the dgrad output never reaches memory and one pass over 2-4 maps disappears; other shapes run the two calls.
 * ws >= crfr_conv_dgrad_norm_bwd_workspace_bytes(d). */
size_t crfr_conv_dgrad_norm_bwd_workspace_bytes(const crfr_conv_desc* d);
int crfr_conv_dgrad_norm_bwd(int engine, const crfr_conv_desc* d, const void* dout, const void* w_packed_t, int cout_pad,
                             const void* dx_b, int dxb_ld, const void* y, int y_ld, const float* stats,
                             const float* gamma, const float* beta, const float* alpha, int relu, const void* res,
                             int res_ld, void* dz, int dz_ld, void* dy, int dy_ld, float* dgamma, float* dbeta,
                             float* dalpha, void* ws, size_t ws_bytes, void* stream);

/* ref: train-mode nn.BatchNorm2d / BatchNorm1d buffer update (model/resnet.py:24,27,159,167,172):
 * running = (1-momentum)*running + momentum*batch, with the unbiased batch variance (count = N*H*W samples);
 * stats is the [c][2] (mean, rstd) produced by crfr_norm_stats with n = 1.  num_batches_tracked (int64, may be NULL) += 1. */
int crfr_bn_update_running(const float* stats, float* running_mean, float* running_var,
                           long long* num_batches_tracked, int c, long long count, float momentum, float eps,
                           void* stream);
/* eval-mode BatchNorm: stats[c][2] = (running_mean, 1/sqrt(running_var + eps)), to be used with crfr_norm_act_fwd */
int crfr_bn_running_to_stats(const float* running_mean, const float* running_var, int c, float eps, float* stats,
                             void* stream);

/* ---------------------------------------------------------------- hourglass resampling --------------------- */
/* ref: F.max_pool2d(x,2,2) FSRnet.py:202 ; F.interpolate(scale_factor=2)+add :210-211 */
int crfr_maxpool2_fwd(const void* x, int x_ld, void* out, int out_ld, int n, int h, int w, int c, void* stream);
int crfr_maxpool2_bwd(const void* x, int x_ld, const void* dout, int dout_ld, void* dx, int dx_ld, int n, int h,
                      int w, int c, void* stream);
int crfr_upnearest2_add_fwd(const void* up, int up_ld, const void* low, int low_ld, void* out, int out_ld, int n,
                            int h, int w, int c, void* stream); /* h,w: size of `low`; out is 2h x 2w */
int crfr_upnearest2_bwd(const void* dout, int dout_ld, void* dlow, int dlow_ld, int n, int h, int w, int c,
                        void* stream);
/* out = a + b (+ c) elementwise on NHWC bf16 views */
int crfr_add_n(const void* a, int a_ld, const void* b, int b_ld, const void* c3, int c_ld, void* out, int out_ld,
               long long pixels, int c, void* stream);

/* ---------------------------------------------------------------- losses ---------------------------------- */
/* ref: MSELossFunc loss/loss.py:7-15.  x,t fp32 NCHW [n][c][hw]; loss[0] = mean((x-t)^2)*97;
 * dx (NHWC bf16, stride dx_ld, may be NULL) = gscale * dloss/dx. */
int crfr_loss_mse97(const float* x, const float* t, int n, int c, int hw, float gscale, float* loss, void* dx,
                    int dx_ld, void* ws, size_t ws_bytes, void* stream);
/* ref: MSELoss_Landmark loss/loss.py:17-32.  x fp32 NCHW [n][c][hw], t fp32 [n][hw]. dx written at channel
 * offset dx_coff of an NHWC bf16 buffer. */
int crfr_loss_landmark(const float* x, const float* t, int n, int c, int hw, float gscale, float* loss, void* dx,
                       int dx_ld, int dx_coff, void* ws, size_t ws_bytes, void* stream);
/* ref: CrossEntropyLoss2d loss/loss.py:34-62.  logits fp32 NCHW [n][c][hw], target int64 [n][hw]. */
int crfr_loss_ce2d(const float* logits, const long long* target, int n, int c, int hw, float gscale, float* loss,
                   void* dx, int dx_ld, int dx_coff, void* ws, size_t ws_bytes, void* stream);
/* ref: nn.MSELoss over (t - s) vs a, distill_main.py:63,68-70.  All NHWC bf16 or all fp32 flat (is_f32).
 * loss = mean(((t - s) - a)^2) with s NULL meaning 0.  Gradients (scaled by gscale) are optional. */
int crfr_loss_kd(const void* t, const void* s, const void* a, long long numel, int is_f32, float gscale,
                 float* loss, void* dt, void* ds, void* da, void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------- optimiser ------------------------------- */
/* ref: torch.optim.RMSprop(lr, alpha=.99, eps=1e-8, weight_decay=1e-5) FSR_main.py:185, distill_main.py:222-225.
 * g is multiplied by gscale first (1/world_size after the all-reduce). */
int crfr_rmsprop_step(float* p, const float* g, float* sq, long long n, float lr, float alpha, float eps,
                      float weight_decay, float gscale, void* stream);

/* ---------------------------------------------------------------- bicubic --------------------------------- */
/* ref: PIL Image.resize(BICUBIC) at bicubic_interpolation.py:188, SUPER_RESOLUTION/FHN_loader.py:66.
 * src u8 NHWC [n][ih][iw][c] -> dst u8 NHWC [n][oh][ow][c] (bit-exact with Pillow's 8-bit path) and/or
 * dst_f32 NCHW normalised (x/255-0.5)/0.5 (helen_loader.py:53-58).  Coefficient tables are built on the host
 * (double precision, exactly as Pillow) by crfr_bicubic_tables into host_tab, then copied by the caller. */
int crfr_bicubic_table_size(int in_size, int out_size);                   /* number of int32 entries */
int crfr_bicubic_tables(int in_size, int out_size, int32_t* host_tab);    /* [out][2+ksize]: xmin, count, kk[] */
int crfr_bicubic_u8(const uint8_t* src, int n, int ih, int iw, int c, const int32_t* tab_h, const int32_t* tab_w,
                    int oh, int ow, uint8_t* tmp, uint8_t* dst, float* dst_f32, void* stream);

/* ref: the augmentation of HelenLoader.__getitem__ helen_loader.py:75-104 (Pillow, third party): Image.rotate(angle) -
 * NEAREST, no expand, zero fill: Pillow's 16.16 fixed-point affine gather - followed by one
 * ImageEnhance.Contrast(img).enhance(f) per factor (blend with the rounded mean luma in float32, truncated for
 * 0 <= f <= 1, clipped otherwise).  Bit-exact with Pillow 12.2.0.
 * crfr_rotate_coeffs: the six fixed-point coefficients of one image (HOST, double precision, exactly as Pillow).
 * crfr_augment_u8: src/dst u8 NHWC [n][h][w][c] (c = 1 or 3, src != dst); coef int32 [n][6] and factors fp32 [n][nfac] on
 * the device; nfac = 0 rotates only (the parsing map, :103-104). */
int crfr_rotate_coeffs(int h, int w, double angle_deg, int32_t* host_coef6);
int crfr_augment_u8(const uint8_t* src, int n, int h, int w, int c, const int32_t* coef, const float* factors, int nfac,
                    uint8_t* dst, void* stream);
/* ref: the random crop of SUPER_RESOLUTION/FHN_loader.py:61-63,92 (Image.crop((nw, nh, nw + 112, nh + 112))):
 * dst[n][y][x] = src[n][off[n][0] + y][off[n][1] + x]; offsets int32 [n][2] = (nh, nw) on the device; the caller keeps the
 * windows inside the image (random.randint(0, 128 - 112)). */
int crfr_crop_u8(const uint8_t* src, int n, int h, int w, int c, const int32_t* offsets_yx, int oh, int ow, uint8_t* dst,
                 void* stream);

/* ref: HelenLoader.generate_hm / gaussian_k helen_loader.py:118-143 - the landmark heat-map target of the prior loss:
 * hm[n][y][x] = sum_j exp(-((x - lx_j)^2 + (y - ly_j)^2) / (2 sigma^2)), Gaussians in fp64, running sum rounded to fp32
 * after every landmark (as numpy's in-place += on a float32 array).  landmarks fp32 [n][k][2] = (x, y) in heat-map
 * pixels (helen_loader.py:104-113: already rotated / scaled by the loader). */
int crfr_landmark_heatmap(const float* landmarks, int n, int k, float sigma, int h, int w, float* hm, void* stream);

/* ---------------------------------------------------------------- matcher --------------------------------- */
/* ref: l2_norm DISTILLATION/model/model_irse.py:16-20 ; accuracy()/topk utils/eval.py:6-19 ; threshold decision
 * utils/utils.py:14-24.  rows of x (fp32 [rows][dim]) -> unit-norm bf16. */
int crfr_l2norm_bf16(const float* x, void* out, long long rows, int dim, void* stream);
/* probes bf16 [p][dim], gallery bf16 [g][dim] (both unit norm).  Writes top-k (k<=8) scores fp32 [p][k] and global
 * indices int32 [p][k] (+ index_base), sorted descending, ties -> lowest index. */
int crfr_cosine_topk(int engine, const void* probes, const void* gallery, int p, long long g, int dim, int k,
                     int index_base, float* top_val, int* top_idx, void* ws, size_t ws_bytes, void* stream);
size_t crfr_cosine_topk_workspace_bytes(int p, long long g, int dim, int k);
/* merges `parts` per-shard top-k lists ([parts][p][k]) into one (gallery-sharded multi-GPU path) */
int crfr_topk_merge(const float* vals, const int* idx, int parts, int p, int k, float* out_val, int* out_idx,
                    void* stream);
/* ref: output.topk(maxk, 1, True, True) on a materialised score matrix (utils/eval.py:11): scores fp32 [p][g],
 * k <= 8, sorted descending, ties -> lowest index. */
int crfr_topk_rows(const float* scores, int p, long long g, int k, float* out_val, int* out_idx, void* stream);
/* ref: calculate_accuracy utils/utils.py:14-24: counts[4] = tp, fp, tn, fn of (dist < thr) vs issame (u8) */
int crfr_verify_counts(const float* dist, const uint8_t* issame, long long n, float thr, unsigned long long* counts,
                       void* stream);
/* ref: the threshold sweeps of calculate_roc utils/utils.py:70-82: counts[t][4] = tp, fp, tn, fn of (dist < thresholds[t])
 * over the pairs listed in subset[n] (indices into dist / issame; NULL = the first n pairs).  fp32 thresholds. */
int crfr_verify_sweep(const float* dist, const uint8_t* issame, const int* subset, int n, const float* thresholds,
                      int nthr, unsigned int* counts, void* stream);
/* verification: same[i] = (sum((e1-e2)^2) < thr) for fp32 pairs; also writes dist */
int crfr_pair_verify(const float* e1, const float* e2, long long pairs, int dim, float thr, float* dist,
                     uint8_t* same, void* stream);

/* ---------------------------------------------------------------- reflection padding, tanh ----------------- */
/* ref: nn.ReflectionPad2d / nn.Tanh of the SUPER_RESOLUTION FSRNet variant (SUPER_RESOLUTION/model/FSRnet.py:251-416).
 * x: NHWC bf16 [n][h][w][ld], out: [n][h+2p][w+2p][ld]; c a multiple of 8, or <= 4 with ld 4.  bwd folds dout back. */
int crfr_reflect_pad_fwd(const void* x, int x_ld, void* out, int out_ld, int n, int h, int w, int c, int pad, void* stream);
int crfr_reflect_pad_bwd(const void* dout, int dout_ld, void* dx, int dx_ld, int n, int h, int w, int c, int pad,
                         void* stream);
int crfr_tanh_fwd(const float* x, float* y, long long numel, void* stream);
int crfr_tanh_bwd(const float* y, const float* dy, float* dx, long long numel, void* stream);

/* ---------------------------------------------------------------- fully connected layer ------------------- */
/* ref: nn.Linear on `x.view(B, -1)` of an NCHW map (model/FSRnet.py:469,484-486 Discriminator.fc; model/resnet.py:170,
 * 221-222).  x: NHWC bf16 [B][hw][c]; w: fp32 [out][c * hw] in the reference's NCHW-flatten order; y / dy: bf16 [B][out].
 * in_features = c * hw must be a multiple of 64, out 64 or a multiple of 128.  dw / dbias are accumulated (+=). */
size_t crfr_linear_workspace_bytes(int batch, int hw, int c, int out);
int crfr_linear_fwd(const void* x, int batch, int hw, int c, const float* w, const float* bias, int out, void* y,
                    void* ws, size_t ws_bytes, void* stream);
int crfr_linear_bwd(const void* x, const void* dy, int batch, int hw, int c, const float* w, int out, void* dx,
                    float* dw, float* dbias, void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------- FSRNet network program ------------------ */
#define CRFR_FSRNET_NPARAMS 202
typedef struct crfr_fsrnet_io {
  int batch, size;          /* size = H = W of the (already upsampled) network input, multiple of 16 */
  const float* x;           /* [B,3,H,W] fp32 NCHW */
  float* coarse;            /* [B,3,H,W]      (out) */
  float* out;               /* [B,3,H,W]      (out) */
  float* landmark;          /* [B,97,H/4,W/4] (out) */
  float* parsing;           /* [B,11,H/4,W/4] (out) */
  /* training targets (crfr_fsrnet_train_step only) */
  const float* hr;          /* [B,3,H,W] */
  const float* heatmap;     /* [B,H/4,W/4] */
  const long long* labels;  /* [B,1,H/4,W/4] int64 */
  float loss_div;           /* the 2*train_batch of FSR_main.py:234 (global batch under data parallelism) */
  float w_pix;              /* 5.0 at FSR_main.py:233 (7.0 at :319) */
  /* optional cudaEvent_t handles recorded on `stream` during backward when a gradient bucket is complete:
   * [0] decoder (params 167..201), [1] prior + encoder (33..166), [2] coarse (0..32).  The data-parallel host
   * loop starts each bucket's all-reduce on a side stream behind its event (overlap with the rest of backward). */
  void* bucket_events[3];
} crfr_fsrnet_io;

/* One recorded op of the network program (test / debugging aid: where the saved forward tensors live in the workspace).
 * kind: 0 conv, 1 InstanceNorm(+PReLU)(+residual), 2 max-pool, 3 nearest-up + add, 4 concat (view), 5 heads,
 * 6 3-channel image conv.  Offsets are bytes from the workspace base, -1 when absent. */
typedef struct crfr_tape_entry {
  int kind;
  int n, h, w, c, ld;      /* output tensor: NHWC bf16 with a pixel stride of ld elements */
  long long out_off;
  long long in_off;        /* first input */
  long long stats_off;     /* kind 1: fp32 (mean, rstd) [n][c][2] */
  int w_idx, has_res;
} crfr_tape_entry;
/* fills up to max_entries entries (entries may be NULL) and returns the number of recorded ops, < 0 on bad arguments */
int crfr_fsrnet_tape(int batch, int size, int training, crfr_tape_entry* entries, int max_entries);
/* Where crfr_fsrnet_id_train_step leaves its tensors (test aid, from the dry run of the step itself).  Offsets are bytes
 * from the base of the step's workspace; the entries, in order:
 *   1. those of crfr_fsrnet_tape(batch, size, 1): the FSRNet arena starts at 0;
 *   2. kind 19: the output-image gradient d_out4, bf16 NHWC [batch][size][size], c = 3, ld 4;
 *   3. crfr_irnet_tape of the crop(hr) program, shifted by the base of its arena;
 *   4. the same for the crop(sr) program;
 *   5. kind 17, one per selected term k in increasing k: the bf16 seed slot of the feature gradient (w_idx = k, in_off =
 *      out_off of the crop(sr) tensor it is the gradient of);
 *   6. the crop(sr) backward's gradient tape (kinds 11-16, as crfr_irnet_grad_tape);
 *   7. kind 18: dx4, the bf16 NHWC [batch][112][112] (c = 3, ld 4) input gradient the window kernel adds to d_out4.
 * A kind-12 entry shares its buffer with the kind-15 entry of the next unit, the head's kind 11 or a kind-17 seed when
 * that is the unit output's only gradient.  Fills up to max_entries entries (entries may be NULL) and returns the count;
 * -1 where crfr_fsrnet_id_workspace_bytes is 0 or terms is outside 1..31. */
int crfr_fsrnet_id_tape(int teacher_layers, int teacher_se, int batch, int size, int terms, crfr_tape_entry* entries,
                        int max_entries);

/* ref: OverallNetwork.forward model/FSRnet.py:497-508 with the runnable wiring of :538-541.
 * params: 202 fp32 device pointers in state_dict order.  engine selects the conv engine for eligible layers. */
size_t crfr_fsrnet_workspace_bytes(int batch, int size, int training);
int crfr_fsrnet_forward(int engine, const float* const* host_params, const crfr_fsrnet_io* io, int training,
                        void* ws, size_t ws_bytes, void* stream);
/* grads w.r.t. the four outputs (fp32 NCHW, any may be NULL) -> accumulates into host_grads[202] (NULL entries skipped) */
int crfr_fsrnet_backward(int engine, const float* const* host_params, float* const* host_grads,
                         const crfr_fsrnet_io* io, const float* d_coarse, const float* d_out,
                         const float* d_landmark, const float* d_parsing, void* ws, size_t ws_bytes, void* stream);
/* The four sub-networks on their own: Course_SR_Network / Fine_SR_Encoder / Prior_Estimation_Network / Fine_SR_Decoder
 * .forward of the reference (model/FSRnet.py:328-340, 359-379, 408-426, 448-459), each with its own backward.
 * params / grads are the same 202-entry tables (only the section's entries are touched). */
enum { CRFR_FSRNET_COARSE = 0, CRFR_FSRNET_ENCODER = 1, CRFR_FSRNET_PRIOR = 2, CRFR_FSRNET_DECODER = 3 };
typedef struct crfr_fsrnet_section_io {
  int section, batch;
  int size;                 /* full-resolution H = W; the encoder / prior outputs and the decoder input live at size / 4 */
  const float* x;           /* coarse, encoder, prior: [B,3,size,size]; decoder: [B,192,size/4,size/4]   (fp32 NCHW) */
  float* out[3];            /* coarse: {feat [B,64,S,S], coarse [B,3,S,S]}; encoder: {feat [B,64,S/4,S/4]};
                               prior: {feat [B,128,S/4,S/4], landmark [B,97,..], parsing [B,11,..]}; decoder: {sr [B,3,S,S]} */
} crfr_fsrnet_section_io;
size_t crfr_fsrnet_section_workspace_bytes(int section, int batch, int size, int training);
int crfr_fsrnet_section_forward(int engine, const float* const* host_params, const crfr_fsrnet_section_io* io,
                                int training, void* ws, size_t ws_bytes, void* stream);
/* d_out: gradients w.r.t. out[0..2] (fp32 NCHW, NULL entries = no gradient); accumulates into host_grads; dx (optional):
 * gradient w.r.t. the section input, same shape as x */
int crfr_fsrnet_section_backward(int engine, const float* const* host_params, float* const* host_grads,
                                 const crfr_fsrnet_section_io* io, const float* const* d_out, float* dx, void* ws,
                                 size_t ws_bytes, void* stream);

/* forward + losses (FSR_main.py:233-234) + backward in one call.  losses: device fp32[5] =
 * (total, L_sr, L_coarse, L_landmark, L_ce). */
int crfr_fsrnet_train_step(int engine, const float* const* host_params, float* const* host_grads,
                           const crfr_fsrnet_io* io, float* losses, void* ws, size_t ws_bytes, void* stream);

/* ref: the identity / perceptual loss through a frozen face-recognition network, SUPER_RESOLUTION/train_FHN.py:255-265.
 * crfr_fsrnet_train_step plus an identity term on the 112 x 112 centre of the super-resolved output (size 128 only):
 *   L = L_FSR + w_id * sum_{k in terms} MSE(f(sr)[k], f(hr)[k]),  f(t) = Backbone.forward_features(t[:, :, 8:120, 8:120])
 * with f an IR / IR-SE teacher (crfr_irnet_*, eval mode, frozen: no parameter gradient, buffers unchanged).  Each MSE is
 * the mean over the chunk; id_scale = chunk / global batch makes the summed chunk gradients, SUM-reduced across ranks, the
 * gradient of the global-batch mean (as loss_div does for L_FSR).  losses: device fp32[6] = (total, L_sr, L_coarse,
 * L_landmark, L_ce, w_id * sum_k MSE_k), total = the L_FSR share + id_scale * losses[5].  io as for crfr_fsrnet_train_step;
 * the same three bucket events are recorded.  No host synchronisation or allocation (graph-capturable). */
typedef struct crfr_fsrnet_id_io {
  int teacher_layers, teacher_se;       /* the IR variant: 50 / 100 / 152 layers, se 1 = IR-SE */
  const float* const* teacher_params;   /* device pointers, named_parameters() order (crfr_irnet_sizes) */
  void* const* teacher_buffers;         /* 3 per BatchNorm, named_buffers() order */
  float w_id;                           /* weight of the identity term (1.0) */
  int terms;                            /* bit k selects output k of (embedding, x1, x2, x3, x4); 31 = all five */
  float id_scale;                       /* this chunk's share of the global batch: chunk / global batch */
} crfr_fsrnet_id_io;
/* the FSRNet training arena, the teacher's forward arena for hr and its gradient arena for sr; 0 when unsupported */
size_t crfr_fsrnet_id_workspace_bytes(int teacher_layers, int teacher_se, int batch, int size);
int crfr_fsrnet_id_train_step(int engine, const float* const* host_params, float* const* host_grads,
                              const crfr_fsrnet_io* io, const crfr_fsrnet_id_io* id, float* losses, void* ws,
                              size_t ws_bytes, void* stream);

/* ----------------------------------------------------------- SUPER_RESOLUTION FSRNet variant program ---- */
/* ref: SUPER_RESOLUTION/model/FSRnet.py:251-416 (Coarse_SR_Network, Fine_SR_Encoder, Prior_Estimation_Network,
 * Fine_SR_Decoder) and the SRNetwork wiring of its unconstructible OverallNetwork (:449): coarse image -> encoder and
 * prior network -> cat(prior, encoder) -> decoder.  One call per forward and per backward over a caller-provided arena;
 * every layer keeps the routing of crfr_conv_fwd / _dgrad / _wgrad, the two 1x1 prior heads (fc 13 channels with bias,
 * fc_landmark 68 without) run as one tensor-core GEMM 64 -> 128.
 * params / grads: device pointers in the section's state_dict order - CRFR_SRNET_NPARAMS for SRNetwork
 * (_coarse_sr_network, _prior_estimation_network, _fine_sr_encoder, _fine_sr_decoder), 52 / 51 / 954 / 51 for the
 * coarse network / encoder / prior network / decoder alone.
 * Shapes (h and w separately; what the composed modules compute without a size mismatch):
 *   coarse, encoder, decoder: h, w >= 5 (the second stride-2 stage's reflection pad needs 2 rows); their outputs are
 *     4 * ceil(h / 4) x 4 * ceil(w / 4) (two stride-2 stages, two exact 2x transposed stages);
 *   prior, SRNetwork: h, w multiples of 16 (the hourglass pools four times and adds the up-sampled map back);
 *   batch * (4 * ceil(h / 4) + 6) * (4 * ceil(w / 4) + 6) * 128 < 2^31 (element indices of the widest padded map).
 * Anything else is CRFR_EINVAL before any launch; the size query returns 0 and the tape -1.  The tables must come from
 * modules built with the reference's default constructor arguments (the program's channel counts are fixed). */
#define CRFR_SRNET_NPARAMS 1108
enum { CRFR_SRNET_COARSE = 0, CRFR_SRNET_ENCODER = 1, CRFR_SRNET_PRIOR = 2, CRFR_SRNET_DECODER = 3,
       CRFR_SRNET_NETWORK = 4 };
typedef struct crfr_srnet_io {
  int section, batch, h, w;
  const float* x;   /* fp32 NCHW [B,3,h,w]; decoder: [B,128,h,w] */
  float* out[4];    /* fp32 NCHW, (H, W) = the output size above:
                       SRNetwork {coarse [B,3,h,w], out [B,3,h,w], landmark [B,68,h,w], parsing [B,13,h,w]};
                       coarse {[B,3,H,W]}; encoder {[B,64,H,W]}; prior {feat [B,64,h,w], landmark, parsing};
                       decoder {[B,3,H,W]} */
} crfr_srnet_io;
/* ref: SUPER_RESOLUTION/model/FSRnet.py:251-416.  The arena of one call; training != 0 also holds what the backward
 * needs (a backward follows a training forward over the same arena).  0 for an unsupported shape. */
size_t crfr_srnet_workspace_bytes(int section, int batch, int h, int w, int training);
/* ref: SUPER_RESOLUTION/model/FSRnet.py:251-416.  Layout of the stored forward tensors (a dry run, as crfr_fsrnet_tape):
 * one entry per op in program order, offsets from the workspace base.  Kinds: 0 convolution (w_idx: its weight; the
 * input is the stored padded map), 1 InstanceNorm (+ affine) (+ ReLU / PReLU) (+ residual), 2 max-pool, 3 nearest-up + add
 * (stats_off: the low-resolution input), 4 concat view (out: the decoder's 128-channel input, in_off / stats_off: its prior
 * / encoder halves), 5 the combined prior heads (w_idx: fc.weight; in_off: the features; out_off -1, the outputs go to
 * the caller), 20 reflection pad (w_idx: the padding), 21 Bottleneck add (in_off: conv3's output, stats_off: the block
 * input), 22 Tanh image head (in_off: the 3-channel bf16 NHWC4 convolution output; out_off: the bf16 NHWC4 copy of the
 * coarse image inside SRNetwork, else -1). */
int crfr_srnet_tape(int section, int batch, int h, int w, int training, crfr_tape_entry* entries, int max_entries);
/* ref: SUPER_RESOLUTION/model/FSRnet.py:251-416.  Where crfr_srnet_backward leaves its bf16 gradients in the workspace (a
 * dry run of that call, in backward order; offsets from the workspace base).  grad_mask: bit i set = d_out[i] given (at
 * least one, only the section's outputs); input_grad: dx requested.  Kind 30: a gradient the op at forward-tape index
 * w_idx consumes for its output (one entry per summed slot; n, h, w, c the tensor's, ld the buffer's; in_off the
 * crfr_srnet_tape offset of the tensor, -1 for the prior heads' gathered [pixel][128] output gradient).  Kind 31: a
 * gradient that op produces for an input (has_res: 0 first input, 1 second - residual, Bottleneck input, low-resolution
 * map, encoder half; in_off: that input's offset).  A tensor's producer consumes the sum of the kind-31 gradients of its
 * consumers.  Gradients that only pass through (add, concat, up-add's first input) share the consumed buffer.  Returns the
 * count, -1 on bad arguments. */
int crfr_srnet_grad_tape(int section, int batch, int h, int w, int grad_mask, int input_grad, crfr_tape_entry* entries,
                         int max_entries);
/* ref: SUPER_RESOLUTION/model/FSRnet.py:251-416, forward of the section io->section.  ws_bytes below
 * crfr_srnet_workspace_bytes is CRFR_EWORKSPACE with nothing written. */
int crfr_srnet_forward(int engine, const float* const* host_params, const crfr_srnet_io* io, int training, void* ws,
                       size_t ws_bytes, void* stream);
/* ref: autograd through SUPER_RESOLUTION/model/FSRnet.py:251-416.  ws holds a training forward of the same section and
 * shape (x and out are not read).  d_out[i]: fp32 gradient of io->out[i], NULL = none.  Parameter gradients are
 * accumulated into host_grads (NULL entries skipped); dx (optional, the shape of x) is overwritten with the input
 * gradient.  The saved forward is not modified: repeated calls give the same bits. */
int crfr_srnet_backward(int engine, const float* const* host_params, float* const* host_grads, const crfr_srnet_io* io,
                        const float* const* d_out, float* dx, void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------- ResNet_34 embedding network program ------ */
#define CRFR_RESNET34_NPARAMS 114 /* named_parameters() order of model/resnet.py:ResNet_34 */
#define CRFR_RESNET34_NBN 38      /* BatchNorm layers in module order */
typedef struct crfr_resnet_io {
  int batch, size;       /* size = 112 (model/resnet.py:156,168: Linear(25088, 512)) */
  const float* x;        /* [B,3,S,S] fp32 NCHW */
  float* emb;            /* [B,512]                                   (out) */
  float* feat[4];        /* x1..x4: [B,64,56,56] [B,128,28,28] [B,256,14,14] [B,512,7,7]; NULL entries are skipped */
  int training;          /* 1: batch statistics + running-statistics update; 0: running statistics (eval) */
  float momentum, eps;   /* nn.BatchNorm defaults 0.1, 1e-5 */
} crfr_resnet_io;

/* ref: ResNet.forward model/resnet.py:207-225 -> (x, x1, x2, x3, x4).
 * params: 114 fp32 device pointers in named_parameters() order.  buffers: 3 * 38 device pointers in named_buffers()
 * order (running_mean fp32, running_var fp32, num_batches_tracked int64 per BatchNorm; NULL table in training mode
 * skips the buffer update). */
size_t crfr_resnet34_workspace_bytes(int batch, int size, int training);
/* Layout of the stored forward tensors of the ResNet_34 program (dry run), as crfr_fsrnet_tape: one entry per op in program
 * order - kind 0 convolution, 1 BatchNorm (+ residual) (+ ReLU), 7 linear head.  For teacher-forced parity tests. */
int crfr_resnet34_tape(int batch, int size, int training, crfr_tape_entry* entries, int max_entries);
int crfr_resnet34_forward(int engine, const float* const* host_params, void* const* host_buffers,
                          const crfr_resnet_io* io, void* ws, size_t ws_bytes, void* stream);
/* grads w.r.t. the embedding and the four stage features (fp32 NCHW, any may be NULL) -> accumulates into
 * host_grads[114] (NULL entries skipped).  ws must be the workspace of the matching training-mode forward. */
int crfr_resnet34_backward(int engine, const float* const* host_params, float* const* host_grads,
                           const crfr_resnet_io* io, const float* d_emb, const float* const* d_feat, void* ws,
                           size_t ws_bytes, void* stream);

/* ref: the residual knowledge-distillation step distill_main.py:59-74 evaluated on ONE forward (the committed order -
 * optimiser step between two backward passes over one graph - raises on torch >= 1.5, SURVEY.md 0.3 / 8c-iii):
 *   L_s = MSE(s_emb, t_emb.detach());  L_a = sum_{k=1..4} MSE(t_k - s_k, a_k) + MSE(t_emb - s_emb, a_emb)
 * teacher (ResNet_34, eval), student and assistant (ResNet_34, train).  Accumulates dL_s/dtheta_S
 * (+ dL_a/dtheta_S when assistant_grad_to_student, as the reference graph does) into student_grads and dL_a/dtheta_A
 * into assistant_grads; losses: device fp32[2] = (L_s, L_a).  Parameter / buffer tables as for crfr_resnet34_forward. */
typedef struct crfr_kd_io {
  int batch, size;               /* size = 112 */
  const float* x;                /* [B,3,112,112] fp32 NCHW, the same batch for all three networks (distill_main.py:60-62) */
  float momentum, eps;           /* BatchNorm: 0.1, 1e-5 */
  int assistant_grad_to_student; /* 1: keep the reference's un-detached t_k - s_k in L_a */
  const float* x_lr;             /* optional: the LR batch for the student and the assistant ("HR teacher / LR student");
                                    NULL: all three networks see x, as distill_main.py:59-61 feeds them */
  int teacher_ir50;              /* 1: teacher_params / teacher_buffers are the tables of an IR teacher (IR_50: 187 / 3 x 54; the
                                    variant is teacher_ir_layers / teacher_ir_se below), its four stage outputs are the t_k
                                    (DISTILLATION/model/model_irse.py: 64@56^2, 128@28^2, 256@14^2, 512@7^2) */
  void* events[2];               /* optional cudaEvent_t handles recorded on `stream`: [0] student gradients final (the data-
                                    parallel loop starts their all-reduce behind it, overlapping the assistant's backward),
                                    [1] assistant gradients final */
  int teacher_ir_layers;         /* read only when teacher_ir50 != 0: 50 (or 0), 100 or 152 */
  int teacher_ir_se;             /* read only when teacher_ir50 != 0: 1 = the IR_SE variant (tables of crfr_irnet_sizes) */
} crfr_kd_io;
size_t crfr_kd_workspace_bytes(int batch, int size);
size_t crfr_kd_workspace_bytes_ex(int batch, int size, int teacher_ir50);
/* the workspace of crfr_kd_train_step with the IR teacher (teacher_ir_layers, teacher_ir_se); 0 for an unsupported variant */
size_t crfr_kd_workspace_bytes_ir(int batch, int size, int teacher_ir_layers, int teacher_ir_se);
int crfr_kd_train_step(int engine, const float* const* teacher_params, void* const* teacher_buffers,
                       const float* const* student_params, void* const* student_buffers, float* const* student_grads,
                       const float* const* assistant_params, void* const* assistant_buffers,
                       float* const* assistant_grads, const crfr_kd_io* io, float* losses, void* ws, size_t ws_bytes,
                       void* stream);

/* ---------------------------------------------------------------- IR_50 teacher ----------------------------- */
#define CRFR_IR50_NPARAMS 187 /* named_parameters() order of DISTILLATION/model/model_irse.py:IR_50 */
#define CRFR_IR50_NBN 54      /* BatchNorm layers in module order (input_layer, output_layer, body) */
/* ref: Backbone.forward model_irse.py:167-172 in eval mode (the frozen teacher of distill_main.py:43,201): returns the
 * 512-d embedding in io->emb and, for non-NULL io->feat[k], the output of body stage k (the "extracted layers" use of
 * DISTILLATION/model/utils.py:36-52 and the t_k of the KD loss); io->training must be 0.  buffers: 3 * 54 pointers as above. */
size_t crfr_ir50_workspace_bytes(int batch, int size);
int crfr_ir50_forward(int engine, const float* const* host_params, void* const* host_buffers,
                      const crfr_resnet_io* io, void* ws, size_t ws_bytes, void* stream);
/* ref: autograd through Backbone.forward model_irse.py:167-172 in eval mode, with respect to the input image only (an
 * identity / perceptual loss on the features of a super-resolved face, SUPER_RESOLUTION/train_FHN.py:255-265).
 * crfr_ir50_grad_workspace_bytes: the forward arena (the same layout as crfr_ir50_workspace_bytes) plus the backward
 * buffers.  crfr_ir50_backward: ws holds a crfr_ir50_forward of the same io over a workspace of at least that size;
 * d_emb [B,512] and d_feat[k] (the shapes of io->feat[k]) are fp32 upstream gradients, any of them NULL; dx [B,3,112,112]
 * fp32 is overwritten.  No parameter gradient is computed.  The saved forward is not modified: repeated calls give the
 * same bits. */
size_t crfr_ir50_grad_workspace_bytes(int batch, int size);
/* Layout of the stored forward tensors of crfr_ir50_forward (dry run), as crfr_resnet34_tape: kind 0 convolution,
 * 1 BatchNorm (+ residual) (+ PReLU at the stem), 7 linear head, 8 PReLU pass, 9 stride-2 subsampling (MaxPool2d(1, 2)).
 * For teacher-forced parity tests. */
int crfr_ir50_tape(int batch, int size, crfr_tape_entry* entries, int max_entries);
int crfr_ir50_backward(int engine, const float* const* host_params, void* const* host_buffers,
                       const crfr_resnet_io* io, const float* d_emb, const float* const* d_feat, float* dx, void* ws,
                       size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------- IR / IR-SE teachers ----------------------- */
/* ref: IR_50 / IR_101 / IR_152 / IR_SE_50 / IR_SE_101 / IR_SE_152 and Backbone(input_size, num_layers, mode),
 * DISTILLATION/model/model_irse.py:129-172 (get_blocks :101-126; mode "ir_se": bottleneck_IR_SE, whose res_layer ends in
 * SEModule(depth, 16) = x * sigmoid(fc2(relu(fc1(mean_hw(x)))))), at 112 x 112 in eval mode.  The variant is
 * (num_layers in {50, 100, 152}, se in {0, 1}); crfr_irnet_*(50, 0, ...) is crfr_ir50_* (same arena, launches and bits).
 * Any other variant is rejected: the size queries return 0 (the tape -1), the calls an error code with a message.
 * crfr_irnet_sizes: the number of named_parameters() and of BatchNorm layers (buffers: 3 per BatchNorm), host pointers,
 * either may be NULL.  The other calls behave as their crfr_ir50_* counterparts; the tape adds kind 10, an SE unit's
 * output (res_layer.4 BatchNorm x excitation + shortcut), whose stats_off is the excitation e [n][c] fp32. */
int crfr_irnet_sizes(int num_layers, int se, int* n_params, int* n_bn);
size_t crfr_irnet_workspace_bytes(int num_layers, int se, int batch, int size);
int crfr_irnet_forward(int engine, int num_layers, int se, const float* const* host_params, void* const* host_buffers,
                       const crfr_resnet_io* io, void* ws, size_t ws_bytes, void* stream);
size_t crfr_irnet_grad_workspace_bytes(int num_layers, int se, int batch, int size);
int crfr_irnet_tape(int num_layers, int se, int batch, int size, crfr_tape_entry* entries, int max_entries);
/* Where crfr_irnet_backward leaves its stored bf16 gradients in the workspace (a dry run of that call), in backward order.
 * seed_mask: the upstream gradients given (1 = d_emb, 2 / 4 / 8 / 16 = d_feat[0..3], at least one); the layout depends
 * on it.  Kinds: 11 the head's input gradient, then per unit with a gradient 12 its summed output gradient g, 13 (SE) dr
 * at the SE input BN_4(y) with stats_off the fp32 shift [n][c] = dpool / hw, 14 the gradient at res_layer.1's output,
 * 15 its input gradient; last 16 the stem's gradient at input_layer.0's output.  in_off is the out_off of the
 * crfr_irnet_tape entry whose tensor the gradient is of (for kind 13: the res_layer.3 output y); w_idx is the unit (-1
 * for 11 and 16).  A kind-12 entry may share its buffer with the entry that produced it.  -1 on bad arguments. */
int crfr_irnet_grad_tape(int num_layers, int se, int batch, int size, int seed_mask, crfr_tape_entry* entries,
                         int max_entries);
int crfr_irnet_backward(int engine, int num_layers, int se, const float* const* host_params, void* const* host_buffers,
                        const crfr_resnet_io* io, const float* d_emb, const float* const* d_feat, float* dx, void* ws,
                        size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CRFR_H_ */
