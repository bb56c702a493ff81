// C-ABI convolution entry points: shape validation + engine dispatch (tcgen05 implicit GEMM or CUDA-core direct).
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>

#include "common.cuh"
#include "crfr.h"
#include "internal.h"

// ---- error string / counters -------------------------------------------------------------------
static thread_local char g_err[512] = "";
unsigned long long g_crfr_launches = 0;

void crfr_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
extern "C" const char* crfr_last_error(void) { return g_err; }
extern "C" int crfr_version(void) { return 100; }
extern "C" unsigned long long crfr_launch_count(void) { return g_crfr_launches; }

// ---- tuning switches (internal.h) ------------------------------------------------------------------------------
namespace {
struct OptDef { const char* name; const char* env; int dflt; };
const OptDef kOpts[CRFR_OPT_COUNT] = {
    {"rowconv_pair", "CRFR_ROWCONV_PAIR", 1},   {"wgrad_stream", "CRFR_WGRAD_STREAM", 1},
    {"norm_bwd_impl", "CRFR_NORM_BWD", 1},      {"norm_fwd_stream", "CRFR_NORM_FWD_STREAM", 1},
    {"fuse_norm_bwd", "CRFR_FUSE_NORM_BWD", 1}};
std::atomic<int> g_opt[CRFR_OPT_COUNT];
std::atomic<int> g_opt_init{0};
void opts_init() {
  if (g_opt_init.load(std::memory_order_acquire) == 2) return;
  int expect = 0;
  if (g_opt_init.compare_exchange_strong(expect, 1)) {
    for (int i = 0; i < CRFR_OPT_COUNT; ++i) {
      const char* e = getenv(kOpts[i].env);
      int v = kOpts[i].dflt;
      if (e && *e) v = (i == CRFR_OPT_NORM_BWD_STREAM) ? (e[0] == 'r' || e[0] == '0' ? 0 : 1) : atoi(e);
      g_opt[i].store(v, std::memory_order_relaxed);
    }
    g_opt_init.store(2, std::memory_order_release);
  } else {
    while (g_opt_init.load(std::memory_order_acquire) != 2) {}
  }
}
std::atomic<int> g_sms[64];
}  // namespace

int crfr_opt(int id) {
  opts_init();
  return (id >= 0 && id < CRFR_OPT_COUNT) ? g_opt[id].load(std::memory_order_relaxed) : 0;
}

int crfr_sm_count() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  int v = g_sms[dev].load(std::memory_order_relaxed);
  if (!v) {
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
    g_sms[dev].store(v, std::memory_order_relaxed);
  }
  return v;
}

extern "C" int crfr_set_option(const char* name, int value) {
  CRFR_CHECK_ARG(name, "set_option: null name");
  opts_init();
  for (int i = 0; i < CRFR_OPT_COUNT; ++i)
    if (!strcmp(name, kOpts[i].name)) {
      g_opt[i].store(value, std::memory_order_relaxed);
      return CRFR_OK;
    }
  crfr_set_error("set_option: unknown option '%s'", name);
  return CRFR_EINVAL;
}

static int check_desc(const crfr_conv_desc* d, const char* who) {
  CRFR_CHECK_ARG(d, "%s: null descriptor", who);
  CRFR_CHECK_ARG(d->n > 0 && d->h > 0 && d->w > 0 && d->cin > 0 && d->cout > 0 && d->k > 0 && d->stride > 0 &&
                     d->pad >= 0 && d->oh > 0 && d->ow > 0,
                 "%s: non-positive dimension", who);
  CRFR_CHECK_ARG(d->in_ld >= d->cin && d->out_ld >= d->cout, "%s: ld smaller than channel count", who);
  if (!d->transposed) {
    CRFR_CHECK_ARG(d->oh == (d->h + 2 * d->pad - d->k) / d->stride + 1 &&
                       d->ow == (d->w + 2 * d->pad - d->k) / d->stride + 1,
                   "%s: output size %dx%d inconsistent with Conv2d geometry", who, d->oh, d->ow);
  } else {
    int lo_h = (d->h - 1) * d->stride - 2 * d->pad + d->k, lo_w = (d->w - 1) * d->stride - 2 * d->pad + d->k;
    CRFR_CHECK_ARG(d->oh >= lo_h && d->oh < lo_h + d->stride && d->ow >= lo_w && d->ow < lo_w + d->stride,
                   "%s: output size %dx%d inconsistent with ConvTranspose2d geometry", who, d->oh, d->ow);
  }
  return CRFR_OK;
}

extern "C" size_t crfr_conv_workspace_bytes(const crfr_conv_desc* d) {
  if (!d) return 0;
  size_t norm = d->cout >= 8 ? crfr_norm_ws_bytes(d->n, d->oh * d->ow, d->cout) : 0;
  size_t tc = crfr_tc_workspace_bytes(d);
  size_t low = crfr_lowered_ws_bytes(d);
  size_t m = norm > tc ? norm : tc;
  return (m > low ? m : low) + 1024;
}

extern "C" int crfr_conv_engine_supported(int engine, int op, int h, int w, int cin, int cout, int k, int stride,
                                          int pad) {
  if (engine == CRFR_ENGINE_DIRECT) return 1;
  if (crfr_tc_supported(op, h, w, cin, cout, k, stride, pad)) return 1;
  crfr_conv_desc d = {1, h, w, cin, cout, k, stride, pad, (h + 2 * pad - k) / stride + 1, (w + 2 * pad - k) / stride + 1,
                      cin < 8 ? 4 : cin, cout < 8 ? 4 : cout, 0};
  const int r = crfr_lowered_recipe(&d);
  return r != 0 && !(r == 1 && op == 1);
}

extern "C" int crfr_conv_fwd(int engine, const crfr_conv_desc* d, const void* x, const void* w_packed, int cin_pad,
                             const float* bias, void* y, float* y_nchw, float* stats, float eps, void* ws,
                             size_t ws_bytes, void* stream) {
  CRFR_TRY(check_desc(d, "conv_fwd"));
  CRFR_CHECK_ARG(x && w_packed && (y || y_nchw), "conv_fwd: null pointer");
  CRFR_CHECK_ARG(cin_pad >= d->cin && d->in_ld >= cin_pad, "conv_fwd: cin_pad %d vs cin %d / in_ld %d", cin_pad,
                 d->cin, d->in_ld);
  CRFR_CHECK_ARG(!stats || y, "conv_fwd: statistics need the bf16 output");
  cudaStream_t st = (cudaStream_t)stream;
  if (engine != CRFR_ENGINE_DIRECT) {
    const int r = crfr_lowered_recipe(d);
    if (r == 2 || (r != 0 && y && !y_nchw)) {
      int stats_done = 0;
      CRFR_TRY(crfr_lowered_fwd(d, x, w_packed, cin_pad, bias, y, y_nchw, ws, ws_bytes, st, stats, eps, &stats_done));
      if (stats && !stats_done)
        CRFR_TRY(crfr_norm_stats(y, d->n, d->oh * d->ow, d->cout, d->out_ld, eps, stats, ws, ws_bytes, stream));
      return CRFR_OK;
    }
  }
  bool tc = false;
  if (engine != CRFR_ENGINE_DIRECT && !d->transposed && y && !y_nchw && cin_pad == d->cin &&
      crfr_tc_supported(0, d->h, d->w, d->cin, d->cout, d->k, d->stride, d->pad)) {
    tc = true;
  }
  if (engine == CRFR_ENGINE_TCGEN05 && !tc) {
    crfr_set_error("conv_fwd: shape not supported by the tcgen05 engine");
    return CRFR_EUNSUPPORTED;
  }
  if (tc) return crfr_tc_conv(d, 0, x, w_packed, bias, y, stats, eps, ws, ws_bytes, st);
  if (!d->transposed)
    CRFR_TRY(crfr_direct_gather(1, d->n, d->h, d->w, d->oh, d->ow, d->k, d->stride, d->pad, x, d->in_ld, w_packed,
                                d->cout, cin_pad, bias, y, d->out_ld, y_nchw, st));
  else
    CRFR_TRY(crfr_direct_gather(0, d->n, d->oh, d->ow, d->h, d->w, d->k, d->stride, d->pad, x, d->in_ld, w_packed,
                                d->cout, cin_pad, bias, y, d->out_ld, y_nchw, st));
  if (stats) CRFR_TRY(crfr_norm_stats(y, d->n, d->oh * d->ow, d->cout, d->out_ld, eps, stats, ws, ws_bytes, stream));
  return CRFR_OK;
}

int crfr_conv_fwd_bnstats(int engine, const crfr_conv_desc* d, const void* x, const void* w_packed, int cin_pad, void* y,
                          float* bn_stats, float eps, void* ws, size_t ws_bytes, cudaStream_t st) {
  const long long count = (long long)d->n * d->oh * d->ow;
  if (engine != CRFR_ENGINE_DIRECT && !d->transposed && cin_pad == d->cin &&
      crfr_lowered_recipe(d) == 0 && crfr_tc_supported(0, d->h, d->w, d->cin, d->cout, d->k, d->stride, d->pad) &&
      count < (1ll << 31))
    return crfr_tc_conv(d, 0, x, w_packed, nullptr, y, bn_stats, eps, ws, ws_bytes, st, 1);
  CRFR_TRY(crfr_conv_fwd(engine, d, x, w_packed, cin_pad, nullptr, y, nullptr, nullptr, eps, ws, ws_bytes, (void*)st));
  return crfr_norm_stats(y, 1, (int)count, d->cout, d->out_ld, eps, bn_stats, ws, ws_bytes, (void*)st);
}

extern "C" int crfr_conv_dgrad(int engine, const crfr_conv_desc* d, const void* dy, const void* w_packed_t,
                               int cout_pad, void* dx, void* ws, size_t ws_bytes, void* stream) {
  CRFR_TRY(check_desc(d, "conv_dgrad"));
  CRFR_CHECK_ARG(dy && w_packed_t && dx, "conv_dgrad: null pointer");
  CRFR_CHECK_ARG(cout_pad >= d->cout && d->out_ld >= cout_pad, "conv_dgrad: cout_pad %d vs cout %d / out_ld %d",
                 cout_pad, d->cout, d->out_ld);
  cudaStream_t st = (cudaStream_t)stream;
  if (engine != CRFR_ENGINE_DIRECT) {
    const int r = crfr_lowered_recipe(d);
    if (r >= 2) return crfr_lowered_dgrad(d, dy, w_packed_t, cout_pad, dx, ws, ws_bytes, st);
  }
  bool tc = engine != CRFR_ENGINE_DIRECT && !d->transposed && cout_pad == d->cout &&
            crfr_tc_supported(1, d->h, d->w, d->cin, d->cout, d->k, d->stride, d->pad);
  if (engine == CRFR_ENGINE_TCGEN05 && !tc) {
    crfr_set_error("conv_dgrad: shape not supported by the tcgen05 engine");
    return CRFR_EUNSUPPORTED;
  }
  if (tc) return crfr_tc_conv(d, 1, dy, w_packed_t, nullptr, dx, nullptr, 0.f, ws, ws_bytes, st);
  if (!d->transposed)
    return crfr_direct_gather(0, d->n, d->h, d->w, d->oh, d->ow, d->k, d->stride, d->pad, dy, d->out_ld, w_packed_t,
                              d->cin, cout_pad, nullptr, dx, d->in_ld, nullptr, st);
  return crfr_direct_gather(1, d->n, d->oh, d->ow, d->h, d->w, d->k, d->stride, d->pad, dy, d->out_ld, w_packed_t,
                            d->cin, cout_pad, nullptr, dx, d->in_ld, nullptr, st);
}

// ---- dgrad + backward of the normalisation that produced the convolution's input, as one operation ----------------
static bool dgrad_norm_fusable(int engine, const crfr_conv_desc* d, int cout_pad) {
  return engine != CRFR_ENGINE_DIRECT && crfr_opt(CRFR_OPT_FUSE_NORM_BWD) && crfr_opt(CRFR_OPT_ROWCONV_PAIR) &&
         !d->transposed && cout_pad == d->cout && crfr_lowered_recipe(d) < 2 &&
         crfr_rowconv_supported(d->h, d->w, d->cin, d->cout, d->k, d->stride, d->pad) &&
         crfr_rowconv_pair_supported(d->n, d->h);
}

extern "C" size_t crfr_conv_dgrad_norm_bwd_workspace_bytes(const crfr_conv_desc* d) {
  if (!d) return 0;
  const size_t conv = crfr_conv_workspace_bytes(d), norm = crfr_norm_ws_bytes(d->n, d->h * d->w, d->cin);
  size_t fused = 0;
  if (crfr_rowconv_supported(d->h, d->w, d->cin, d->cout, d->k, d->stride, d->pad) && crfr_rowconv_pair_supported(d->n, d->h))
    fused = sizeof(float) * ((size_t)d->n * crfr_rowconv_pair_parts(d->n, d->h) * 3 * d->cin + (size_t)d->n * d->cin * 5) + 256;
  size_t m = conv > norm ? conv : norm;
  return (m > fused ? m : fused) + 1024;
}

extern "C" int crfr_conv_dgrad_norm_bwd(int engine, const crfr_conv_desc* d, const void* dout, const void* w_packed_t,
                                        int cout_pad, const void* dx_b, int dxb_ld, const void* y, int y_ld,
                                        const float* stats, const float* gamma, const float* beta, const float* alpha,
                                        int relu, const void* res, int res_ld, void* dz, int dz_ld, void* dy, int dy_ld,
                                        float* dgamma, float* dbeta, float* dalpha, void* ws, size_t ws_bytes,
                                        void* stream) {
  CRFR_TRY(check_desc(d, "conv_dgrad_norm_bwd"));
  CRFR_CHECK_ARG(dout && w_packed_t && y && stats && dz && dy, "conv_dgrad_norm_bwd: null pointer");
  CRFR_CHECK_ARG(dz_ld >= d->cin && dy_ld >= d->cin && y_ld >= d->cin, "conv_dgrad_norm_bwd: ld smaller than channel count");
  const size_t need = crfr_conv_dgrad_norm_bwd_workspace_bytes(d);
  if (!ws || ws_bytes < need) {
    crfr_set_error("conv_dgrad_norm_bwd: workspace %zu < %zu", ws_bytes, need);
    return CRFR_EWORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int n = d->n, hw = d->h * d->w, c = d->cin;
  if (dgrad_norm_fusable(engine, d, cout_pad)) {
    const int parts = crfr_rowconv_pair_parts(n, d->h, !dx_b && !res);
    float* partial = (float*)ws;
    float* bstats = partial + (size_t)n * parts * 3 * c;
    float* tot = bstats + (size_t)n * c * 2;
    crfr_rowconv_fuse f = {y, y_ld, dx_b, dx_b ? dxb_ld : 8, res, res ? res_ld : 8, stats, gamma, beta, alpha, relu, partial};
    CRFR_TRY(crfr_rowconv_pair(dout, d->out_ld, n, d->h, w_packed_t, 1, nullptr, dz, dz_ld, nullptr, 0.f, nullptr, 0, st, &f));
    const void* views[3] = {dz, y, dy};
    const int lds[3] = {dz_ld, y_ld, dy_ld};
    const int use_stream = crfr_opt(CRFR_OPT_NORM_BWD_STREAM) >= 1 && crfr_norm_stream_supported(c, (long long)n * hw, views, lds, 3);
    return crfr_norm_bwd_finish(partial, parts, dz, dz_ld, 0, y, y_ld, stats, gamma, beta, alpha, relu, dy, dy_ld, dgamma,
                                dbeta, dalpha, n, hw, c, bstats, tot, use_stream, st);
  }
  // unfused: the dgrad output goes through the dz buffer, which the first pass then rewrites in place (element-wise,
  // each element read before it is written by the same thread)
  crfr_conv_desc dd = *d;
  dd.in_ld = dz_ld;
  CRFR_TRY(crfr_conv_dgrad(engine, &dd, dout, w_packed_t, cout_pad, dz, ws, ws_bytes, stream));
  return crfr_norm_act_bwd(dz, dz_ld, dx_b, dx_b ? dxb_ld : 8, y, y_ld, stats, gamma, beta, alpha, relu, res, res ? res_ld : 8,
                           dz, dz_ld, dy, dy_ld, dgamma, dbeta, dalpha, n, hw, c, ws, ws_bytes, stream);
}

extern "C" int crfr_conv_wgrad(int engine, const crfr_conv_desc* d, const void* x, const void* dy, float* dw,
                               float* dbias, void* ws, size_t ws_bytes, void* stream) {
  CRFR_TRY(check_desc(d, "conv_wgrad"));
  CRFR_CHECK_ARG(x && dy && (dw || dbias), "conv_wgrad: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (dw && engine != CRFR_ENGINE_DIRECT && crfr_lowered_recipe(d) != 0) {
    CRFR_TRY(crfr_lowered_wgrad(d, x, dy, dw, ws, ws_bytes, st));
  } else if (dw) {
    bool tc = engine != CRFR_ENGINE_DIRECT && !d->transposed &&
              crfr_tc_supported(2, d->h, d->w, d->cin, d->cout, d->k, d->stride, d->pad);
    if (engine == CRFR_ENGINE_TCGEN05 && !tc) {
      crfr_set_error("conv_wgrad: shape not supported by the tcgen05 engine");
      return CRFR_EUNSUPPORTED;
    }
    if (tc) {
      CRFR_TRY(crfr_tc_wgrad(d, x, dy, dw, ws, ws_bytes, st));
    } else if (!d->transposed) {
      CRFR_TRY(crfr_direct_wgrad(d->n, d->h, d->w, d->oh, d->ow, d->k, d->stride, d->pad, dy, d->out_ld, d->cout, x,
                                 d->in_ld, d->cin, dw, ws, ws_bytes, st));
    } else {
      CRFR_TRY(crfr_direct_wgrad(d->n, d->oh, d->ow, d->h, d->w, d->k, d->stride, d->pad, x, d->in_ld, d->cin, dy,
                                 d->out_ld, d->cout, dw, ws, ws_bytes, st));
    }
  }
  if (dbias) CRFR_TRY(crfr_colsum(dy, d->out_ld, d->cout, (long long)d->n * d->oh * d->ow, dbias, ws, ws_bytes, st));
  return CRFR_OK;
}
