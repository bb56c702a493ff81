// Fully connected layer on a flattened NHWC feature map as tcgen05 GEMMs (nn.Linear after `x.view(B, -1)` of an NCHW
// tensor: model/FSRnet.py:469,484-486 Discriminator.fc, model/resnet.py:170,221-222): the weight [O][c * hw] is in the
// reference's NCHW-flatten order, the activation [B][hw][c] is NHWC bf16, so the packs permute K once per call.
//   forward : y[B][O]  = x[B][K] . Wp[O][K]^T + bias          (crfr_tc_gemm, fp32 accumulate, bf16 out)
//   backward: dx[B][K] = dy[B][O] . Wpt[K][O]^T;  dW[O][K] += dy^T x (crfr_tc_wgrad_raw into an fp32 accumulator);
//             dbias += column sums of dy
#include "common.cuh"
#include "crfr.h"
#include "internal.h"

namespace {

// wp[o][hw*C + c] = wpt[hw*C + c][o] = bf16(w[o][c*HW + hw])
__global__ void fc_pack_kernel(const float* __restrict__ w, bf16* __restrict__ wp, bf16* __restrict__ wpt, int O, int C,
                               int HW) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long K = (long long)C * HW;
  if (i >= (long long)O * K) return;
  const int o = (int)(i / K);
  const long long k = i - (long long)o * K;       // hw*C + c
  const int hw = (int)(k / C), c = (int)(k - (long long)hw * C);
  const bf16 v = __float2bfloat16_rn(w[(long long)o * K + (long long)c * HW + hw]);
  if (wp) wp[i] = v;
  if (wpt) wpt[k * O + o] = v;
}

// dW [o][c*HW + hw] += G[hw*C + c][o]
__global__ void fc_unpack_kernel(const float* __restrict__ G, float* __restrict__ dw, int O, int C, int HW) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long K = (long long)C * HW;
  if (i >= (long long)O * K) return;
  const int o = (int)(i / K);
  const long long r = i - (long long)o * K;       // c*HW + hw
  const int c = (int)(r / HW), hw = (int)(r - (long long)c * HW);
  dw[i] += G[((long long)hw * C + c) * O + o];
}

int check_shape(const char* who, int batch, int hw, int c, int out) {
  CRFR_CHECK_ARG(batch > 0 && hw > 0 && c > 0 && out > 0, "%s: non-positive dimension", who);
  CRFR_CHECK_ARG(((long long)hw * c) % 64 == 0 && c % 8 == 0, "%s: in_features %lld must be a multiple of 64 (c of 8)", who,
                 (long long)hw * c);
  CRFR_CHECK_ARG(out % 128 == 0 || out == 64, "%s: out_features %d must be 64 or a multiple of 128", who, out);
  return CRFR_OK;
}

}  // namespace

extern "C" size_t crfr_linear_workspace_bytes(int batch, int hw, int c, int out) {
  if (batch <= 0 || hw <= 0 || c <= 0 || out <= 0) return 0;
  const size_t K = (size_t)hw * c;
  return K * out * sizeof(bf16) + K * out * sizeof(float) + 4096;   // packed weight + (backward) fp32 dW accumulator
}

extern "C" int crfr_linear_fwd(const void* x, int batch, int hw, int c, const float* w, const float* bias, int out,
                               void* y, void* ws, size_t ws_bytes, void* stream) {
  CRFR_TRY(check_shape("linear_fwd", batch, hw, c, out));
  CRFR_CHECK_ARG(x && w && y && ws, "linear_fwd: null pointer");
  const long long K = (long long)hw * c;
  if (ws_bytes < (size_t)K * out * sizeof(bf16)) {
    crfr_set_error("linear_fwd: workspace %zu < %zu", ws_bytes, (size_t)K * out * sizeof(bf16));
    return CRFR_EWORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  bf16* wp = (bf16*)ws;
  fc_pack_kernel<<<crfr_cdiv(K * out, 256), 256, 0, st>>>(w, wp, nullptr, out, c, hw);
  CRFR_COUNT_LAUNCH();
  CRFR_LAUNCH_CHECK();
  TcGemm g{x, batch, 1, 1, (int)K, (int)K, wp, 1, 0, 1, out, 64, y, out, 0, bias};
  return crfr_tc_gemm(g, st);
}

extern "C" int crfr_linear_bwd(const void* x, const void* dy, int batch, int hw, int c, const float* w, int out, void* dx,
                               float* dw, float* dbias, void* ws, size_t ws_bytes, void* stream) {
  CRFR_TRY(check_shape("linear_bwd", batch, hw, c, out));
  CRFR_CHECK_ARG(x && dy && w && ws && (dx || dw || dbias), "linear_bwd: null pointer");
  const long long K = (long long)hw * c;
  if (ws_bytes < crfr_linear_workspace_bytes(batch, hw, c, out) - 4096) {
    crfr_set_error("linear_bwd: workspace %zu < %zu", ws_bytes, crfr_linear_workspace_bytes(batch, hw, c, out));
    return CRFR_EWORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  bf16* wpt = (bf16*)ws;
  float* G = (float*)((uint8_t*)ws + (((size_t)K * out * sizeof(bf16) + 255) & ~(size_t)255));
  if (dx) {
    fc_pack_kernel<<<crfr_cdiv(K * out, 256), 256, 0, st>>>(w, nullptr, wpt, out, c, hw);
    CRFR_COUNT_LAUNCH();
    CRFR_LAUNCH_CHECK();
    TcGemm g{dy, batch, 1, 1, out, out, wpt, 1, 0, 1, (int)K, 0, dx, (int)K, 0, nullptr};
    CRFR_TRY(crfr_tc_gemm(g, st));
  }
  if (dw) {
    CRFR_CUDA(cudaMemsetAsync(G, 0, sizeof(float) * (size_t)K * out, st));
    TcWgrad wg{x, batch, 1, 1, (int)K, (int)K, dy, out, out, 0, G};
    CRFR_TRY(crfr_tc_wgrad_raw(wg, st));
    fc_unpack_kernel<<<crfr_cdiv(K * out, 256), 256, 0, st>>>(G, dw, out, c, hw);
    CRFR_COUNT_LAUNCH();
    CRFR_LAUNCH_CHECK();
  }
  if (dbias) CRFR_TRY(crfr_colsum(dy, out, out, batch, dbias, ws, ws_bytes, st));
  return CRFR_OK;
}
