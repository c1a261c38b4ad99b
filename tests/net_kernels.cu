// Test harness for the network kernels (tests/test_gpu_net_kernels.py): launches k_mlp_tc<m>,
// k_mlp_tc1<m> and k_mlp_f32 directly, with a chosen grid, a static or device-side row count, a
// probability leading dimension and a zero2 pointer, so that tests reach the kernel forms and
// grid-stride loops that the public API only meets in production-sized runs.
#include <cstring>
#include <vector>

#include "../corintho_ai_b200/csrc/mlp.cuh"
#include "../corintho_ai_b200/csrc/mlp_tc.cuh"

using namespace cb200;

namespace {
NetTC g_tc;
NetF32 g_f32;
int g_precision = -1;  // as cb200_trainer_set_weights: 0 fp32, 1 bf16, 2 fp16, 3 bf16x3

// 70-float encoded rows -> cstates, as cb200_trainer_evaluate packs them
std::vector<ulonglong2> pack_rows(const float *rows, int n) {
  std::vector<ulonglong2> hs(n);
  for (int i = 0; i < n; ++i) {
    const float *r = rows + (size_t)i * CB200_STATE_SIZE;
    uint64_t w0 = 0, w1 = 0;
    for (int j = 0; j < 64; ++j)
      if (r[j] != 0.0f) w0 |= 1ull << (16 * (j & 3) + (j >> 2));
    for (int j = 0; j < 6; ++j) w1 |= (uint64_t)(int)(r[64 + j] * 4.0f + 0.5f) << (8 * j);
    hs[i] = make_ulonglong2(w0, w1);
  }
  return hs;
}

template <int kMode>
cudaError_t launch_tc(int form, int grid, const ulonglong2 *st, const int32_t *d_n, int n_static, float *eval,
                      float *probs, int ld, int32_t *zero2) {
  if (form == 0) {
    const size_t smem = kMode == 2 ? kTcSmemBytesX3 : kTcSmemBytes;
    cudaFuncSetAttribute(k_mlp_tc<kMode>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    k_mlp_tc<kMode><<<grid, kTcThreads, smem>>>((const uint8_t *)g_tc.w, st, d_n, n_static, eval, probs, ld, zero2);
  } else {
    const size_t smem = tc_smem_bytes(1, kMode == 2 ? 2 : 1);
    cudaFuncSetAttribute(k_mlp_tc1<kMode>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    k_mlp_tc1<kMode><<<grid, 128, smem>>>((const uint8_t *)g_tc.w, st, d_n, n_static, eval, probs, ld, zero2);
  }
  return cudaGetLastError();
}
}  // namespace

extern "C" {

const char *nk_last_error() { return last_error_ref().c_str(); }

// Uploads the C-ABI weight vector with net_f32_upload (precision 0) or net_tc_upload (1..3).
int nk_upload(const float *weights, int precision) {
  const int rc = precision == 0 ? net_f32_upload(g_f32, weights)
                                : net_tc_upload(g_tc, weights, precision == 1 ? 0 : (precision == 2 ? 1 : 2));
  if (rc == CB200_OK) g_precision = precision;
  return rc;
}

// Runs one kernel form on `n_rows` encoded rows: form 0 = k_mlp_tc (two tiles per CTA), 1 = k_mlp_tc1
// (one tile), 2 = k_mlp_f32. grid <= 0 takes the grid launch_mlp_tc / launch_mlp_f32 would choose
// for n_max rows. count < 0: the row count is n_static; otherwise it is read from device memory
// (value `count`). eval [n_max], probs ([96][ld] for the tensor-core forms, [n_max][96] for fp32)
// and zero2 [4] are copied in, the kernel runs, and they are copied back.
int nk_run(int form, const float *rows, int n_rows, int n_max, int n_static, int count, int grid, int ld,
           float *eval, float *probs, int32_t *zero2) {
  if (g_precision < 0 || (form == 2) != (g_precision == 0) || n_rows > n_max)
    return set_error(CB200_ERR_ARG, "nk_run: form / precision / size mismatch");
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (grid <= 0) {
    const int tiles = (n_max + 127) / 128, pairs = (n_max + 255) / 256;
    grid = form == 0 ? (g_tc.mode == 2 ? (pairs < sms ? pairs : sms) : (pairs < 2 * sms ? pairs : 2 * sms))
                     : (tiles < sms ? tiles : sms);
  }
  const size_t probs_floats = form == 2 ? (size_t)n_max * CB200_NUM_MOVES : (size_t)CB200_NUM_MOVES * ld;
  std::vector<ulonglong2> hs = pack_rows(rows, n_rows);
  hs.resize(n_max > 0 ? n_max : 1, make_ulonglong2(0, 0));
  ulonglong2 *d_st = nullptr;
  float *d_eval = nullptr, *d_probs = nullptr;
  int32_t *d_i = nullptr;  // zero2 [4], device count
  CB_CUDA(cudaMalloc(&d_st, hs.size() * sizeof(ulonglong2)));
  CB_CUDA(cudaMalloc(&d_eval, (n_max > 0 ? n_max : 1) * sizeof(float)));
  CB_CUDA(cudaMalloc(&d_probs, (probs_floats > 0 ? probs_floats : 1) * sizeof(float)));
  CB_CUDA(cudaMalloc(&d_i, 5 * sizeof(int32_t)));
  CB_CUDA(cudaMemcpy(d_st, hs.data(), hs.size() * sizeof(ulonglong2), cudaMemcpyHostToDevice));
  CB_CUDA(cudaMemcpy(d_eval, eval, n_max * sizeof(float), cudaMemcpyHostToDevice));
  CB_CUDA(cudaMemcpy(d_probs, probs, probs_floats * sizeof(float), cudaMemcpyHostToDevice));
  CB_CUDA(cudaMemcpy(d_i, zero2, 4 * sizeof(int32_t), cudaMemcpyHostToDevice));
  CB_CUDA(cudaMemcpy(d_i + 4, &count, sizeof(int32_t), cudaMemcpyHostToDevice));
  const int32_t *d_n = count >= 0 ? d_i + 4 : nullptr;
  cudaError_t e;
  if (form == 2) {
    cudaFuncSetAttribute(k_mlp_f32, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMlpSmemBytes);
    k_mlp_f32<<<grid, kNetThreads, kMlpSmemBytes>>>(g_f32.w, d_st, d_n, n_static, d_eval, d_probs, d_i);
    e = cudaGetLastError();
  } else if (g_tc.mode == 0) {
    e = launch_tc<0>(form, grid, d_st, d_n, n_static, d_eval, d_probs, ld, d_i);
  } else if (g_tc.mode == 1) {
    e = launch_tc<1>(form, grid, d_st, d_n, n_static, d_eval, d_probs, ld, d_i);
  } else {
    e = launch_tc<2>(form, grid, d_st, d_n, n_static, d_eval, d_probs, ld, d_i);
  }
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) return set_error(CB200_ERR_CUDA, std::string("nk_run: ") + cudaGetErrorString(e));
  CB_CUDA(cudaMemcpy(eval, d_eval, n_max * sizeof(float), cudaMemcpyDeviceToHost));
  CB_CUDA(cudaMemcpy(probs, d_probs, probs_floats * sizeof(float), cudaMemcpyDeviceToHost));
  CB_CUDA(cudaMemcpy(zero2, d_i, 4 * sizeof(int32_t), cudaMemcpyDeviceToHost));
  cudaFree(d_st), cudaFree(d_eval), cudaFree(d_probs), cudaFree(d_i);
  return CB200_OK;
}

}  // extern "C"
