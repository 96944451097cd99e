// C-ABI entry points that dispatch between the fp32 (FFMA) and bf16 (tcgen05) GEMM kernels,
// plus version / error reporting.
#include <string.h>

#include <mutex>
#include <unordered_map>

#include "edg_common.cuh"

namespace edg {

static thread_local char g_cuda_err[256] = "";
void set_cuda_error(cudaError_t e) {
  const char* s = cudaGetErrorString(e);
  strncpy(g_cuda_err, s ? s : "unknown", sizeof(g_cuda_err) - 1);
  g_cuda_err[sizeof(g_cuda_err) - 1] = 0;
}

int ensure_dyn_smem(const void* kernel, size_t smem) {
  static std::mutex mu;      // (no shortcut for small sizes: static + dynamic shared memory together may exceed 48 KB)
  static std::unordered_map<uint64_t, size_t> seen;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return check_launch();
  const uint64_t key = ((uint64_t)(uint32_t)dev << 56) ^ (uint64_t)reinterpret_cast<uintptr_t>(kernel);
  std::lock_guard<std::mutex> lock(mu);
  size_t& have = seen[key];
  if (smem > have) {
    if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return check_launch();
    have = smem;
  }
  return EDG_OK;
}

// edg_gemm_simt.cu
template <typename TA>
int launch_linear_simt(const void* A, int64_t lda, int M, int K, const void* W, int64_t ldw, int Nout,
                       const float* bias, int act, void* C, int c_dtype, int64_t ldc, cudaStream_t s);
template <typename T>
int launch_wgrad_simt(const void* A, int64_t lda, int K1, const void* B, int64_t ldb, int K2, int R,
                      float* dW, int64_t lddw, int accumulate, float* ws, cudaStream_t s);
size_t wgrad_simt_workspace(int R, int K1, int K2);
// edg_gemm_tc.cu
int launch_linear_tc(const void* A, int64_t lda, int M, int K, const void* W, int64_t ldw, int Nout,
                     const float* bias, int act, void* C, int c_dtype, int64_t ldc, cudaStream_t s);
int launch_wgrad_tc(const void* A, int64_t lda, int K1, const void* B, int64_t ldb, int K2, int R, float* dW,
                    int64_t lddw, float* dbias, int bias_of, int accumulate, float* ws, cudaStream_t s);
size_t wgrad_tc_workspace(int R, int K1, int K2);
int launch_wgrad_tc_batch(int n, const void* const* A, int64_t lda, int K1, const void* const* B, int64_t ldb, int K2, int R,
                          float* const* dW, int64_t lddw, float* const* dbias, int bias_of, float* ws, cudaStream_t s);
size_t wgrad_tc_batch_workspace(int n, int R, int K1, int K2);

}  // namespace edg

using namespace edg;

extern "C" int edg_version(void) { return EDG_ABI_VERSION; }

extern "C" const char* edg_strerror(int status) {
  switch (status) {
    case EDG_OK: return "ok";
    case EDG_ERR_ARG: return "invalid argument (null pointer, negative size or bad enum)";
    case EDG_ERR_ALIGN: return "pointer or leading dimension is not 16-byte aligned";
    case EDG_ERR_DTYPE: return "dtype combination not implemented";
    case EDG_ERR_ARCH: return "device is not sm_100";
    case EDG_ERR_WORKSPACE: return "workspace too small";
    case EDG_ERR_CUDA: return "CUDA call failed at enqueue (see edg_last_cuda_error)";
    case EDG_ERR_UNSUPPORTED: return "shape outside what the kernels implement";
    default: return "unknown status";
  }
}

extern "C" const char* edg_last_cuda_error(void) { return g_cuda_err; }

extern "C" int edg_linear(const void* A, int ab_dtype, int64_t lda, int32_t M, int32_t K,
                          const void* W, int64_t ldw, int32_t Nout, const float* bias, int act,
                          void* C, int c_dtype, int64_t ldc, edg_stream stream) {
  if (M < 0 || K <= 0 || Nout <= 0) return EDG_ERR_ARG;
  if (M == 0) return EDG_OK;
  if (!A || !W || !C) return EDG_ERR_ARG;
  if (act < EDG_ACT_NONE || act > EDG_ACT_RELU) return EDG_ERR_ARG;
  if (c_dtype != EDG_F32 && c_dtype != EDG_BF16) return EDG_ERR_DTYPE;
  if (lda < K || ldw < K || ldc < Nout) return EDG_ERR_ARG;
  if (!aligned16(A) || !aligned16(W) || !aligned16(C)) return EDG_ERR_ALIGN;
  if (!row_pitch_ok(ab_dtype, lda) || !row_pitch_ok(ab_dtype, ldw) || !row_pitch_ok(c_dtype, ldc)) return EDG_ERR_ALIGN;
  cudaStream_t s = (cudaStream_t)stream;
  if (ab_dtype == EDG_F32) return launch_linear_simt<float>(A, lda, M, K, W, ldw, Nout, bias, act, C, c_dtype, ldc, s);
  if (ab_dtype == EDG_BF16) return launch_linear_tc(A, lda, M, K, W, ldw, Nout, bias, act, C, c_dtype, ldc, s);
  return EDG_ERR_DTYPE;
}

extern "C" size_t edg_wgrad_workspace(int32_t R, int32_t K1, int32_t K2, int dtype) {
  if (R <= 0 || K1 <= 0 || K2 <= 0) return 16;
  size_t m = (dtype == EDG_BF16) ? wgrad_tc_workspace(R, K1, K2) : wgrad_simt_workspace(R, K1, K2);
  size_t c = edg_colsum_workspace(R, K1 > K2 ? K1 : K2);
  return m + c + 256;
}

extern "C" int edg_wgrad(const void* A, int64_t lda, int32_t K1, const void* B, int64_t ldb, int32_t K2,
                         int dtype, int32_t R, float* dW, int64_t lddw, float* dbias, int bias_of,
                         int accumulate, void* ws, size_t ws_bytes, edg_stream stream) {
  if (R < 0 || K1 <= 0 || K2 <= 0 || !dW || lddw < K2) return EDG_ERR_ARG;
  if (bias_of < 0 || bias_of > 2 || (bias_of && !dbias)) return EDG_ERR_ARG;
  if (dtype != EDG_F32 && dtype != EDG_BF16) return EDG_ERR_DTYPE;
  cudaStream_t s = (cudaStream_t)stream;
  if (R == 0) {
    if (!accumulate) {
      cudaMemset2DAsync(dW, lddw * sizeof(float), 0, K2 * sizeof(float), K1, s);
      if (bias_of) cudaMemsetAsync(dbias, 0, (bias_of == 1 ? K1 : K2) * sizeof(float), s);
    }
    return check_launch();
  }
  if (!A || !B || !ws) return EDG_ERR_ARG;
  if (lda < K1 || ldb < K2) return EDG_ERR_ARG;
  if (!aligned16(A) || !aligned16(B) || !aligned16(ws) || !row_pitch_ok(dtype, lda) || !row_pitch_ok(dtype, ldb)) return EDG_ERR_ALIGN;
  if (ws_bytes < edg_wgrad_workspace(R, K1, K2, dtype)) return EDG_ERR_WORKSPACE;
  if (dtype == EDG_BF16) return launch_wgrad_tc(A, lda, K1, B, ldb, K2, R, dW, lddw, dbias, bias_of, accumulate, (float*)ws, s);
  int rc = launch_wgrad_simt<float>(A, lda, K1, B, ldb, K2, R, dW, lddw, accumulate, (float*)ws, s);
  if (rc) return rc;
  if (bias_of) {
    char* cws = (char*)ws + ((wgrad_simt_workspace(R, K1, K2) + 255) & ~(size_t)255);
    const void* X = bias_of == 1 ? A : B;
    const int64_t ldx = bias_of == 1 ? lda : ldb;
    const int Cc = bias_of == 1 ? K1 : K2;
    rc = edg_colsum(X, dtype, ldx, R, Cc, dbias, accumulate, cws, edg_colsum_workspace(R, Cc), stream);
  }
  return rc;
}

extern "C" size_t edg_wgrad_batch_workspace(int32_t n, int32_t R, int32_t K1, int32_t K2) {
  if (n <= 0 || R <= 0 || K1 <= 0 || K2 <= 0) return 16;
  return wgrad_tc_batch_workspace(n, R, K1, K2) + 256;
}

extern "C" int edg_wgrad_batch(int32_t n, const void* const* A, int64_t lda, int32_t K1, const void* const* B, int64_t ldb,
                               int32_t K2, int dtype, int32_t R, float* const* dW, int64_t lddw, float* const* dbias,
                               int bias_of, void* ws, size_t ws_bytes, edg_stream stream) {
  if (n <= 0 || R <= 0 || K1 <= 0 || K2 <= 0 || !A || !B || !dW || lddw < K2 || !ws) return EDG_ERR_ARG;
  if (bias_of < 0 || bias_of > 2 || (bias_of && !dbias)) return EDG_ERR_ARG;
  if (dtype != EDG_BF16) return EDG_ERR_DTYPE;              // the fp32-parity mode keeps one launch per problem
  if (n > 8) return EDG_ERR_UNSUPPORTED;
  if (lda < K1 || ldb < K2) return EDG_ERR_ARG;
  if (!aligned16(ws) || !row_pitch_ok(dtype, lda) || !row_pitch_ok(dtype, ldb)) return EDG_ERR_ALIGN;
  for (int i = 0; i < n; ++i) {
    if (!A[i] || !B[i] || !dW[i] || (bias_of && !dbias[i])) return EDG_ERR_ARG;
    if (!aligned16(A[i]) || !aligned16(B[i])) return EDG_ERR_ALIGN;
  }
  if (ws_bytes < edg_wgrad_batch_workspace(n, R, K1, K2)) return EDG_ERR_WORKSPACE;
  return launch_wgrad_tc_batch(n, A, lda, K1, B, ldb, K2, R, dW, lddw, dbias, bias_of, (float*)ws, (cudaStream_t)stream);
}
