/* Internal header, NOT part of the product ABI (include/pixelnerf_b200.h): test hooks of the training GEMMs, used by
 * tests/test_gpu_train.py, scripts/rowgemm_bench.py and scripts/wgrad_probe.py. */
#ifndef PNR_LAB_H
#define PNR_LAB_H
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif
/* Stand-alone entry points of the tcgen05 training GEMMs (train_umma.cu): fp32 device inputs are rounded to bf16, then
 * out[M,N] = epilogue(A[M,K] W[N,K]^T) (rowgemm: optional bias [N], relu mask source [M,N], residual [M,N]; fp32 and / or bf16
 * outputs) and dW[N,K] += dY[M,N]^T X[M,K] (wgrad).  workspace: pnr_lab_gemm_workspace_bytes(M, N, K). */
size_t pnr_lab_gemm_workspace_bytes(long long M, int N, int K);
int pnr_lab_rowgemm(const float* A, const float* W, const float* bias, const float* mask_src, const float* res_in, float* out_f32,
                    void* out_bf16, long long M, int N, int K, int relu_out, void* workspace, size_t workspace_bytes, void* stream);
int pnr_lab_wgrad(const float* dY, const float* X, float* dW, long long M, int N, int K, void* workspace, size_t workspace_bytes,
                  void* stream);
#ifdef __cplusplus
}
#endif
#endif
