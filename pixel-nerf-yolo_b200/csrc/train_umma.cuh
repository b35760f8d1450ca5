// Host-side interface of the tcgen05 training GEMMs (train_umma.cu), used by field_bwd.cu.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace pnr {
namespace tg {

// OUT[M, n_valid] = epilogue(sum over sources A_s[M, K_s] . W_s^T), W_s packed by pack_rowgemm (n_out padded to 256, K to 64).
// epilogue: v = acc; if mask_src: v = mask_src[row, col] > 0 ? v : 0; v += bias[col] + bias2[col]; v += res_in[row, col];
//           out_f32[row, col] = v; out_bf16[row, col] = bf16(relu_out ? max(v, 0) : v).   res_in may alias out_f32.
struct RowGemmArgs {
  long long M;
  int n_valid;                       // output columns stored (the packed weights are padded to a multiple of 256)
  const float* bias;                 // [>= n_valid rounded up to 4 inside the padded extent] or null
  const float* bias2;                // second bias vector added the same way (lin_z bias next to fc_1 / lin_in bias) or null
  const __nv_bfloat16* mask_src; long long ld_mask;
  const float* res_in; long long ld_res;
  float* out_f32; long long ld_f32;
  __nv_bfloat16* out_bf16; long long ld_bf16;
  int relu_out;
  float* colsum_out;                 // [n_valid] or null: += column sums of v over the rows (bias gradients), fused into the epilogue
  float* colsum_out2;                // a second destination for the same sums (fc_1 bias and lin_z bias see the same gradient)
  int nN, n_pad, nK0, nK1;           // filled in by rowgemm()
};
struct RowGemmSrc {
  const __nv_bfloat16* A; long long lda;   // [M, K] row-major bf16, lda multiple of 8
  int K;                                    // multiple of 64 (columns beyond the logical width must be zero)
  const void* Wp;                           // packed weights (pack_rowgemm), 1024-byte aligned
};
struct WgradArgs {
  float* dW; int ldw;
  long long M; int N, K;
  int nNb, nKb, n_slabs;
};

size_t packed_rowgemm_bytes(int n_out, int n_in);
// W (rows x cols, leading dimension ldw) -> packed stream; transposed = 1 packs W^T (input gradients)
int pack_rowgemm(const float* W, int rows, int cols, int ldw, int transposed, void* dst, cudaStream_t st);
// the same for up to kMaxPackJobs matrices in ONE launch
constexpr int kMaxPackJobs = 24;
struct PackJob { const float* W; int rows, cols, ldw; void* dst; };
int pack_rowgemm_many(const PackJob* jobs, int n_jobs, int transposed, cudaStream_t st);
int rowgemm(const RowGemmSrc& s0, const RowGemmSrc* s1, RowGemmArgs g, cudaStream_t st);
// dW[N, K] (leading dimension ldw) += dY[M, N]^T X[M, K]; dY / X row-major bf16 with leading dimensions ldy / ldx (multiples of 8;
// columns up to the next multiple of 64 must be readable or beyond the declared width, where TMA zero-fills)
int wgrad(const __nv_bfloat16* dY, long long ldy, const __nv_bfloat16* X, long long ldx, float* dW, int ldw, long long M, int N, int K,
          cudaStream_t st);

}  // namespace tg
}  // namespace pnr
