// Training path of the field function: PixelNeRFNet.forward (src/model/models.py:153-318) with every activation
// the backward pass needs kept on a caller-owned tape, and the backward pass itself -- gradients of all ResnetFC
// parameters (src/model/resnetfc.py:103-132), of the encoder's feature maps (SpatialEncoder.latent, through the
// bilinear gather, src/model/encoder.py:79-108) and of the query points (through the projection, models.py:168-230,
// and the positional encoding, src/model/code.py:30-42; the renderer needs them because sample_fine_depth is
// differentiable in the coarse depth, src/render/nerf.py:156-167,296-298).
//
// What autograd does for the reference (PixelNerfTrainer.calc_losses -> loss.backward(), BASELINE config 3) is one
// explicit chain of kernels here.  Arithmetic is fp32 on the CUDA cores (SIMT SGEMM in all four operand layouts):
// the training step is the parity case of this round (gradients vs autograd <= 1e-3 relative), not the timed one.
#include "pnr_common.cuh"
#include "train_umma.cuh"

namespace pnr {

int validate_scene_points(const pnr_scene* sc, const pnr_points* q, const char* who);

namespace bwd {

constexpr int BM = 128, BN = 128, BK = 8;

struct GemmArgs {
  const float* A; long long lda;     // A_T ? A[k*lda + i] : A[i*lda + k]
  const float* B; long long ldb;     // B_T ? B[j*ldb + k] : B[k*ldb + j]
  float* C; long long ldc;           // C[i*ldc + j]
  const float* bias;                 // + bias[j]            (mode 0 only)
  const float* add_src;              // + add_src[i*ldc + j] (mode 0 only; may alias C)
  const float* mask;                 // product *= (mask[i*ldc + j] > 0)
  long long I; int J; long long K;
  int relu_a, relu_b;
  int mode;                          // 0: C = v, 1: C += v, 2: atomicAdd(C, v) (split-K over gridDim.z)
  long long k_per_split;
};

// C[I,J] (op)= sum_k A(i,k) * B(k,j)
template <bool A_T, bool B_T>
__global__ void __launch_bounds__(256) sgemm_kernel(const GemmArgs g) {
  __shared__ __align__(16) float As[BK][BM];
  __shared__ __align__(16) float Bs[BK][BN];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const long long i0 = (long long)blockIdx.x * BM;
  const int j0 = blockIdx.y * BN;
  const long long kbeg = (long long)blockIdx.z * g.k_per_split;
  const long long kend = kbeg + g.k_per_split < g.K ? kbeg + g.k_per_split : g.K;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  // 4 consecutive elements of one row: one 16-byte load when the run is inside the matrix and aligned
  auto load4 = [](const float* base, long long row, long long ld, long long c, long long c_end, bool row_ok, float (&v)[4]) {
    const float* p = base + row * ld + c;
    if (row_ok && c + 4 <= c_end && ((reinterpret_cast<uintptr_t>(p) & 15) == 0)) {
      const float4 x = __ldg(reinterpret_cast<const float4*>(p));
      v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w;
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e) v[e] = (row_ok && c + e < c_end) ? p[e] : 0.f;
    }
  };
  for (long long k0 = kbeg; k0 < kend; k0 += BK) {
    float a[4], b[4];
    if (A_T) {          // i contiguous: thread -> (k = tid / 32, 4 consecutive i)
      const long long k = k0 + (tid >> 5);
      load4(g.A, k, g.lda, i0 + (tid & 31) * 4, g.I, k < kend, a);
    } else {            // k contiguous: thread -> (i = tid / 2, 4 consecutive k)
      const long long i = i0 + (tid >> 1);
      load4(g.A, i, g.lda, k0 + (tid & 1) * 4, kend, i < g.I, a);
    }
    if (!B_T) {         // j contiguous
      const long long k = k0 + (tid >> 5);
      load4(g.B, k, g.ldb, j0 + (tid & 31) * 4, g.J, k < kend, b);
    } else {            // k contiguous
      const long long j = j0 + (tid >> 1);
      load4(g.B, j, g.ldb, k0 + (tid & 1) * 4, kend, j < g.J, b);
    }
    if (g.relu_a) {
#pragma unroll
      for (int e = 0; e < 4; ++e) a[e] = fmaxf(a[e], 0.f);
    }
    if (g.relu_b) {
#pragma unroll
      for (int e = 0; e < 4; ++e) b[e] = fmaxf(b[e], 0.f);
    }
    if (A_T) {
#pragma unroll
      for (int e = 0; e < 4; ++e) As[tid >> 5][(tid & 31) * 4 + e] = a[e];
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e) As[(tid & 1) * 4 + e][tid >> 1] = a[e];
    }
    if (!B_T) {
#pragma unroll
      for (int e = 0; e < 4; ++e) Bs[tid >> 5][(tid & 31) * 4 + e] = b[e];
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e) Bs[(tid & 1) * 4 + e][tid >> 1] = b[e];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 8]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[k][ty * 8 + 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[k][tx * 8]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[k][tx * 8 + 4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const long long gi = i0 + ty * 8 + i;
    if (gi >= g.I) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int gj = j0 + tx * 8 + j;
      if (gj >= g.J) continue;
      const long long o = gi * g.ldc + gj;
      float v = acc[i][j];
      if (g.mask && !(g.mask[o] > 0.f)) v = 0.f;
      if (g.mode == 0) {
        if (g.bias) v += g.bias[gj];
        if (g.add_src) v += g.add_src[o];
        g.C[o] = v;
      } else if (g.mode == 1) {
        g.C[o] += v;
      } else {
        atomicAdd(g.C + o, v);
      }
    }
  }
}

// Same contract on the tensor cores: TF32 operands (10-bit mantissa, round-to-nearest), fp32 accumulate, legacy
// mma.sync.m16n8k8 -- the optional fast arithmetic of the training path (PNR_SCENE_TRAIN_TF32).  128x128x16 tiles, 8 warps
// of 64x32; operands are rounded once when they are staged in shared memory and read back with ldmatrix.
__device__ __forceinline__ float to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
constexpr int TK = 16, TKP = 20;   // k-tile and padded row pitch in floats (80 B: the 8 row addresses of an ldmatrix hit 32 distinct banks)
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const float* p) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
template <bool A_T, bool B_T>
__global__ void __launch_bounds__(256) sgemm_tf32_kernel(const GemmArgs g) {
  // Each operand is staged the way it arrives from global memory, so the staging stores are contiguous and conflict-free:
  //  * k-contiguous operand (A of X W^T and dY W; B = W of X W^T): [row][k], pitch TKP; an 8x8 b16 ldmatrix tile = 8 rows x 4
  //    tf32 values, so one ldmatrix.x4 delivers a whole m16k8 A fragment (or the B fragments of two n8 tiles);
  //  * row-contiguous operand (the transposed ones of dY W and dY^T X): [k][row], pitch TP; fragments by 32-bit loads.
  constexpr int TP = 136;            // [k][row] pitch: 8 banks (mod 32) per k row -> the (k = lane % 4, row = lane / 4) loads are conflict-free
  constexpr int kBufFloats = BM * TKP > TK * TP ? BM * TKP : TK * TP;
  __shared__ __align__(16) float As_raw[2][kBufFloats];
  __shared__ __align__(16) float Bs_raw[2][kBufFloats];
  auto As_rk = [&](int buf, int row, int k) -> float* { return &As_raw[buf][row * TKP + k]; };
  auto As_kr = [&](int buf, int k, int row) -> float* { return &As_raw[buf][k * TP + row]; };
  auto Bs_rk = [&](int buf, int row, int k) -> float* { return &Bs_raw[buf][row * TKP + k]; };
  auto Bs_kr = [&](int buf, int k, int row) -> float* { return &Bs_raw[buf][k * TP + row]; };
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int gq = lane >> 2, tq = lane & 3;
  const int wm = (warp & 1) * 64, wn = (warp >> 1) * 32;
  const long long i0 = (long long)blockIdx.x * BM;
  const int j0 = blockIdx.y * BN;
  const long long kbeg = (long long)blockIdx.z * g.k_per_split;
  const long long kend = kbeg + g.k_per_split < g.K ? kbeg + g.k_per_split : g.K;
  float acc[4][4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[a][b][c] = 0.f;

  // 8 consecutive elements of one row: two 16-byte loads when the run is inside the matrix and aligned
  auto load8 = [](const float* base, long long row, long long ld, long long c, long long c_end, bool row_ok, float (&v)[8]) {
    const float* p = base + row * ld + c;
    if (row_ok && c + 8 <= c_end && ((reinterpret_cast<uintptr_t>(p) & 15) == 0)) {
      const float4 x = __ldg(reinterpret_cast<const float4*>(p)), y = __ldg(reinterpret_cast<const float4*>(p) + 1);
      v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; v[4] = y.x; v[5] = y.y; v[6] = y.z; v[7] = y.w;
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = (row_ok && c + e < c_end) ? p[e] : 0.f;
    }
  };
  // register-prefetched, double-buffered main loop: the global loads of tile k0 + TK are in flight while tile k0 is multiplied
  float a[8], b[8];
  auto gload = [&](long long k0) {
    if (A_T) {          // i contiguous: thread -> (k = tid / 16, 8 consecutive i)
      const long long k = k0 + (tid >> 4);
      load8(g.A, k, g.lda, i0 + (tid & 15) * 8, g.I, k < kend, a);
    } else {            // k contiguous: thread -> (i = tid / 2, 8 consecutive k)
      const long long i = i0 + (tid >> 1);
      load8(g.A, i, g.lda, k0 + (tid & 1) * 8, kend, i < g.I, a);
    }
    if (!B_T) {
      const long long k = k0 + (tid >> 4);
      load8(g.B, k, g.ldb, j0 + (tid & 15) * 8, g.J, k < kend, b);
    } else {
      const long long j = j0 + (tid >> 1);
      load8(g.B, j, g.ldb, k0 + (tid & 1) * 8, kend, j < g.J, b);
    }
  };
  auto sstore = [&](int buf) {
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      if (g.relu_a) a[e] = fmaxf(a[e], 0.f);
      if (g.relu_b) b[e] = fmaxf(b[e], 0.f);
      a[e] = to_tf32(a[e]);
      b[e] = to_tf32(b[e]);
    }
    {
      float4* d = reinterpret_cast<float4*>(A_T ? As_kr(buf, tid >> 4, (tid & 15) * 8) : As_rk(buf, tid >> 1, (tid & 1) * 8));
      d[0] = make_float4(a[0], a[1], a[2], a[3]); d[1] = make_float4(a[4], a[5], a[6], a[7]);
    }
    {
      float4* d = reinterpret_cast<float4*>(!B_T ? Bs_kr(buf, tid >> 4, (tid & 15) * 8) : Bs_rk(buf, tid >> 1, (tid & 1) * 8));
      d[0] = make_float4(b[0], b[1], b[2], b[3]); d[1] = make_float4(b[4], b[5], b[6], b[7]);
    }
  };
  // ldmatrix lane roles: lane = 8 * mat + r
  const int lm = lane >> 3, lr = lane & 7;
  const int a_row = lr + (lm & 1) * 8, a_k = (lm >> 1) * 4;      // A: matrices (rows 0-7, k), (rows 8-15, k), (rows 0-7, k+4), (rows 8-15, k+4)
  const int b_row = lr + (lm >> 1) * 8, b_k = (lm & 1) * 4;      // B: (n 0-7, k), (n 0-7, k+4), (n 8-15, k), (n 8-15, k+4)
  int buf = 0;
  if (kbeg < kend) { gload(kbeg); sstore(0); }
  __syncthreads();
  for (long long k0 = kbeg; k0 < kend; k0 += TK, buf ^= 1) {
    const bool more = k0 + TK < kend;
    if (more) gload(k0 + TK);
#pragma unroll
    for (int ks = 0; ks < TK; ks += 8) {
      uint32_t af[4][4], bf[2][4];
      if (A_T) {
#pragma unroll
        for (int mi = 0; mi < 4; ++mi) {
          const int m = wm + mi * 16 + gq;
          af[mi][0] = __float_as_uint(*As_kr(buf, ks + tq, m));
          af[mi][1] = __float_as_uint(*As_kr(buf, ks + tq, m + 8));
          af[mi][2] = __float_as_uint(*As_kr(buf, ks + tq + 4, m));
          af[mi][3] = __float_as_uint(*As_kr(buf, ks + tq + 4, m + 8));
        }
      } else {
#pragma unroll
        for (int mi = 0; mi < 4; ++mi) ldmatrix_x4(af[mi], As_rk(buf, wm + mi * 16 + a_row, ks + a_k));
      }
      if (!B_T) {
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) {
          const int n = wn + ni * 8 + gq;
          bf[ni >> 1][(ni & 1) * 2] = __float_as_uint(*Bs_kr(buf, ks + tq, n));
          bf[ni >> 1][(ni & 1) * 2 + 1] = __float_as_uint(*Bs_kr(buf, ks + tq + 4, n));
        }
      } else {
#pragma unroll
        for (int np = 0; np < 2; ++np) ldmatrix_x4(bf[np], Bs_rk(buf, wn + np * 16 + b_row, ks + b_k));
      }
#pragma unroll
      for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni)
          asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                       : "+f"(acc[mi][ni][0]), "+f"(acc[mi][ni][1]), "+f"(acc[mi][ni][2]), "+f"(acc[mi][ni][3])
                       : "r"(af[mi][0]), "r"(af[mi][1]), "r"(af[mi][2]), "r"(af[mi][3]), "r"(bf[ni >> 1][(ni & 1) * 2]),
                         "r"(bf[ni >> 1][(ni & 1) * 2 + 1]));
    }
    if (more) sstore(buf ^ 1);
    __syncthreads();
  }
#pragma unroll
  for (int mi = 0; mi < 4; ++mi)
#pragma unroll
    for (int ni = 0; ni < 4; ++ni)
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const long long gi = i0 + wm + mi * 16 + gq + (c >> 1) * 8;
        const int gj = j0 + wn + ni * 8 + tq * 2 + (c & 1);
        if (gi >= g.I || gj >= g.J) continue;
        const long long o = gi * g.ldc + gj;
        float v = acc[mi][ni][c];
        if (g.mask && !(g.mask[o] > 0.f)) v = 0.f;
        if (g.mode == 0) {
          if (g.bias) v += g.bias[gj];
          if (g.add_src) v += g.add_src[o];
          g.C[o] = v;
        } else if (g.mode == 1) {
          g.C[o] += v;
        } else {
          atomicAdd(g.C + o, v);
        }
      }
}

static thread_local int g_use_tf32 = 0;      // set per call from the scene flags (PNR_SCENE_TRAIN_TF32)

static int launch_gemm(GemmArgs g, bool a_t, bool b_t, cudaStream_t st) {
  if (g.I == 0 || g.J == 0) return PNR_OK;
  int splits = 1;
  g.k_per_split = g.K;
  if (g.mode == 2) {                          // weight gradients: reduce over all rows, few output tiles -> split K
    const long long tiles = ((g.I + BM - 1) / BM) * ((g.J + BN - 1) / BN);
    long long want = (148 * 4 + tiles - 1) / tiles;
    long long max_splits = (g.K + 1023) / 1024;
    if (want > max_splits) want = max_splits;
    if (want < 1) want = 1;
    splits = (int)want;
    g.k_per_split = ((g.K + splits - 1) / splits + TK - 1) / TK * TK;
    splits = (int)((g.K + g.k_per_split - 1) / g.k_per_split);
  }
  dim3 grid((unsigned)((g.I + BM - 1) / BM), (unsigned)((g.J + BN - 1) / BN), (unsigned)splits);
  if (g_use_tf32) {
    if (a_t && b_t) sgemm_tf32_kernel<true, true><<<grid, 256, 0, st>>>(g);
    else if (a_t) sgemm_tf32_kernel<true, false><<<grid, 256, 0, st>>>(g);
    else if (b_t) sgemm_tf32_kernel<false, true><<<grid, 256, 0, st>>>(g);
    else sgemm_tf32_kernel<false, false><<<grid, 256, 0, st>>>(g);
    PNR_CHECK_LAUNCH("bwd::sgemm_tf32_kernel");
    return PNR_OK;
  }
  if (a_t && b_t) sgemm_kernel<true, true><<<grid, 256, 0, st>>>(g);
  else if (a_t) sgemm_kernel<true, false><<<grid, 256, 0, st>>>(g);
  else if (b_t) sgemm_kernel<false, true><<<grid, 256, 0, st>>>(g);
  else sgemm_kernel<false, false><<<grid, 256, 0, st>>>(g);
  PNR_CHECK_LAUNCH("bwd::sgemm_kernel");
  return PNR_OK;
}

// Y[M,N] = relu?(X[M,K]) W[N,K]^T + bias (+ add_src)                       nn.Linear forward
static int linear_fwd(const float* X, long long ldx, const float* W, const float* bias, const float* add_src, float* Y,
                      long long M, int N, int K, bool relu_in, cudaStream_t st) {
  GemmArgs g = {};
  g.A = X; g.lda = ldx; g.B = W; g.ldb = K; g.C = Y; g.ldc = N; g.bias = bias; g.add_src = add_src;
  g.I = M; g.J = N; g.K = K; g.relu_a = relu_in; g.mode = 0;
  return launch_gemm(g, false, true, st);
}
// dX[M,K] (=|+=) (dY[M,N] W[N,K]) * (mask > 0)                              grad wrt the input of a Linear
static int linear_bwd_input(const float* dY, const float* W, const float* mask, float* dX, long long M, int N, int K,
                            bool accumulate, cudaStream_t st) {
  GemmArgs g = {};
  g.A = dY; g.lda = N; g.B = W; g.ldb = K; g.C = dX; g.ldc = K; g.mask = mask;
  g.I = M; g.J = K; g.K = N; g.mode = accumulate ? 1 : 0;
  return launch_gemm(g, false, false, st);
}
// dW[N,K] += dY[M,N]^T relu?(X[M,K])                                        grad wrt the weight of a Linear
static int linear_bwd_weight(const float* dY, const float* X, long long ldx, float* dW, long long M, int N, int K,
                             bool relu_x, cudaStream_t st) {
  GemmArgs g = {};
  g.A = dY; g.lda = N; g.B = X; g.ldb = ldx; g.C = dW; g.ldc = K;
  g.I = N; g.J = K; g.K = M; g.relu_b = relu_x; g.mode = 2;
  return launch_gemm(g, true, false, st);
}

// db[N] += column sums of dY[M,N]
__global__ void colsum_kernel(const float* __restrict__ dY, float* __restrict__ db, long long M, int N, int rows_per_block) {
  const long long r0 = (long long)blockIdx.x * rows_per_block;
  const long long r1 = r0 + rows_per_block < M ? r0 + rows_per_block : M;
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
    float acc = 0.f;
    for (long long r = r0; r < r1; ++r) acc += dY[r * N + j];
    atomicAdd(db + j, acc);
  }
}
static int colsum(const float* dY, float* db, long long M, int N, cudaStream_t st) {
  if (M == 0) return PNR_OK;
  const int rpb = 256;
  colsum_kernel<<<(unsigned)((M + rpb - 1) / rpb), 256, 0, st>>>(dY, db, M, N, rpb);
  PNR_CHECK_LAUNCH("bwd::colsum_kernel");
  return PNR_OK;
}

// view pooling over the NS source views (util.py:489-499) and its transpose.  arg == nullptr: mean (combine_type average);
// otherwise elementwise max (combine_type max), and arg (SB, P, H) records the first maximal view, the one torch.max(dim)
// routes the gradient to.
__global__ void view_mean_kernel(const float* __restrict__ x, float* __restrict__ y, uint8_t* __restrict__ arg, int SB, int NS, int P,
                                 int H) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)SB * P * H) return;
  const int h = (int)(i % H);
  const long long sp = i / H;
  const int p = (int)(sp % P), s = (int)(sp / P);
  if (arg) {
    float m = x[((long long)s * NS * P + p) * H + h];
    int win = 0;
    for (int v = 1; v < NS; ++v) {
      const float a = x[(((long long)s * NS + v) * P + p) * H + h];
      if (a > m) { m = a; win = v; }
    }
    y[i] = m;
    arg[i] = (uint8_t)win;
    return;
  }
  float acc = 0.f;
  for (int v = 0; v < NS; ++v) acc += x[(((long long)s * NS + v) * P + p) * H + h];
  y[i] = acc / (float)NS;
}
__global__ void view_mean_bwd_kernel(const float* __restrict__ dy, float* __restrict__ dx, const uint8_t* __restrict__ arg, int SB, int NS,
                                     int P, int H) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)SB * NS * P * H) return;
  const int h = (int)(i % H);
  const long long svp = i / H;
  const int p = (int)(svp % P);
  const int s = (int)(svp / P / NS);
  const long long o = ((long long)s * P + p) * H + h;
  if (arg) { dx[i] = arg[o] == (int)(svp / P - (long long)s * NS) ? dy[o] : 0.f; return; }
  dx[i] = dy[o] / (float)NS;
}

// bf16 path helpers -----------------------------------------------------------------------------------------------------
// view pooling (as view_mean_kernel, arg != nullptr: max) that also emits the relu'd bf16 operand of the next fc_0; 4 consecutive
// features per thread (H % 4 == 0)
__global__ void view_mean_bf16_kernel(const float* __restrict__ x, float* __restrict__ y, __nv_bfloat16* __restrict__ y16,
                                      uint8_t* __restrict__ arg, int SB, int NS, int P, int H) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int H4 = H >> 2;
  if (i >= (long long)SB * P * H4) return;
  const int h4 = (int)(i % H4);
  const long long sp = i / H4;
  const int p = (int)(sp % P), s = (int)(sp / P);
  float4 m;
  if (arg) {
    m = __ldg(reinterpret_cast<const float4*>(x + ((long long)s * NS * P + p) * H) + h4);
    uchar4 win = make_uchar4(0, 0, 0, 0);
    for (int v = 1; v < NS; ++v) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(x + (((long long)s * NS + v) * P + p) * H) + h4);
      if (a.x > m.x) { m.x = a.x; win.x = (unsigned char)v; }
      if (a.y > m.y) { m.y = a.y; win.y = (unsigned char)v; }
      if (a.z > m.z) { m.z = a.z; win.z = (unsigned char)v; }
      if (a.w > m.w) { m.w = a.w; win.w = (unsigned char)v; }
    }
    reinterpret_cast<uchar4*>(arg)[i] = win;
  } else {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int v = 0; v < NS; ++v) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(x + (((long long)s * NS + v) * P + p) * H) + h4);
      acc.x += a.x; acc.y += a.y; acc.z += a.z; acc.w += a.w;
    }
    const float n = (float)NS;
    m = make_float4(acc.x / n, acc.y / n, acc.z / n, acc.w / n);
  }
  reinterpret_cast<float4*>(y)[i] = m;
  __nv_bfloat162* o = reinterpret_cast<__nv_bfloat162*>(y16) + i * 2;
  o[0] = __floats2bfloat162_rn(fmaxf(m.x, 0.f), fmaxf(m.y, 0.f));
  o[1] = __floats2bfloat162_rn(fmaxf(m.z, 0.f), fmaxf(m.w, 0.f));
}
__global__ void view_mean_bwd_bf16_kernel(const float* __restrict__ dy, float* __restrict__ dx, __nv_bfloat16* __restrict__ dx16,
                                          const uint8_t* __restrict__ arg, int SB, int NS, int P, int H) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int H4 = H >> 2;
  if (i >= (long long)SB * NS * P * H4) return;
  const int h4 = (int)(i % H4);
  const long long svp = i / H4;
  const int p = (int)(svp % P);
  const int s = (int)(svp / P / NS);
  const float4 a = __ldg(reinterpret_cast<const float4*>(dy + ((long long)s * P + p) * H) + h4);
  float4 g;
  if (arg) {
    const int v = (int)(svp / P - (long long)s * NS);
    const uchar4 w = reinterpret_cast<const uchar4*>(arg)[((long long)s * P + p) * H4 + h4];
    g = make_float4(w.x == v ? a.x : 0.f, w.y == v ? a.y : 0.f, w.z == v ? a.z : 0.f, w.w == v ? a.w : 0.f);
  } else {
    const float n = (float)NS;
    g = make_float4(a.x / n, a.y / n, a.z / n, a.w / n);
  }
  reinterpret_cast<float4*>(dx)[i] = g;
  __nv_bfloat162* o = reinterpret_cast<__nv_bfloat162*>(dx16) + i * 2;
  o[0] = __floats2bfloat162_rn(g.x, g.y);
  o[1] = __floats2bfloat162_rn(g.z, g.w);
}
__global__ void colsum_bf16_kernel(const __nv_bfloat16* __restrict__ dY, float* __restrict__ db, long long M, int N, int rows_per_block) {
  const long long r0 = (long long)blockIdx.x * rows_per_block;
  const long long r1 = r0 + rows_per_block < M ? r0 + rows_per_block : M;
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
    float acc = 0.f;
    for (long long r = r0; r < r1; ++r) acc += __bfloat162float(dY[r * N + j]);
    atomicAdd(db + j, acc);
  }
}
// z-features (rows, d_in) fp32 -> (rows, 64) bf16, zero padded: the K = 64 operand of lin_in
__global__ void zf_pad_bf16_kernel(const float* __restrict__ zf, __nv_bfloat16* __restrict__ out, long long rows, int d_in) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * 64) return;
  const long long r = i >> 6;
  const int c = (int)(i & 63);
  out[i] = __float2bfloat16_rn(c < d_in ? zf[r * d_in + c] : 0.f);
}

// lin_out (H -> d_out <= 32) on relu(x): sigmoid(rgb) / relu(sigma) (resnetfc.py:185, models.py:312-317), or the raw values
// (YOLO head, models.py:309-310).  T = float (the fp32 tape holds x) or __nv_bfloat16 (the bf16 tape holds relu(x)).
__device__ __forceinline__ float ld_act(const float* p) { return *p; }
__device__ __forceinline__ float ld_act(const __nv_bfloat16* p) { return __bfloat162float(*p); }
template <typename T>
__global__ void lin_out_fwd_kernel(const T* __restrict__ x, const float* __restrict__ W, const float* __restrict__ bias,
                                   float* __restrict__ out, long long rows, int H, int d_out, int raw) {
  const int lane = threadIdx.x & 31;
  const long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= rows) return;
  for (int o = 0; o < d_out; ++o) {
    float acc = 0.f;
    for (int k = lane; k < H; k += 32) acc = fmaf(fmaxf(ld_act(x + row * H + k), 0.f), W[o * H + k], acc);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
    if (lane == 0) {
      float v = acc + bias[o];
      out[row * d_out + o] = raw ? v : ((o < 3) ? 1.0f / (1.0f + expf(-v)) : fmaxf(v, 0.f));
    }
  }
}
// One warp per point: d_raw = d_out * act'(out); dx = (d_raw W) * (x > 0); per-block partial dW / db -> atomics.
// dx (fp32) and, optionally, a bf16 copy dx16 (operand of the tcgen05 GEMMs).
template <typename T>
__global__ void __launch_bounds__(256)
lin_out_bwd_kernel(const T* __restrict__ x, const float* __restrict__ W, const float* __restrict__ out,
                   const float* __restrict__ d_out_act, float* __restrict__ dx, __nv_bfloat16* __restrict__ dx16,
                   float* __restrict__ dW, float* __restrict__ db, float* __restrict__ dx_colsum, long long rows, int H, int d_out,
                   int rows_per_warp, int raw) {
  extern __shared__ float sm[];                 // [d_out][H] partial dW of this block, [d_out] partial db, [H] partial column sums of dx
  float* sW = sm;
  float* sb = sm + d_out * H;
  float* sx = sb + d_out;
  for (int i = threadIdx.x; i < d_out * H + d_out + H; i += blockDim.x) sm[i] = 0.f;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  for (int rr = 0; rr < rows_per_warp; ++rr) {
    const long long row = warp * rows_per_warp + rr;
    if (row >= rows) break;
    float draw[32];
    for (int o = 0; o < d_out; ++o) {
      const float y = out[row * d_out + o], gy = d_out_act[row * d_out + o];
      draw[o] = raw ? gy : ((o < 3) ? gy * y * (1.0f - y) : (y > 0.f ? gy : 0.f));     // sigmoid' = y (1 - y); relu' = [y > 0]
    }
    if (lane == 0) for (int o = 0; o < d_out; ++o) atomicAdd(sb + o, draw[o]);
    for (int k = lane; k < H; k += 32) {
      const float xv = ld_act(x + row * H + k);
      const float r = fmaxf(xv, 0.f);
      float g = 0.f;
      for (int o = 0; o < d_out; ++o) {
        g = fmaf(draw[o], W[o * H + k], g);
        atomicAdd(sW + o * H + k, draw[o] * r);
      }
      g = xv > 0.f ? g : 0.f;
      dx[row * H + k] = g;
      if (dx16) dx16[row * H + k] = __float2bfloat16_rn(g);
      if (dx_colsum) atomicAdd(sx + k, g);
    }
  }
  __syncthreads();
  if (dx_colsum) for (int i = threadIdx.x; i < H; i += blockDim.x) atomicAdd(dx_colsum + i, sx[i]);
  for (int i = threadIdx.x; i < d_out * H; i += blockDim.x) atomicAdd(dW + i, sW[i]);
  for (int i = threadIdx.x; i < d_out; i += blockDim.x) atomicAdd(db + i, sb[i]);
}

// Backward of projection + bilinear gather + positional encoding for one (object, view, point) row per warp.
//   dlat (rows, C), dzf (rows, d_in)  ->  d_feat (fp32 channels-last maps, atomics; may be null),
//   d_xyz (SB*P, 3) (mode 0) or d_z (SB*B*K) (mode 1: x = o + z d  =>  dz = dx . d), atomics; may be null.
__global__ void __launch_bounds__(256)
gather_encode_bwd_kernel(pnr_scene sc, pnr_points q, const float* __restrict__ dlat, const float* __restrict__ dzf,
                         float* __restrict__ d_feat, float* __restrict__ d_xyz, float* __restrict__ d_z, int num_freqs,
                         float freq_factor, long long n_rows) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  const int NS = sc.NS, P = q.P, C = sc.C;
  const int d_in = 6 * num_freqs + 6;
  const bool want_x = d_xyz || d_z;
  for (long long row = warp; row < n_rows; row += n_warps) {
    const int view = (int)(row / P);
    const int p = (int)(row - (long long)view * P);
    const int s = view / NS;
    const long long pidx = (long long)s * P + p;
    float px, py, pz, vx, vy, vz;
    fetch_point(q, pidx, px, py, pz, vx, vy, vz);
    const Projection pr = project_point(sc, view, px, py, pz, vx, vy, vz);
    const Taps t = make_taps(pr.ix, pr.iy, sc.Hl, sc.Wl, C);
    const size_t map_off = (size_t)view * sc.Hl * sc.Wl * C;
    const float* fm = (const float*)sc.feat + map_off;
    float gix = 0.f, giy = 0.f;
    const float fx0 = floorf(pr.ix), fy0 = floorf(pr.iy);
    const float ax = pr.ix - fx0, ay = pr.iy - fy0;          // (ix - x0), (iy - y0); (x1 - ix) = 1 - ax
    for (int c0 = lane * 4; c0 < C; c0 += 128) {
      const float4 g = *reinterpret_cast<const float4*>(dlat + row * C + c0);
      float4 f[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        f[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (t.off[k] >= 0) {
          if (want_x) f[k] = __ldg(reinterpret_cast<const float4*>(fm + t.off[k] + c0));
          if (d_feat) {
            float* dst = d_feat + map_off + t.off[k] + c0;        // 16-byte aligned: one vector reduction instead of four scalar ones
            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "f"(t.w[k] * g.x), "f"(t.w[k] * g.y), "f"(t.w[k] * g.z),
                         "f"(t.w[k] * g.w)
                         : "memory");
          }
        }
      }
      if (want_x) {
        // d/dix = (ne - nw)(y1 - iy) + (se - sw)(iy - y0);  d/diy = (sw - nw)(x1 - ix) + (se - ne)(ix - x0)
        const float bx = 1.0f - ax, by = 1.0f - ay;
#define PNR_ACC(comp)                                                                              \
        gix += g.comp * ((f[1].comp - f[0].comp) * by + (f[3].comp - f[2].comp) * ay);             \
        giy += g.comp * ((f[2].comp - f[0].comp) * bx + (f[3].comp - f[1].comp) * ax);
        PNR_ACC(x) PNR_ACC(y) PNR_ACC(z) PNR_ACC(w)
#undef PNR_ACC
      }
    }
    if (!want_x) continue;
    // positional encoding: element j of the z-feature row depends on coordinate d = (j - 3) % 3 of R x
    float gx[3] = {0.f, 0.f, 0.f};
    const int n_pe = 3 + 6 * num_freqs;
    for (int j = lane; j < n_pe && j < d_in; j += 32) {
      const float gj = dzf[row * d_in + j];
      if (j < 3) { gx[j] += gj; continue; }
      const int qq = j - 3, k = qq / 6, r = qq - k * 6, d = r % 3;
      const float xv = d == 0 ? pr.xr : (d == 1 ? pr.yr : pr.zr);
      const float f = freq_factor * (float)(1 << k);
      const float ph = r >= 3 ? 1.57079637050628662109375f : 0.0f;
      const float dv = gj * f * cosf(fmaf(xv, f, ph));           // d/dx sin(f x + ph)
      gx[d] += dv;
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      gix += __shfl_xor_sync(0xffffffffu, gix, d);
      giy += __shfl_xor_sync(0xffffffffu, giy, d);
      gx[0] += __shfl_xor_sync(0xffffffffu, gx[0], d);
      gx[1] += __shfl_xor_sync(0xffffffffu, gx[1], d);
      gx[2] += __shfl_xor_sync(0xffffffffu, gx[2], d);
    }
    if (lane == 0) {
      const float* M = sc.poses + (size_t)view * 12;
      const float xc = pr.xr + M[3], yc = pr.yr + M[7], zc = pr.zr + M[11];
      const float fxv = sc.focal[view * 2 + 0], fyv = sc.focal[view * 2 + 1];
      // ix = u * (lat_scale_x / image_w) * 0.5 * (Wl - 1),  u = -xc / zc * fx + cx
      const float du = gix * (sc.lat_scale_x / sc.image_w) * 0.5f * (float)(sc.Wl - 1);
      const float dv = giy * (sc.lat_scale_y / sc.image_h) * 0.5f * (float)(sc.Hl - 1);
      const float inv_z = 1.0f / zc;
      float gc[3];
      gc[0] = -fxv * inv_z * du;
      gc[1] = -fyv * inv_z * dv;
      gc[2] = (xc * fxv * du + yc * fyv * dv) * inv_z * inv_z;
      if (!isfinite(gc[0]) || !isfinite(gc[1]) || !isfinite(gc[2])) gc[0] = gc[1] = gc[2] = 0.f;   // point on the camera plane
      const float r0 = gx[0] + gc[0], r1 = gx[1] + gc[1], r2 = gx[2] + gc[2];
      // x_rot = R x  =>  dx = R^T d(x_rot)
      const float wx = M[0] * r0 + M[4] * r1 + M[8] * r2;
      const float wy = M[1] * r0 + M[5] * r1 + M[9] * r2;
      const float wz = M[2] * r0 + M[6] * r1 + M[10] * r2;
      if (d_xyz) { atomicAdd(d_xyz + pidx * 3 + 0, wx); atomicAdd(d_xyz + pidx * 3 + 1, wy); atomicAdd(d_xyz + pidx * 3 + 2, wz); }
      if (d_z) atomicAdd(d_z + pidx, wx * vx + wy * vy + wz * vz);
    }
  }
}

// fp32 (rows, H) -> bf16 slice of a wider channels-last map
__global__ void store_bf16_slice_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, long long rows, int H,
                                        int ld_dst, int c0) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * H) return;
  const long long r = i / H;
  const int c = (int)(i - r * H);
  dst[r * ld_dst + c0 + c] = __float2bfloat16_rn(src[i]);
}

struct Tape {
  float *lat, *zf;
  float* X[9];      // rows x H: input of pre-combine block b (b < CL); X[CL] = output of the last pre-combine block
  float* NET[8];    // rows x H: fc_0 output of pre-combine block b
  float* XM[9];     // pts x H : input of post-combine block b (b >= CL); XM[n_blocks] = input of lin_out
  float* NETM[8];   // pts x H
  uint8_t* ARG;     // pts x H: winning view of the max pooling (combine_type max only)
  size_t floats;
};
// combine_type max with more than one view to pool: the tape records the winning view of every (point, feature)
static bool pool_max(const pnr_scene* sc, const pnr_mlp_params* mp) {
  return mp->combine_type == PNR_COMBINE_MAX && sc->NS > 1 && mp->combine_layer < mp->n_blocks;
}
static Tape carve_tape(float* base, long long rows, long long pts, int C, int d_in, int H, int nb, int CL, bool vmax) {
  Tape t = {};
  float* p = base;
  t.lat = p; p += rows * C;
  t.zf = p; p += rows * d_in;
  for (int b = 0; b <= CL; ++b) { t.X[b] = p; p += rows * H; }
  for (int b = 0; b < CL; ++b) { t.NET[b] = p; p += rows * H; }
  for (int b = CL; b <= nb; ++b) { t.XM[b] = p; p += pts * H; }
  for (int b = CL; b < nb; ++b) { t.NETM[b] = p; p += pts * H; }
  if (vmax) { t.ARG = reinterpret_cast<uint8_t*>(p); p += (pts * H + 3) / 4; }
  t.floats = (size_t)(p - base);
  return t;
}

static int check_train(const pnr_scene* sc, const pnr_points* q, const pnr_mlp_params* mp, int num_freqs, const char* who) {
  int rc = validate_scene_points(sc, q, who);
  if (rc) return rc;
  PNR_REQUIRE(mp, PNR_ERR_ARG, "%s: null params", who);
  PNR_REQUIRE(sc->feat_fp32, PNR_ERR_ARG, "%s: the training path reads fp32 channels-last feature maps", who);
  PNR_REQUIRE((sc->flags & PNR_SCENE_PROJECTED) == 0, PNR_ERR_UNSUPPORTED, "%s: pre-projected feature maps (PNR_SCENE_PROJECTED) have no training path: the projection depends on the weights being trained", who);
  PNR_REQUIRE(!((sc->flags & PNR_SCENE_TRAIN_TF32) && (sc->flags & PNR_SCENE_TRAIN_BF16)), PNR_ERR_ARG, "%s: choose one of PNR_SCENE_TRAIN_TF32 / PNR_SCENE_TRAIN_BF16", who);
  g_use_tf32 = (sc->flags & PNR_SCENE_TRAIN_TF32) ? 1 : 0;
  if (sc->flags & PNR_SCENE_TRAIN_BF16) {
    PNR_REQUIRE(hidden_width_supported(mp->d_hidden) && sc->C % 64 == 0, PNR_ERR_UNSUPPORTED,
                "%s: the tcgen05 training path needs d_hidden in " PNR_HIDDEN_WIDTHS " and C a multiple of 64 (got %d, %d)", who,
                mp->d_hidden, sc->C);
    PNR_REQUIRE(mp->d_in <= 64, PNR_ERR_UNSUPPORTED, "%s: d_in=%d > 64", who, mp->d_in);
  }
  PNR_REQUIRE(sc->C % 4 == 0, PNR_ERR_UNSUPPORTED, "%s: C=%d must be a multiple of 4", who, sc->C);
  PNR_REQUIRE(mp->d_latent == sc->C, PNR_ERR_ARG, "%s: d_latent=%d but maps have C=%d", who, mp->d_latent, sc->C);
  PNR_REQUIRE(mp->d_in == 6 * num_freqs + 6, PNR_ERR_ARG, "%s: d_in/num_freqs mismatch", who);
  PNR_REQUIRE(mp->n_blocks >= 1 && mp->n_blocks <= 8, PNR_ERR_UNSUPPORTED, "%s: n_blocks=%d", who, mp->n_blocks);
  PNR_REQUIRE(mp->combine_layer >= 1 && mp->combine_layer <= mp->n_blocks, PNR_ERR_ARG, "%s: combine_layer=%d", who, mp->combine_layer);
  PNR_REQUIRE(mp->combine_layer < mp->n_blocks || sc->NS == 1, PNR_ERR_UNSUPPORTED, "%s: combine_layer >= n_blocks needs NS=1", who);
  PNR_REQUIRE(mp->combine_type == PNR_COMBINE_AVERAGE || mp->combine_type == PNR_COMBINE_MAX, PNR_ERR_ARG, "%s: combine_type=%d", who,
              mp->combine_type);
  PNR_REQUIRE(mp->d_out >= 1 && mp->d_out <= 32, PNR_ERR_UNSUPPORTED, "%s: d_out=%d", who, mp->d_out);
  PNR_REQUIRE((long long)sc->SB * sc->NS * q->P < (1LL << 31), PNR_ERR_ARG, "%s: too many rows per call", who);
  return PNR_OK;
}

// ======================================================================================================================
// tcgen05 training path (PNR_SCENE_TRAIN_BF16): bf16 operands on the tape, fp32 accumulation in TMEM (train_umma.cu).
// The tape keeps what the backward pass needs and nothing else: the relu'd bf16 OPERAND of every layer (the weight gradient's
// second factor; its sign pattern is the relu mask), the gathered latent and z-feature rows -- 1 KiB per row and layer instead of
// the fp32 path's 2 x 2 KiB.  The fp32 residual stream x lives in a scratch buffer that the next block overwrites.
struct TapeB {
  __nv_bfloat16 *lat, *zf;          // rows x C, rows x 64
  __nv_bfloat16* RX[9];             // rows x H: relu(x_b), operand of fc_0 of pre-combine block b
  __nv_bfloat16* RN[8];             // rows x H: relu(fc_0 output) of pre-combine block b, operand of fc_1
  __nv_bfloat16* RXM[9];            // pts x H: same for the post-combine blocks; RXM[n_blocks] = operand of lin_out
  __nv_bfloat16* RNM[8];
  float *x, *xm;                    // rows x H, pts x H fp32 residual stream (scratch of the forward pass)
  uint8_t* arg;                     // pts x H winning view of the max pooling (combine_type max only)
  uint8_t* wpack;                   // forward packed weights
  size_t bytes;
};
struct WPack { size_t lin_in, linz[8], fc0[8], fc1[8], total; };
static WPack wpack_layout(int C, int d_in_pad, int H, int nb, int CL, bool transposed) {
  // forward: out = H, in = K.  transposed (input gradients): out = K (lin_z: C, lin_in: d_in_pad), in = H.
  WPack w = {};
  size_t off = 0;
  auto take = [&](int n_out, int n_in) { size_t o = off; off += (tg::packed_rowgemm_bytes(n_out, n_in) + 1023) & ~(size_t)1023; return o; };
  w.lin_in = transposed ? take(d_in_pad, H) : take(H, d_in_pad);
  for (int b = 0; b < CL; ++b) w.linz[b] = transposed ? take(C, H) : take(H, C);
  for (int b = 0; b < nb; ++b) { w.fc0[b] = take(H, H); w.fc1[b] = take(H, H); }
  w.total = off;
  return w;
}
static TapeB carve_tape_b(uint8_t* base, long long rows, long long pts, int C, int H, int nb, int CL, bool vmax) {
  TapeB t = {};
  size_t off = 0;
  auto take = [&](size_t bytes) { uint8_t* p = base ? base + off : nullptr; off += (bytes + 1023) & ~(size_t)1023; return p; };
  t.lat = (__nv_bfloat16*)take((size_t)rows * C * 2);
  t.zf = (__nv_bfloat16*)take((size_t)rows * 64 * 2);
  for (int b = 0; b < CL; ++b) t.RX[b] = (__nv_bfloat16*)take((size_t)rows * H * 2);
  for (int b = 0; b < CL; ++b) t.RN[b] = (__nv_bfloat16*)take((size_t)rows * H * 2);
  for (int b = CL; b <= nb; ++b) t.RXM[b] = (__nv_bfloat16*)take((size_t)pts * H * 2);
  for (int b = CL; b < nb; ++b) t.RNM[b] = (__nv_bfloat16*)take((size_t)pts * H * 2);
  t.x = (float*)take((size_t)rows * H * 4);
  t.xm = (float*)take((size_t)pts * H * 4);
  if (vmax) t.arg = take((size_t)pts * H);
  t.wpack = take(wpack_layout(C, 64, H, nb, CL, false).total);
  t.bytes = off + 1024;
  return t;
}
static uint8_t* align1k(void* p) { return (uint8_t*)(((uintptr_t)p + 1023) & ~(uintptr_t)1023); }

static int pack_all(const pnr_mlp_params* mp, int C, bool transposed, uint8_t* dst, const WPack& w, cudaStream_t st, int* launches) {
  const int H = mp->d_hidden, nb = mp->n_blocks, CL = mp->combine_layer;
  tg::PackJob jobs[tg::kMaxPackJobs];
  int n = 0;
  auto add = [&](const float* W, int rows, int cols, size_t off) { jobs[n++] = tg::PackJob{W, rows, cols, cols, dst + off}; };
  add(mp->lin_in_w, H, mp->d_in, w.lin_in);
  for (int b = 0; b < CL; ++b) add(mp->linz_w[b], H, C, w.linz[b]);
  for (int b = 0; b < nb; ++b) { add(mp->fc0_w[b], H, H, w.fc0[b]); add(mp->fc1_w[b], H, H, w.fc1[b]); }
  int rc = tg::pack_rowgemm_many(jobs, n, transposed ? 1 : 0, st);
  if (rc) return rc;
  ++*launches;
  return PNR_OK;
}

// y = epilogue(A0 W0^T [+ A1 W1^T]) with the common argument patterns of the chain
static int rg(const __nv_bfloat16* A0, long long lda0, int K0, const void* W0, const __nv_bfloat16* A1, long long lda1, int K1, const void* W1,
              tg::RowGemmArgs g, cudaStream_t st, int* launches) {
  tg::RowGemmSrc s0 = {A0, lda0, K0, W0}, s1 = {A1, lda1, K1, W1};
  int rc = tg::rowgemm(s0, A1 ? &s1 : nullptr, g, st);
  if (rc) return rc;
  ++*launches;
  return PNR_OK;
}

static int forward_bf16(const pnr_scene* sc, const pnr_points* q, const pnr_mlp_params* mp, float* out, void* tape, int num_freqs,
                        float freq_factor, cudaStream_t st) {
  const long long rows = (long long)sc->SB * sc->NS * q->P, pts = (long long)sc->SB * q->P;
  const int H = mp->d_hidden, C = sc->C, d_in = mp->d_in, nb = mp->n_blocks, CL = mp->combine_layer;
  const TapeB t = carve_tape_b(align1k(tape), rows, pts, C, H, nb, CL, pool_max(sc, mp));
  const WPack w = wpack_layout(C, 64, H, nb, CL, false);
  int launches = 0, rc;
  // gather: latent rows straight to bf16; z-features via an fp32 scratch (the x buffer, not yet in use) then padded to K = 64
  float* zf32 = t.x;
  rc = pnr_gather_encode(sc, q, t.lat, zf32, 0, num_freqs, freq_factor, (void*)st);
  if (rc) return rc;
  ++launches;
  zf_pad_bf16_kernel<<<(unsigned)((rows * 64 + 255) / 256), 256, 0, st>>>(zf32, t.zf, rows, d_in);
  PNR_CHECK_LAUNCH("bwd::zf_pad_bf16_kernel");
  ++launches;
  if ((rc = pack_all(mp, C, false, t.wpack, w, st, &launches))) return rc;
  tg::RowGemmArgs g;
  auto base = [&](long long M) { tg::RowGemmArgs a = {}; a.M = M; a.n_valid = H; return a; };
  // x_0 = lin_in(zf) + lin_z[0](z)                                             resnetfc.py:149,176-180
  g = base(rows); g.bias = mp->lin_in_b; g.bias2 = mp->linz_b[0]; g.out_f32 = t.x; g.ld_f32 = H; g.out_bf16 = t.RX[0]; g.ld_bf16 = H; g.relu_out = 1;
  if ((rc = rg(t.zf, 64, 64, t.wpack + w.lin_in, t.lat, C, C, t.wpack + w.linz[0], g, st, &launches))) return rc;
  for (int b = 0; b < CL; ++b) {
    g = base(rows); g.bias = mp->fc0_b[b]; g.out_bf16 = t.RN[b]; g.ld_bf16 = H; g.relu_out = 1;                       // net = fc_0(relu(x))
    if ((rc = rg(t.RX[b], H, H, t.wpack + w.fc0[b], nullptr, 0, 0, nullptr, g, st, &launches))) return rc;
    const bool more = b + 1 < CL;                                                                                      // x += fc_1(relu(net)) [+ lin_z[b+1](z)]
    g = base(rows); g.bias = mp->fc1_b[b]; g.bias2 = more ? mp->linz_b[b + 1] : nullptr; g.res_in = t.x; g.ld_res = H; g.out_f32 = t.x; g.ld_f32 = H;
    if (more) { g.out_bf16 = t.RX[b + 1]; g.ld_bf16 = H; g.relu_out = 1; }
    if ((rc = rg(t.RN[b], H, H, t.wpack + w.fc1[b], more ? t.lat : nullptr, C, C, more ? t.wpack + w.linz[b + 1] : nullptr, g, st, &launches))) return rc;
  }
  {
    const long long n = pts * H / 4;
    view_mean_bf16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(t.x, t.xm, t.RXM[CL], t.arg, sc->SB, sc->NS, q->P, H);  // util.py:489-499
    PNR_CHECK_LAUNCH("bwd::view_mean_bf16_kernel");
    ++launches;
  }
  for (int b = CL; b < nb; ++b) {
    g = base(pts); g.bias = mp->fc0_b[b]; g.out_bf16 = t.RNM[b]; g.ld_bf16 = H; g.relu_out = 1;
    if ((rc = rg(t.RXM[b], H, H, t.wpack + w.fc0[b], nullptr, 0, 0, nullptr, g, st, &launches))) return rc;
    g = base(pts); g.bias = mp->fc1_b[b]; g.res_in = t.xm; g.ld_res = H; g.out_f32 = t.xm; g.ld_f32 = H; g.out_bf16 = t.RXM[b + 1]; g.ld_bf16 = H; g.relu_out = 1;
    if ((rc = rg(t.RNM[b], H, H, t.wpack + w.fc1[b], nullptr, 0, 0, nullptr, g, st, &launches))) return rc;
  }
  lin_out_fwd_kernel<__nv_bfloat16><<<(unsigned)((pts * 32 + 255) / 256), 256, 0, st>>>(t.RXM[nb], mp->lin_out_w, mp->lin_out_b, out, pts, H, mp->d_out,
                                                                                         (sc->flags & PNR_SCENE_RAW_OUTPUT) ? 1 : 0);
  PNR_CHECK_LAUNCH("bwd::lin_out_fwd_kernel");
  ++launches;
  reset_launch_count();
  count_launch(launches);
  return PNR_OK;
}

struct BwdWsB { float *dx, *dxm, *dlat, *dzf; __nv_bfloat16 *dx16, *dn16; uint8_t* wpack; size_t bytes; };
static BwdWsB carve_bwd_b(uint8_t* base, long long rows, long long pts, int C, int d_in, int H, int nb, int CL) {
  BwdWsB b = {};
  size_t off = 0;
  auto take = [&](size_t bytes) { uint8_t* p = base ? base + off : nullptr; off += (bytes + 1023) & ~(size_t)1023; return p; };
  b.dx = (float*)take((size_t)rows * H * 4);
  b.dxm = (float*)take((size_t)pts * H * 4);
  b.dlat = (float*)take((size_t)rows * C * 4);
  b.dzf = (float*)take((size_t)rows * d_in * 4);
  b.dx16 = (__nv_bfloat16*)take((size_t)rows * H * 2);
  b.dn16 = (__nv_bfloat16*)take((size_t)rows * H * 2);
  b.wpack = take(wpack_layout(C, 64, H, nb, CL, true).total);
  b.bytes = off + 1024;
  return b;
}

static int backward_bf16(const pnr_scene* sc, const pnr_points* q, const pnr_mlp_params* mp, const void* tape, const float* out,
                         const float* d_out, const pnr_mlp_grads* gr, float* d_feat, float* d_xyz, float* d_z, void* workspace,
                         int num_freqs, float freq_factor, cudaStream_t st) {
  const long long rows = (long long)sc->SB * sc->NS * q->P, pts = (long long)sc->SB * q->P;
  const int H = mp->d_hidden, C = sc->C, d_in = mp->d_in, nb = mp->n_blocks, CL = mp->combine_layer, NS = sc->NS;
  const TapeB t = carve_tape_b(align1k(const_cast<void*>(tape)), rows, pts, C, H, nb, CL, pool_max(sc, mp));
  const BwdWsB ws = carve_bwd_b(align1k(workspace), rows, pts, C, d_in, H, nb, CL);
  const WPack w = wpack_layout(C, 64, H, nb, CL, true);
  int launches = 0, rc;
  if ((rc = pack_all(mp, C, true, ws.wpack, w, st, &launches))) return rc;
  const int raw = (sc->flags & PNR_SCENE_RAW_OUTPUT) ? 1 : 0;
  {
    const int rpw = 4;
    const long long warps = (pts + rpw - 1) / rpw;
    const size_t smem = (size_t)(mp->d_out * H + mp->d_out + H) * sizeof(float);
    if (smem > 48 * 1024) cudaFuncSetAttribute(lin_out_bwd_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    lin_out_bwd_kernel<__nv_bfloat16><<<(unsigned)((warps * 32 + 255) / 256), 256, smem, st>>>(            // + d fc_1 bias of the last block
        t.RXM[nb], mp->lin_out_w, out, d_out, ws.dxm, ws.dx16, gr->lin_out_w, gr->lin_out_b, gr->fc1_b[nb - 1], pts, H, mp->d_out, rpw, raw);
    PNR_CHECK_LAUNCH("bwd::lin_out_bwd_kernel");
    ++launches;
  }
#define STEP(call) do { rc = (call); if (rc) return rc; ++launches; } while (0)
  // Bias gradients are column sums of the gradient g_b that ENTERS block b from above (= leaves block b + 1 downwards):
  //   d fc_1.bias[b] = colsum(g_{b+1}),  d lin_z.bias[b] = d lin_in.bias (b = 0) = colsum(g_b).
  // Each is accumulated by the epilogue that produces the tensor (lin_out_bwd for g_nb, the dx GEMM of block b for g_b); the
  // view-pooling transpose preserves column sums (mean: sum over views of g / NS; max: all of g goes to one view), so g_CL's sum
  // is taken in the post-combine space.
  // One residual block backwards (resnetfc.py:53-62); dx (fp32 master + bf16 operand copy) is updated in place.
  auto block_bwd = [&](const __nv_bfloat16* RXb, const __nv_bfloat16* RNb, int b, float* dx, long long M) -> int {
    STEP(tg::wgrad(ws.dx16, H, RNb, H, gr->fc1_w[b], H, M, H, H, st));                          // dW1 += dx^T relu(net)
    tg::RowGemmArgs g = {};                                                                      // dnet = (dx W1) * [net > 0]
    g.M = M; g.n_valid = H; g.mask_src = RNb; g.ld_mask = H; g.out_bf16 = ws.dn16; g.ld_bf16 = H; g.colsum_out = gr->fc0_b[b];
    if ((rc = rg(ws.dx16, H, H, ws.wpack + w.fc1[b], nullptr, 0, 0, nullptr, g, st, &launches))) return rc;
    STEP(tg::wgrad(ws.dn16, H, RXb, H, gr->fc0_w[b], H, M, H, H, st));                          // dW0 += dnet^T relu(x)
    g = {};                                                                                      // dx += (dnet W0) * [x > 0]
    g.M = M; g.n_valid = H; g.mask_src = RXb; g.ld_mask = H; g.res_in = dx; g.ld_res = H; g.out_f32 = dx; g.ld_f32 = H; g.out_bf16 = ws.dx16; g.ld_bf16 = H;
    g.colsum_out = b >= 1 ? gr->fc1_b[b - 1] : gr->lin_in_b;
    g.colsum_out2 = b < CL ? gr->linz_b[b] : nullptr;
    if ((rc = rg(ws.dn16, H, H, ws.wpack + w.fc0[b], nullptr, 0, 0, nullptr, g, st, &launches))) return rc;
    return PNR_OK;
  };
  for (int b = nb - 1; b >= CL; --b)
    if ((rc = block_bwd(t.RXM[b], t.RNM[b], b, ws.dxm, pts))) return rc;
  {
    const long long n4 = rows * H / 4;
    view_mean_bwd_bf16_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, st>>>(ws.dxm, ws.dx, ws.dx16, t.arg, sc->SB, NS, q->P, H);
    PNR_CHECK_LAUNCH("bwd::view_mean_bwd_bf16_kernel");
    ++launches;
  }
  for (int b = CL - 1; b >= 0; --b) {
    if ((rc = block_bwd(t.RX[b], t.RN[b], b, ws.dx, rows))) return rc;                           // dx is now g_b, the gradient at x_b + lin_z[b](z)
    STEP(tg::wgrad(ws.dx16, H, t.lat, C, gr->linz_w[b], C, rows, H, C, st));                     // x += lin_z[b](z): resnetfc.py:176-182
    if (d_feat || d_xyz || d_z) {
      tg::RowGemmArgs g = {};                                                                    // dlat (+)= g_b Wz_b
      g.M = rows; g.n_valid = C; g.out_f32 = ws.dlat; g.ld_f32 = C;
      if (b != CL - 1) { g.res_in = ws.dlat; g.ld_res = C; }
      if ((rc = rg(ws.dx16, H, H, ws.wpack + w.linz[b], nullptr, 0, 0, nullptr, g, st, &launches))) return rc;
    }
  }
  STEP(tg::wgrad(ws.dx16, H, t.zf, 64, gr->lin_in_w, d_in, rows, H, d_in, st));
#undef STEP
  if (d_feat || d_xyz || d_z) {
    tg::RowGemmArgs g = {};                                                                      // dzf = dx W_in
    g.M = rows; g.n_valid = d_in; g.out_f32 = ws.dzf; g.ld_f32 = d_in;
    if ((rc = rg(ws.dx16, H, H, ws.wpack + w.lin_in, nullptr, 0, 0, nullptr, g, st, &launches))) return rc;
    long long blocks = (rows + 7) / 8;
    if (blocks > 148LL * 64) blocks = 148LL * 64;
    gather_encode_bwd_kernel<<<(unsigned)blocks, 256, 0, st>>>(*sc, *q, ws.dlat, ws.dzf, d_feat, d_xyz, d_z, num_freqs, freq_factor, rows);
    PNR_CHECK_LAUNCH("bwd::gather_encode_bwd_kernel");
    ++launches;
  }
  reset_launch_count();
  count_launch(launches);
  return PNR_OK;
}

}  // namespace bwd
}  // namespace pnr

using namespace pnr;
using namespace pnr::bwd;

extern "C" size_t pnr_field_tape_bytes(const pnr_scene* sc, const pnr_points* q, const pnr_mlp_params* mp) {
  if (!sc || !q || !mp) return 0;
  const long long rows = (long long)sc->SB * sc->NS * q->P, pts = (long long)sc->SB * q->P;
  const bool vmax = pool_max(sc, mp);
  if (sc->flags & PNR_SCENE_TRAIN_BF16) return carve_tape_b(nullptr, rows, pts, sc->C, mp->d_hidden, mp->n_blocks, mp->combine_layer, vmax).bytes;
  return carve_tape(nullptr, rows, pts, sc->C, mp->d_in, mp->d_hidden, mp->n_blocks, mp->combine_layer, vmax).floats * sizeof(float) + 256;
}

extern "C" int pnr_field_forward_train(const pnr_scene* sc, const pnr_points* q, const pnr_mlp_params* mp, float* out,
                                       void* tape, size_t tape_bytes, int num_freqs, float freq_factor, void* stream) {
  reset_launch_count();
  int rc = check_train(sc, q, mp, num_freqs, "pnr_field_forward_train");
  if (rc) return rc;
  PNR_REQUIRE(out && tape && tape_bytes >= pnr_field_tape_bytes(sc, q, mp), PNR_ERR_ARG, "pnr_field_forward_train: tape too small");
  const long long rows = (long long)sc->SB * sc->NS * q->P, pts = (long long)sc->SB * q->P;
  if (pts == 0) return PNR_OK;
  if (sc->flags & PNR_SCENE_TRAIN_BF16) return forward_bf16(sc, q, mp, out, tape, num_freqs, freq_factor, (cudaStream_t)stream);
  const int H = mp->d_hidden, C = sc->C, d_in = mp->d_in, nb = mp->n_blocks, CL = mp->combine_layer;
  cudaStream_t st = (cudaStream_t)stream;
  const Tape t = carve_tape((float*)tape, rows, pts, C, d_in, H, nb, CL, pool_max(sc, mp));
  int launches = 0;
  rc = pnr_gather_encode(sc, q, t.lat, t.zf, 1, num_freqs, freq_factor, stream);
  if (rc) return rc;
  launches += 1;
#define STEP(call) do { rc = (call); if (rc) return rc; ++launches; } while (0)
  STEP(linear_fwd(t.zf, d_in, mp->lin_in_w, mp->lin_in_b, nullptr, t.X[0], rows, H, d_in, false, st));        // resnetfc.py:149
  for (int b = 0; b < CL; ++b) {
    STEP(linear_fwd(t.lat, C, mp->linz_w[b], mp->linz_b[b], t.X[b], t.X[b], rows, H, C, false, st));          // x += lin_z[b](z)
    STEP(linear_fwd(t.X[b], H, mp->fc0_w[b], mp->fc0_b[b], nullptr, t.NET[b], rows, H, H, true, st));          // resnetfc.py:55
    STEP(linear_fwd(t.NET[b], H, mp->fc1_w[b], mp->fc1_b[b], t.X[b], t.X[b + 1], rows, H, H, true, st));       // resnetfc.py:56,62
  }
  {
    const long long n = pts * H;
    view_mean_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(t.X[CL], t.XM[CL], t.ARG, sc->SB, sc->NS, q->P, H);  // util.py:489-499
    PNR_CHECK_LAUNCH("bwd::view_mean_kernel");
    ++launches;
  }
  for (int b = CL; b < nb; ++b) {
    STEP(linear_fwd(t.XM[b], H, mp->fc0_w[b], mp->fc0_b[b], nullptr, t.NETM[b], pts, H, H, true, st));
    STEP(linear_fwd(t.NETM[b], H, mp->fc1_w[b], mp->fc1_b[b], t.XM[b], t.XM[b + 1], pts, H, H, true, st));
  }
  lin_out_fwd_kernel<float><<<(unsigned)((pts * 32 + 255) / 256), 256, 0, st>>>(t.XM[nb], mp->lin_out_w, mp->lin_out_b, out, pts, H, mp->d_out,
                                                                                (sc->flags & PNR_SCENE_RAW_OUTPUT) ? 1 : 0);
  PNR_CHECK_LAUNCH("bwd::lin_out_fwd_kernel");
  ++launches;
  reset_launch_count();
  count_launch(launches);
  return PNR_OK;
}

extern "C" size_t pnr_field_backward_workspace_bytes(const pnr_scene* sc, const pnr_points* q, const pnr_mlp_params* mp) {
  if (!sc || !q || !mp) return 0;
  const size_t rows = (size_t)sc->SB * sc->NS * q->P;
  if (sc->flags & PNR_SCENE_TRAIN_BF16)
    return carve_bwd_b(nullptr, (long long)rows, (long long)sc->SB * q->P, sc->C, mp->d_in, mp->d_hidden, mp->n_blocks, mp->combine_layer).bytes;
  return sizeof(float) * rows * (2 * (size_t)mp->d_hidden + (size_t)sc->C + (size_t)mp->d_in) + 256;
}

extern "C" int pnr_field_backward(const pnr_scene* sc, const pnr_points* q, const pnr_mlp_params* mp, const void* tape,
                                  const float* out, const float* d_out, const pnr_mlp_grads* gr, float* d_feat,
                                  float* d_xyz, float* d_z, void* workspace, size_t workspace_bytes, int num_freqs,
                                  float freq_factor, void* stream) {
  reset_launch_count();
  int rc = check_train(sc, q, mp, num_freqs, "pnr_field_backward");
  if (rc) return rc;
  PNR_REQUIRE(tape && out && d_out && gr, PNR_ERR_ARG, "pnr_field_backward: null pointer");
  PNR_REQUIRE(workspace && workspace_bytes >= pnr_field_backward_workspace_bytes(sc, q, mp), PNR_ERR_ARG,
              "pnr_field_backward: workspace too small");
  PNR_REQUIRE(!(d_xyz && q->mode != 0) && !(d_z && q->mode != 1), PNR_ERR_ARG,
              "pnr_field_backward: d_xyz goes with explicit points (mode 0), d_z with rays x depths (mode 1)");
  const long long rows = (long long)sc->SB * sc->NS * q->P, pts = (long long)sc->SB * q->P;
  if (pts == 0) return PNR_OK;
  if (sc->flags & PNR_SCENE_TRAIN_BF16)
    return backward_bf16(sc, q, mp, tape, out, d_out, gr, d_feat, d_xyz, d_z, workspace, num_freqs, freq_factor, (cudaStream_t)stream);
  const int H = mp->d_hidden, C = sc->C, d_in = mp->d_in, nb = mp->n_blocks, CL = mp->combine_layer, NS = sc->NS;
  cudaStream_t st = (cudaStream_t)stream;
  const Tape t = carve_tape((float*)const_cast<void*>(tape), rows, pts, C, d_in, H, nb, CL, pool_max(sc, mp));
  float* dA = (float*)workspace;            // current dx
  float* dB = dA + rows * H;                // dnet / scratch
  float* dlat = dB + rows * H;
  float* dzf = dlat + rows * C;
  int launches = 0;
  {
    const int rpw = 4;
    const long long warps = (pts + rpw - 1) / rpw;
    const size_t smem = (size_t)(mp->d_out * H + mp->d_out + H) * sizeof(float);
    if (smem > 48 * 1024) cudaFuncSetAttribute(lin_out_bwd_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    lin_out_bwd_kernel<float><<<(unsigned)((warps * 32 + 255) / 256), 256, smem, st>>>(t.XM[nb], mp->lin_out_w, out, d_out, dA, nullptr,
                                                                                       gr->lin_out_w, gr->lin_out_b, nullptr, pts, H, mp->d_out, rpw,
                                                                                       (sc->flags & PNR_SCENE_RAW_OUTPUT) ? 1 : 0);
    PNR_CHECK_LAUNCH("bwd::lin_out_bwd_kernel");
    ++launches;
  }
  // one residual block backwards (resnetfc.py:53-62): dx is updated in place, dn is scratch
  auto block_bwd = [&](const float* Xb, const float* NETb, int b, float* dx, float* dn, long long M) -> int {
    int r;
    if ((r = linear_bwd_weight(dx, NETb, H, gr->fc1_w[b], M, H, H, true, st))) return r;
    if ((r = colsum(dx, gr->fc1_b[b], M, H, st))) return r;
    if ((r = linear_bwd_input(dx, mp->fc1_w[b], NETb, dn, M, H, H, false, st))) return r;
    if ((r = linear_bwd_weight(dn, Xb, H, gr->fc0_w[b], M, H, H, true, st))) return r;
    if ((r = colsum(dn, gr->fc0_b[b], M, H, st))) return r;
    if ((r = linear_bwd_input(dn, mp->fc0_w[b], Xb, dx, M, H, H, true, st))) return r;
    launches += 6;
    return PNR_OK;
  };
  for (int b = nb - 1; b >= CL; --b)
    if ((rc = block_bwd(t.XM[b], t.NETM[b], b, dA, dB, pts))) return rc;
  {
    const long long n = rows * H;
    view_mean_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dA, dB, t.ARG, sc->SB, NS, q->P, H);
    PNR_CHECK_LAUNCH("bwd::view_mean_bwd_kernel");
    ++launches;
    float* tmp = dA; dA = dB; dB = tmp;
  }
  for (int b = CL - 1; b >= 0; --b) {
    if ((rc = block_bwd(t.X[b], t.NET[b], b, dA, dB, rows))) return rc;
    STEP(linear_bwd_weight(dA, t.lat, C, gr->linz_w[b], rows, H, C, false, st));      // x += lin_z[b](z): resnetfc.py:176-182
    STEP(colsum(dA, gr->linz_b[b], rows, H, st));
    STEP(linear_bwd_input(dA, mp->linz_w[b], nullptr, dlat, rows, H, C, b != CL - 1, st));
  }
  STEP(linear_bwd_weight(dA, t.zf, d_in, gr->lin_in_w, rows, H, d_in, false, st));
  STEP(colsum(dA, gr->lin_in_b, rows, H, st));
  STEP(linear_bwd_input(dA, mp->lin_in_w, nullptr, dzf, rows, H, d_in, false, st));
#undef STEP
  if (d_feat || d_xyz || d_z) {
    long long blocks = (rows + 7) / 8;
    if (blocks > 148LL * 64) blocks = 148LL * 64;
    gather_encode_bwd_kernel<<<(unsigned)blocks, 256, 0, st>>>(*sc, *q, dlat, dzf, d_feat, d_xyz, d_z, num_freqs, freq_factor, rows);
    PNR_CHECK_LAUNCH("bwd::gather_encode_bwd_kernel");
    ++launches;
  }
  reset_launch_count();
  count_launch(launches);
  return PNR_OK;
}

extern "C" int pnr_project_features(const pnr_mlp_params* p, const float* feat, long long n_pixels, void* out,
                                    void* workspace, size_t workspace_bytes, void* stream) {
  reset_launch_count();
  PNR_REQUIRE(p && feat && out && workspace, PNR_ERR_ARG, "pnr_project_features: null pointer");
  PNR_REQUIRE(p->d_latent > 0 && p->d_hidden > 0 && p->combine_layer >= 1 && p->combine_layer <= 8, PNR_ERR_ARG,
              "pnr_project_features: bad MLP dimensions");
  PNR_REQUIRE(n_pixels >= 0 && n_pixels < (1LL << 31), PNR_ERR_ARG, "pnr_project_features: bad pixel count");
  const int H = p->d_hidden, C = p->d_latent, n_linz = p->combine_layer < p->n_blocks ? p->combine_layer : p->n_blocks;
  PNR_REQUIRE(workspace_bytes >= (size_t)n_pixels * H * sizeof(float), PNR_ERR_ARG, "pnr_project_features: workspace too small");
  if (n_pixels == 0) return PNR_OK;
  cudaStream_t st = (cudaStream_t)stream;
  float* tmp = (float*)workspace;
  int launches = 0;
  g_use_tf32 = 0;
  for (int b = 0; b < n_linz; ++b) {
    PNR_REQUIRE(p->linz_w[b], PNR_ERR_ARG, "pnr_project_features: lin_z %d missing", b);
    int rc = linear_fwd(feat, C, p->linz_w[b], nullptr, nullptr, tmp, n_pixels, H, C, false, st);
    if (rc) return rc;
    const long long n = n_pixels * H;
    store_bf16_slice_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(tmp, (__nv_bfloat16*)out, n_pixels, H, n_linz * H, b * H);
    PNR_CHECK_LAUNCH("bwd::store_bf16_slice_kernel");
    launches += 2;
  }
  reset_launch_count();
  count_launch(launches);
  return PNR_OK;
}
