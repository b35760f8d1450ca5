// fp32 check path of the field function (PNR_PREC_FP32): fp32 operands, fp32 accumulate, CUDA cores.
// It exists so that parity can be stated twice (north_star): <=1e-4 against the oracle with fp32
// arithmetic (only the summation order differs), and <=1e-2 for the bf16 tcgen05 production path.
// Structure follows ResnetFC.forward (src/model/resnetfc.py:134-186) layer by layer over a workspace.
#include "pnr_common.cuh"

namespace pnr {

int validate_scene_points(const pnr_scene* sc, const pnr_points* q, const char* who);

// Y[M,N] = (ACCUM ? Y : 0) + relu?(X[M,K]) * W[N,K]^T + bias[N]      (nn.Linear on row-major activations)
constexpr int BM = 128, BN = 128, BK = 8;

template <bool RELU_IN, bool ACCUM>
__global__ void __launch_bounds__(256)
sgemm_nt_kernel(const float* __restrict__ X, const float* __restrict__ W, const float* __restrict__ bias,
                float* __restrict__ Y, int M, int N, int K, int ldx) {
  __shared__ __align__(16) float As[BK][BM];
  __shared__ __align__(16) float Bs[BK][BN];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const long long m0 = (long long)blockIdx.x * BM;
  const int n0 = blockIdx.y * BN;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  const int lrow = tid >> 1;          // 0..127
  const int lk = (tid & 1) * 4;       // 0 or 4
  for (int k0 = 0; k0 < K; k0 += BK) {
    float a[4], b[4];
    const long long gm = m0 + lrow;
    const int gn = n0 + lrow;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int k = k0 + lk + i;
      float av = (gm < M && k < K) ? X[gm * ldx + k] : 0.f;
      if (RELU_IN) av = fmaxf(av, 0.f);
      a[i] = av;
      b[i] = (gn < N && k < K) ? W[(long long)gn * K + k] : 0.f;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) { As[lk + i][lrow] = a[i]; Bs[lk + i][lrow] = b[i]; }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 8]);
      float4 a1 = *reinterpret_cast<const float4*>(&As[k][ty * 8 + 4]);
      float4 b0 = *reinterpret_cast<const float4*>(&Bs[k][tx * 8]);
      float4 b1 = *reinterpret_cast<const float4*>(&Bs[k][tx * 8 + 4]);
      float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    long long gm = m0 + ty * 8 + i;
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int gn = n0 + tx * 8 + j;
      if (gn >= N) continue;
      float v = acc[i][j] + (bias ? bias[gn] : 0.f);
      if (ACCUM) v += Y[gm * N + gn];
      Y[gm * N + gn] = v;
    }
  }
}

// mean (combine_type average) or elementwise max (max) over the NS source views: x (SB, NS, P, H) -> (SB, P, H)   util.py:489-499
__global__ void view_mean_kernel(const float* __restrict__ x, float* __restrict__ y, int SB, int NS, int P, int H, int vmax) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long n = (long long)SB * P * H;
  if (i >= n) return;
  int h = (int)(i % H);
  long long sp = i / H;
  int p = (int)(sp % P);
  int s = (int)(sp / P);
  const float* xv = x + ((long long)s * NS * P + p) * H + h;
  if (vmax) {
    float m = xv[0];
    for (int v = 1; v < NS; ++v) m = fmaxf(m, xv[(long long)v * P * H]);
    y[i] = m;
    return;
  }
  float acc = 0.f;
  for (int v = 0; v < NS; ++v) acc += xv[(long long)v * P * H];
  y[i] = acc / (float)NS;
}

// lin_out (H -> d_out<=32) on relu(x), then sigmoid(rgb) / relu(sigma)       resnetfc.py:185, models.py:312-317
__global__ void lin_out_act_kernel(const float* __restrict__ x, const float* __restrict__ W,
                                   const float* __restrict__ bias, float* __restrict__ out, long long rows, int H,
                                   int d_out, int raw) {
  const int lane = threadIdx.x & 31;
  long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= rows) return;
  for (int o = 0; o < d_out; ++o) {
    float acc = 0.f;
    for (int k = lane; k < H; k += 32) acc = fmaf(fmaxf(x[row * H + k], 0.f), W[o * H + k], acc);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
    if (lane == 0) {
      float v = acc + bias[o];
      if (!raw) v = (o < 3) ? 1.0f / (1.0f + expf(-v)) : fmaxf(v, 0.f);
      out[row * d_out + o] = v;
    }
  }
}

static int gemm(const float* X, int ldx, const float* W, const float* b, float* Y, long long M, int N, int K,
                bool relu_in, bool accum, cudaStream_t st) {
  dim3 grid((unsigned)((M + BM - 1) / BM), (N + BN - 1) / BN);
  if (relu_in && accum) sgemm_nt_kernel<true, true><<<grid, 256, 0, st>>>(X, W, b, Y, (int)M, N, K, ldx);
  else if (relu_in) sgemm_nt_kernel<true, false><<<grid, 256, 0, st>>>(X, W, b, Y, (int)M, N, K, ldx);
  else if (accum) sgemm_nt_kernel<false, true><<<grid, 256, 0, st>>>(X, W, b, Y, (int)M, N, K, ldx);
  else sgemm_nt_kernel<false, false><<<grid, 256, 0, st>>>(X, W, b, Y, (int)M, N, K, ldx);
  PNR_CHECK_LAUNCH("sgemm_nt_kernel");
  return PNR_OK;
}

// ResnetFC.forward over materialised inputs: lat (rows, ld_lat), zf (rows, ld_zf); x,h (rows,H); xm (pts,H).
static int resnetfc_chain(const pnr_mlp_params* mp, const float* lat, int ld_lat, const float* zf, int ld_zf,
                          long long rows, int NS, int P, float* x, float* h, float* xm, float* out, int raw,
                          cudaStream_t st, int* launches) {
  const int H = mp->d_hidden, C = mp->d_latent;
  const long long pts = rows / NS;
  const int SB = (int)(pts / P);
  int rc = gemm(zf, ld_zf, mp->lin_in_w, mp->lin_in_b, x, rows, H, mp->d_in, false, false, st);   // lin_in
  if (rc) return rc;
  ++*launches;
  float* cur = x;
  long long cur_rows = rows;
  for (int b = 0; b < mp->n_blocks; ++b) {
    if (b == mp->combine_layer) {                                                             // view pooling
      long long n = pts * H;
      view_mean_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(x, xm, SB, NS, P, H, mp->combine_type == PNR_COMBINE_MAX);
      PNR_CHECK_LAUNCH("view_mean_kernel");
      cur = xm; cur_rows = pts; ++*launches;
    }
    if (b < mp->combine_layer) {                                                              // x += lin_z[b](z)
      rc = gemm(lat, ld_lat, mp->linz_w[b], mp->linz_b[b], cur, cur_rows, H, C, false, true, st);
      if (rc) return rc;
      ++*launches;
    }
    rc = gemm(cur, H, mp->fc0_w[b], mp->fc0_b[b], h, cur_rows, H, H, true, false, st);        // net = fc_0(relu(x))
    if (rc) return rc;
    rc = gemm(h, H, mp->fc1_w[b], mp->fc1_b[b], cur, cur_rows, H, H, true, true, st);         // x += fc_1(relu(net))
    if (rc) return rc;
    *launches += 2;
  }
  lin_out_act_kernel<<<(unsigned)((cur_rows * 32 + 255) / 256), 256, 0, st>>>(cur, mp->lin_out_w, mp->lin_out_b, out,
                                                                             cur_rows, H, mp->d_out, raw);
  PNR_CHECK_LAUNCH("lin_out_act_kernel");
  ++*launches;
  return PNR_OK;
}

static int check_mlp(const pnr_mlp_params* mp, int NS, const char* who) {
  PNR_REQUIRE(mp, PNR_ERR_ARG, "%s: null params", who);
  PNR_REQUIRE(mp->d_hidden > 0 && mp->d_in > 0 && mp->d_latent > 0, PNR_ERR_ARG, "%s: bad dims", who);
  PNR_REQUIRE(mp->n_blocks >= 1 && mp->n_blocks <= 8, PNR_ERR_UNSUPPORTED, "%s: n_blocks=%d", who, mp->n_blocks);
  PNR_REQUIRE(mp->combine_layer >= 1 && mp->combine_layer <= mp->n_blocks, PNR_ERR_ARG,
              "%s: combine_layer=%d (pass min(combine_layer, n_blocks))", who, mp->combine_layer);
  PNR_REQUIRE(mp->combine_layer < mp->n_blocks || NS == 1, PNR_ERR_UNSUPPORTED,
              "%s: combine_layer >= n_blocks never pools the views; only valid with one source view", who);
  PNR_REQUIRE(mp->combine_type == PNR_COMBINE_AVERAGE || mp->combine_type == PNR_COMBINE_MAX, PNR_ERR_ARG,
              "%s: combine_type=%d", who, mp->combine_type);
  PNR_REQUIRE(mp->d_out >= 1 && mp->d_out <= 64, PNR_ERR_UNSUPPORTED, "%s: d_out=%d", who, mp->d_out);
  return PNR_OK;
}

size_t field_workspace_fp32(const pnr_scene* sc, const pnr_points* q, int d_in, int H) {
  size_t rows = (size_t)sc->SB * sc->NS * q->P, pts = (size_t)sc->SB * q->P;
  return sizeof(float) * (rows * ((size_t)sc->C + d_in + 2 * H) + pts * (size_t)H) + 256;
}

int field_forward_fp32(const pnr_scene* sc, const pnr_points* q, const pnr_mlp_params* mp, float* out, void* ws,
                       size_t ws_bytes, int num_freqs, float freq_factor, int raw, cudaStream_t st) {
  int rc = check_mlp(mp, sc->NS, "field_forward_fp32");
  if (rc) return rc;
  const int H = mp->d_hidden, d_in = mp->d_in, C = sc->C;
  PNR_REQUIRE(d_in == pnr_zfeat_width(sc->flags, num_freqs), PNR_ERR_ARG,
              "field_forward_fp32: d_in=%d but the z-feature layout of the scene flags has width %d at num_freqs=%d", d_in,
              pnr_zfeat_width(sc->flags, num_freqs), num_freqs);
  PNR_REQUIRE(mp->d_latent == C, PNR_ERR_ARG, "field_forward_fp32: d_latent=%d but feature maps have C=%d", mp->d_latent, C);
  PNR_REQUIRE(ws && ws_bytes >= field_workspace_fp32(sc, q, d_in, H), PNR_ERR_ARG, "field_forward_fp32: workspace too small");
  const long long rows = (long long)sc->SB * sc->NS * q->P, pts = (long long)sc->SB * q->P;
  PNR_REQUIRE(rows < (1LL << 31), PNR_ERR_ARG, "field_forward_fp32: too many rows per call (%lld); chunk the points", rows);
  if (pts == 0) return PNR_OK;
  float* lat = (float*)ws;
  float* zf = lat + rows * C;
  float* x = zf + rows * d_in;
  float* h = x + rows * H;
  float* xm = h + rows * H;
  rc = pnr_gather_encode(sc, q, lat, zf, 1, num_freqs, freq_factor, st);
  if (rc) return rc;
  int launches = 1;
  rc = resnetfc_chain(mp, lat, C, zf, d_in, rows, sc->NS, q->P, x, h, xm, out, raw, st, &launches);
  if (rc) return rc;
  reset_launch_count();
  count_launch(launches);
  return PNR_OK;
}

}  // namespace pnr

using namespace pnr;

// ResnetFC.forward as a stand-alone operator (src/model/resnetfc.py:134-186): zx (rows, d_latent + d_in) fp32 with
// rows ordered (object, view, point); returns raw lin_out values (rows/NS, d_out).  fp32 SIMT arithmetic.
extern "C" size_t pnr_resnetfc_workspace_bytes(const pnr_mlp_params* p, long long rows) {
  if (!p || rows < 0) return 0;
  return sizeof(float) * (size_t)rows * 3 * (size_t)p->d_hidden + 256;
}

extern "C" int pnr_resnetfc_forward(const pnr_mlp_params* p, const float* zx, long long rows, int NS, int P,
                                    float* out, void* workspace, size_t workspace_bytes, void* stream) {
  reset_launch_count();
  int rc = check_mlp(p, NS, "pnr_resnetfc_forward");
  if (rc) return rc;
  PNR_REQUIRE(zx && out, PNR_ERR_ARG, "pnr_resnetfc_forward: null pointer");
  PNR_REQUIRE(NS >= 1 && P >= 1 && rows % ((long long)NS * P) == 0, PNR_ERR_ARG,
              "pnr_resnetfc_forward: rows=%lld is not a multiple of NS*P=%d*%d", rows, NS, P);
  PNR_REQUIRE(rows < (1LL << 31), PNR_ERR_ARG, "pnr_resnetfc_forward: too many rows");
  PNR_REQUIRE(workspace && workspace_bytes >= pnr_resnetfc_workspace_bytes(p, rows), PNR_ERR_ARG,
              "pnr_resnetfc_forward: workspace too small");
  if (rows == 0) return PNR_OK;
  const int H = p->d_hidden, ld = p->d_latent + p->d_in;
  float* x = (float*)workspace;
  float* h = x + rows * H;
  float* xm = h + rows * H;
  int launches = 0;
  rc = resnetfc_chain(p, zx, ld, zx + p->d_latent, ld, rows, NS, P, x, h, xm, out, 1, (cudaStream_t)stream, &launches);
  if (rc) return rc;
  reset_launch_count();
  count_launch(launches);
  return PNR_OK;
}
