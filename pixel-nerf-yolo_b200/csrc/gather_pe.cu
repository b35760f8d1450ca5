// F2 (stand-alone form): world->camera transform, perspective projection, 4-tap bilinear gather of the
// channels-last feature maps, and positional encoding (models.py:168-230, encoder.py:79-108,
// code.py:30-42).  One warp per (object, view, point) row: the 32 lanes cover the C channels with
// 16-byte loads, so each tap is one fully coalesced C*2-byte segment.  The fused MLP kernel
// (mlp_umma.cu) uses the same device helpers and writes straight into its shared-memory operand tiles;
// this kernel exists for the fp32 check path and for measuring the gather against HBM/L2 bandwidth.
#include "pnr_common.cuh"

namespace pnr {

// ---- encode-side repack: NCHW fp32 -> NHWC bf16/fp32 (tiled transpose through shared memory) -------
template <typename OutT>
__global__ void pack_features_kernel(const float* __restrict__ src, OutT* __restrict__ dst, int C, int HW) {
  __shared__ float tile[32][33];
  const int n = blockIdx.z;
  const int c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
  const float* s = src + (size_t)n * C * HW;
  OutT* d = dst + (size_t)n * C * HW;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    int c = c0 + r, p = p0 + threadIdx.x;
    tile[r][threadIdx.x] = (c < C && p < HW) ? s[(size_t)c * HW + p] : 0.f;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    int p = p0 + r, c = c0 + threadIdx.x;
    if (p < HW && c < C) {
      float v = tile[threadIdx.x][r];
      if constexpr (sizeof(OutT) == 2) d[(size_t)p * C + c] = __float2bfloat16_rn(v);
      else d[(size_t)p * C + c] = v;
    }
  }
}

// ---- gather + encode -----------------------------------------------------------------------------
template <bool FEAT_FP32, bool OUT_FP32>
__global__ void __launch_bounds__(256)
gather_encode_kernel(pnr_scene sc, pnr_points q, void* __restrict__ latent_out, float* __restrict__ zfeat_out,
                     int num_freqs, float freq_factor, long long n_rows) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
  const int NS = sc.NS, P = q.P, C = sc.C;
  for (long long row = warp; row < n_rows; row += n_warps) {
    // row = (s*NS + v)*P + p   (the reference's (object, view, point) order, models.py:244-246)
    const int view = (int)(row / P);
    const int p = (int)(row - (long long)view * P);
    const int s = view / NS;
    float px, py, pz, vx, vy, vz;
    fetch_point(q, (long long)s * P + p, px, py, pz, vx, vy, vz);
    const Projection pr = project_point(sc, view, px, py, pz, vx, vy, vz);
    if (zfeat_out) {
      const ZfLayout L = zf_layout(sc.flags, num_freqs);
      for (int j = lane; j < L.width; j += 32) zfeat_out[row * L.width + j] = zfeat_value<false>(pr, L, j, num_freqs, freq_factor);
    }
    if (latent_out) {
      const Taps t = make_taps(pr.ix, pr.iy, sc.Hl, sc.Wl, C);
      const size_t map_off = (size_t)view * sc.Hl * sc.Wl * C;
      // 8 channels per lane per step (16 B of bf16 / 32 B of fp32)
      for (int c0 = lane * 8; c0 < C; c0 += 256) {
        float acc[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] = 0.f;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (t.off[k] < 0) continue;
          if constexpr (FEAT_FP32) {
            const float4* f = reinterpret_cast<const float4*>((const float*)sc.feat + map_off + t.off[k] + c0);
            float4 a = __ldg(f), b = __ldg(f + 1);
            acc[0] += t.w[k] * a.x; acc[1] += t.w[k] * a.y; acc[2] += t.w[k] * a.z; acc[3] += t.w[k] * a.w;
            acc[4] += t.w[k] * b.x; acc[5] += t.w[k] * b.y; acc[6] += t.w[k] * b.z; acc[7] += t.w[k] * b.w;
          } else {
            const uint4 raw = __ldg(reinterpret_cast<const uint4*>((const __nv_bfloat16*)sc.feat + map_off + t.off[k] + c0));
            const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              float2 f = __bfloat1622float2(h[i]);
              acc[2 * i] += t.w[k] * f.x;
              acc[2 * i + 1] += t.w[k] * f.y;
            }
          }
        }
        if constexpr (OUT_FP32) {
          float4* o = reinterpret_cast<float4*>((float*)latent_out + row * C + c0);
          o[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
          o[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
        } else {
          uint4 pk;
          __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&pk);
#pragma unroll
          for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(acc[2 * i], acc[2 * i + 1]);
          *reinterpret_cast<uint4*>((__nv_bfloat16*)latent_out + row * C + c0) = pk;
        }
      }
    }
  }
}

// ---- stand-alone operators (API completeness: PositionalEncoding.forward, SpatialEncoder.index) ------------
// code.py:30-42: x (n, d) -> [x, sin(f_k x + phase)] (n, d * (2*num_freqs + include_input))
__global__ void positional_encoding_kernel(const float* __restrict__ x, float* __restrict__ out, long long n, int d,
                                           int num_freqs, float freq_factor, int include_input) {
  const int d_out = d * (2 * num_freqs + (include_input ? 1 : 0));
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * d_out) return;
  long long row = i / d_out;
  int j = (int)(i - row * d_out);
  float v;
  if (include_input && j < d) v = x[row * d + j];
  else {
    int q = j - (include_input ? d : 0);
    int k = q / (2 * d);
    int r = q - k * 2 * d;
    float f = freq_factor * (float)(1 << k);
    float ph = r >= d ? 1.57079637050628662109375f : 0.0f;
    v = sinf(fmaf(x[row * d + (r % d)], f, ph));   // addcmul is a fused multiply-add in ATen
  }
  out[i] = v;
}

// encoder.py:79-108: uv (V, P, 2) pixel coordinates -> (V, C, P) fp32 (the reference's output layout)
template <bool FEAT_FP32>
__global__ void index_kernel(pnr_scene sc, const float* __restrict__ uv, float* __restrict__ out, int P, int uv_views) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int V = sc.SB * sc.NS, C = sc.C;
  if (warp >= (long long)V * P) return;
  const int view = (int)(warp / P), p = (int)(warp - (long long)view * P);
  const float* q = uv + ((size_t)(uv_views == 1 ? 0 : view) * P + p) * 2;     // uv.expand when uv has one view
  float gx = q[0] * __fdiv_rn(sc.lat_scale_x, sc.image_w) - 1.0f;
  float gy = q[1] * __fdiv_rn(sc.lat_scale_y, sc.image_h) - 1.0f;
  float ix = ((gx + 1.0f) * 0.5f) * (float)(sc.Wl - 1);
  float iy = ((gy + 1.0f) * 0.5f) * (float)(sc.Hl - 1);
  const Taps t = make_taps(ix, iy, sc.Hl, sc.Wl, C);
  const size_t map_off = (size_t)view * sc.Hl * sc.Wl * C;
  for (int c = lane; c < C; c += 32) {
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (t.off[k] < 0) continue;
      float f = FEAT_FP32 ? ((const float*)sc.feat)[map_off + t.off[k] + c]
                          : __bfloat162float(((const __nv_bfloat16*)sc.feat)[map_off + t.off[k] + c]);
      acc += t.w[k] * f;
    }
    out[((size_t)view * C + c) * P + p] = acc;
  }
}

}  // namespace pnr

using namespace pnr;

extern "C" int pnr_pack_features(const float* src, void* dst, int N, int C, int H, int W, int to_fp32,
                                 void* stream) {
  reset_launch_count();
  PNR_REQUIRE(src && dst, PNR_ERR_ARG, "pnr_pack_features: null pointer");
  PNR_REQUIRE(N > 0 && C > 0 && H > 0 && W > 0, PNR_ERR_ARG, "pnr_pack_features: bad shape");
  PNR_REQUIRE(N <= 65535, PNR_ERR_ARG, "pnr_pack_features: too many maps");
  int HW = H * W;
  dim3 grid((HW + 31) / 32, (C + 31) / 32, N), block(32, 8);
  if (to_fp32) pack_features_kernel<float><<<grid, block, 0, (cudaStream_t)stream>>>(src, (float*)dst, C, HW);
  else pack_features_kernel<__nv_bfloat16><<<grid, block, 0, (cudaStream_t)stream>>>(src, (__nv_bfloat16*)dst, C, HW);
  PNR_CHECK_LAUNCH("pack_features_kernel");
  return PNR_OK;
}

namespace pnr {
int validate_scene_points(const pnr_scene* sc, const pnr_points* q, const char* who) {
  PNR_REQUIRE(sc && q, PNR_ERR_ARG, "%s: null scene/points", who);
  PNR_REQUIRE(sc->feat && sc->poses && sc->focal && sc->center, PNR_ERR_ARG, "%s: scene has null pointers", who);
  PNR_REQUIRE(sc->SB > 0 && sc->NS > 0 && sc->C > 0 && sc->Hl > 1 && sc->Wl > 1, PNR_ERR_ARG,
              "%s: bad scene shape SB=%d NS=%d C=%d Hl=%d Wl=%d", who, sc->SB, sc->NS, sc->C, sc->Hl, sc->Wl);
  PNR_REQUIRE(sc->C % 8 == 0, PNR_ERR_UNSUPPORTED, "%s: latent channels must be a multiple of 8 (got %d)", who, sc->C);
  PNR_REQUIRE(q->P >= 0, PNR_ERR_ARG, "%s: negative point count", who);
  PNR_REQUIRE(q->total == (long long)sc->SB * q->P, PNR_ERR_ARG,
              "%s: the point buffers hold %lld points but the scene has SB=%d objects x P=%d points (encode() and the ray batch disagree?)",
              who, (long long)q->total, sc->SB, q->P);
  if (q->mode == 0) PNR_REQUIRE(q->xyz || q->P == 0, PNR_ERR_ARG, "%s: xyz is null", who);
  else if (q->mode == 1) {
    PNR_REQUIRE((q->rays && q->z) || q->P == 0, PNR_ERR_ARG, "%s: rays/z is null", who);
    PNR_REQUIRE(q->K > 0 && q->P % q->K == 0, PNR_ERR_ARG, "%s: P=%d is not a multiple of K=%d", who, q->P, q->K);
  } else if (q->mode == 2) {
    PNR_REQUIRE((q->rays && q->steps && q->noise) || q->P == 0, PNR_ERR_ARG, "%s: rays/steps/noise is null", who);
    PNR_REQUIRE(q->K > 0 && q->P % q->K == 0, PNR_ERR_ARG, "%s: P=%d is not a multiple of K=%d", who, q->P, q->K);
  } else PNR_REQUIRE(false, PNR_ERR_ARG, "%s: unknown point mode %d", who, q->mode);
  return PNR_OK;
}
}  // namespace pnr

extern "C" int pnr_gather_encode(const pnr_scene* scene, const pnr_points* pts, void* latent_out,
                                 float* zfeat_out, int out_fp32, int num_freqs, float freq_factor, void* stream) {
  reset_launch_count();
  int rc = validate_scene_points(scene, pts, "pnr_gather_encode");
  if (rc) return rc;
  PNR_REQUIRE(num_freqs >= 0 && num_freqs <= 12, PNR_ERR_ARG, "pnr_gather_encode: num_freqs=%d", num_freqs);
  long long n_rows = (long long)scene->SB * scene->NS * pts->P;
  if (n_rows == 0) return PNR_OK;
  long long blocks = (n_rows + 7) / 8;
  if (blocks > 148LL * 64) blocks = 148LL * 64;   // grid-stride, multiple of the SM count
  cudaStream_t st = (cudaStream_t)stream;
#define LAUNCH(FF, OF) gather_encode_kernel<FF, OF><<<(unsigned)blocks, 256, 0, st>>>(*scene, *pts, latent_out, zfeat_out, num_freqs, freq_factor, n_rows)
  if (scene->feat_fp32) { if (out_fp32) LAUNCH(true, true); else LAUNCH(true, false); }
  else { if (out_fp32) LAUNCH(false, true); else LAUNCH(false, false); }
#undef LAUNCH
  PNR_CHECK_LAUNCH("gather_encode_kernel");
  return PNR_OK;
}

extern "C" int pnr_zfeat_width(int flags, int num_freqs) { return zf_layout(flags, num_freqs).width; }

extern "C" int pnr_positional_encoding(const float* x, float* out, long long n, int d, int num_freqs,
                                       float freq_factor, int include_input, void* stream) {
  reset_launch_count();
  PNR_REQUIRE(x && out, PNR_ERR_ARG, "pnr_positional_encoding: null pointer");
  PNR_REQUIRE(n >= 0 && d > 0 && num_freqs >= 0 && num_freqs <= 24, PNR_ERR_ARG, "pnr_positional_encoding: bad shape");
  if (n == 0) return PNR_OK;
  long long total = n * d * (2 * num_freqs + (include_input ? 1 : 0));
  positional_encoding_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, out, n, d, num_freqs,
                                                                                               freq_factor, include_input);
  PNR_CHECK_LAUNCH("positional_encoding_kernel");
  return PNR_OK;
}

extern "C" int pnr_index_features(const pnr_scene* scene, const float* uv, int uv_views, int P, float* out, void* stream) {
  reset_launch_count();
  PNR_REQUIRE(scene && uv && out, PNR_ERR_ARG, "pnr_index_features: null pointer");
  PNR_REQUIRE(scene->feat && scene->C > 0 && scene->Hl > 1 && scene->Wl > 1 && scene->SB > 0 && scene->NS > 0, PNR_ERR_ARG,
              "pnr_index_features: bad scene");
  const int V = scene->SB * scene->NS;
  PNR_REQUIRE(uv_views == 1 || uv_views == V, PNR_ERR_ARG, "pnr_index_features: uv has %d views, maps have %d", uv_views, V);
  if (P == 0) return PNR_OK;
  long long warps = (long long)V * P;
  unsigned blocks = (unsigned)((warps * 32 + 255) / 256);
  if (scene->feat_fp32) index_kernel<true><<<blocks, 256, 0, (cudaStream_t)stream>>>(*scene, uv, out, P, uv_views);
  else index_kernel<false><<<blocks, 256, 0, (cudaStream_t)stream>>>(*scene, uv, out, P, uv_views);
  PNR_CHECK_LAUNCH("index_kernel");
  return PNR_OK;
}
