// Shared helpers for the pixelnerf_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "../../include/pixelnerf_b200.h"

namespace pnr {

// thread-local error string + launch counter (api.cu)
void set_error(const char* fmt, ...);
void count_launch(int n = 1);
void reset_launch_count();

#define PNR_REQUIRE(cond, code, ...)                 \
  do {                                               \
    if (!(cond)) {                                   \
      ::pnr::set_error(__VA_ARGS__);                 \
      return (code);                                 \
    }                                                \
  } while (0)

#define PNR_CHECK_LAUNCH(what)                                                        \
  do {                                                                                \
    cudaError_t e__ = cudaGetLastError();                                             \
    if (e__ != cudaSuccess) {                                                         \
      ::pnr::set_error("%s: %s", (what), cudaGetErrorString(e__));                    \
      return PNR_ERR_CUDA;                                                            \
    }                                                                                 \
    ::pnr::count_launch();                                                            \
  } while (0)

constexpr int kHidden = 512;    // widest ResnetFC d_hidden the library runs (that of every shipped conf, conf/default*.conf)
// ResnetFC hidden widths the field and training paths run: the multiples of 64 up to kHidden
__host__ __device__ inline bool hidden_width_supported(int d_hidden) {
  return d_hidden >= 64 && d_hidden <= kHidden && d_hidden % 64 == 0;
}
#define PNR_HIDDEN_WIDTHS "64, 128, ..., 512 (multiples of 64)"

// Per-point camera-space quantities for one source view (models.py:168-230, encoder.py:94-98).
struct Projection {
  float xr, yr, zr;   // R x            (positional-encoding input, normalize_z=True)
  float xc, yc, zc;   // R x + t        (camera coordinates, normalize_z=False)
  float dx, dy, dz;   // R d            (view direction in the source view frame)
  float ix, iy;       // feature-map pixel coordinates (align_corners=True un-normalised)
};

// World point -> source view `row` (= s*NS + v).  Mirrors the reference's sequence of fp32 ops.
__device__ __forceinline__ Projection project_point(const pnr_scene& sc, int row, float px, float py,
                                                    float pz, float vx, float vy, float vz) {
  const float* M = sc.poses + (size_t)row * 12;
  Projection o;
  o.xr = M[0] * px + M[1] * py + M[2] * pz;
  o.yr = M[4] * px + M[5] * py + M[6] * pz;
  o.zr = M[8] * px + M[9] * py + M[10] * pz;
  o.dx = M[0] * vx + M[1] * vy + M[2] * vz;
  o.dy = M[4] * vx + M[5] * vy + M[6] * vz;
  o.dz = M[8] * vx + M[9] * vy + M[10] * vz;
  o.xc = o.xr + M[3]; o.yc = o.yr + M[7]; o.zc = o.zr + M[11];
  const float xc = o.xc, yc = o.yc, zc = o.zc;
  // uv = -xy / z * focal + c                      models.py:220-230
  float u = __fdiv_rn(-xc, zc) * sc.focal[row * 2 + 0] + sc.center[row * 2 + 0];
  float v = __fdiv_rn(-yc, zc) * sc.focal[row * 2 + 1] + sc.center[row * 2 + 1];
  // uv * (latent_scaling / image_size) - 1        encoder.py:97-98
  float gx = u * __fdiv_rn(sc.lat_scale_x, sc.image_w) - 1.0f;
  float gy = v * __fdiv_rn(sc.lat_scale_y, sc.image_h) - 1.0f;
  // grid_sample(align_corners=True): ((g + 1) / 2) * (size - 1)
  o.ix = ((gx + 1.0f) * 0.5f) * (float)(sc.Wl - 1);
  o.iy = ((gy + 1.0f) * 0.5f) * (float)(sc.Hl - 1);
  // YOLO mode: latent[z >= 0] = 0 (models.py:223,254-264) -- NaN coordinates fail every bounds test in make_taps
  if ((sc.flags & PNR_SCENE_MASK_NONNEG_Z) && zc >= 0.0f) o.ix = o.iy = __int_as_float(0x7fc00000);
  return o;
}

// Bilinear tap set with zero padding (ATen GridSampler: taps outside the map contribute 0).
struct Taps {
  int off[4];     // element offset of the tap's C-vector inside the view's map, or -1 if out of bounds
  float w[4];     // nw, ne, sw, se
};

__device__ __forceinline__ Taps make_taps(float ix, float iy, int Hl, int Wl, int C) {
  Taps t;
  // NaN / huge coordinates (points at the camera plane) fall out of every bounds test -> all-zero latent
  float fx = floorf(ix), fy = floorf(iy);
  float x1 = fx + 1.0f, y1 = fy + 1.0f;
  t.w[0] = (x1 - ix) * (y1 - iy);
  t.w[1] = (ix - fx) * (y1 - iy);
  t.w[2] = (x1 - ix) * (iy - fy);
  t.w[3] = (ix - fx) * (iy - fy);
  float xs[4] = {fx, x1, fx, x1};
  float ys[4] = {fy, fy, y1, y1};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    bool ok = xs[i] >= 0.0f && xs[i] <= (float)(Wl - 1) && ys[i] >= 0.0f && ys[i] <= (float)(Hl - 1);
    t.off[i] = ok ? ((int)ys[i] * Wl + (int)xs[i]) * C : -1;
    if (!ok) t.w[i] = 0.0f;
  }
  return t;
}

// z-feature layout of the PNR_SCENE_ZF_* bits (include/pixelnerf_b200.h; models.py:16-90, 183-209).  A row is
//   [u (n_raw columns), sin(f_0 u), cos(f_0 u), sin(f_1 u), ... (up to n_code), R d (up to width)]
// where u (n_u values) is the encoder input: the coordinates (3, or -z alone), then R d with CODE_VIEWDIRS.  Without the
// encoder (NO_CODE) the row is u itself, n_raw = n_code = n_u.  All bits clear: [x, y, z, sin/cos(f_k x,y,z)..., R d].
struct ZfLayout {
  int n_xyz;    // coordinate values of u: 3, or 1 (-z, Z_ONLY)
  int n_u;      // encoder input width: n_xyz, + 3 with CODE_VIEWDIRS
  int n_raw;    // leading columns that are u itself: n_u, or 0 with NO_CODE_INPUT
  int n_code;   // columns of the (encoded) u block
  int width;    // n_code, + 3 raw view-direction columns unless NO_VIEWDIRS or CODE_VIEWDIRS (= d_in)
  bool cam;     // coordinates are R x + t (CAM_COORDS) instead of R x
};
constexpr int kZfFlags = PNR_SCENE_ZF_NO_VIEWDIRS | PNR_SCENE_ZF_CODE_VIEWDIRS | PNR_SCENE_ZF_CAM_COORDS | PNR_SCENE_ZF_Z_ONLY |
                         PNR_SCENE_ZF_NO_CODE | PNR_SCENE_ZF_NO_CODE_INPUT;
__host__ __device__ inline ZfLayout zf_layout(int flags, int num_freqs) {
  const bool dirs = !(flags & PNR_SCENE_ZF_NO_VIEWDIRS);
  const bool code_dirs = dirs && (flags & PNR_SCENE_ZF_CODE_VIEWDIRS);      // models.py: use_viewdirs and use_code_viewdirs
  const bool code = !(flags & PNR_SCENE_ZF_NO_CODE);
  ZfLayout L;
  L.n_xyz = (flags & PNR_SCENE_ZF_Z_ONLY) ? 1 : 3;
  L.n_u = L.n_xyz + (code_dirs ? 3 : 0);
  L.n_raw = (code && (flags & PNR_SCENE_ZF_NO_CODE_INPUT)) ? 0 : L.n_u;
  L.n_code = L.n_raw + (code ? 2 * num_freqs * L.n_u : 0);
  L.width = L.n_code + (dirs && !code_dirs ? 3 : 0);
  L.cam = (flags & PNR_SCENE_ZF_CAM_COORDS) != 0;
  return L;
}

__device__ __forceinline__ float zf_dir(const Projection& p, int d) { return d == 0 ? p.dx : (d == 1 ? p.dy : p.dz); }
// value i of the encoder input u.  The tests are ordered so that a layout known at compile time keeps only its own case.
__device__ __forceinline__ float zf_input(const Projection& p, const ZfLayout& L, int i) {
  if (L.n_u > L.n_xyz && i >= L.n_xyz) return zf_dir(p, i - L.n_xyz);
  if (L.n_xyz == 1) return -(L.cam ? p.zc : p.zr);
  return L.cam ? (i == 0 ? p.xc : (i == 1 ? p.yc : p.zc)) : (i == 0 ? p.xr : (i == 1 ? p.yr : p.zr));
}
// Encoded column j in [n_raw, n_code): input value index i, frequency index k, and whether it is the cosine.
struct ZfCode { int i, k; bool cos; };
__device__ __forceinline__ ZfCode zf_code(const ZfLayout& L, int j) {
  const int q = j - L.n_raw, k = q / (2 * L.n_u), r = q - k * 2 * L.n_u;
  return ZfCode{r % L.n_u, k, r >= L.n_u};
}

// z-feature element j in [0, L.width)   code.py:30-42, models.py:183-209
// FAST = false: sinf of the fp32 argument, as ATen computes it (the fp32 paths).  FAST = true, for the bf16 tensor-core path
// where the value is rounded to bf16 (2^-9 relative) right after: explicit range reduction in turns + the SFU sine (abs error
// < 1e-5 for |f x| < 128) instead of the ~40-instruction libm sinf, which was 45 % of the gather warps' issue slots in the
// fused kernel (ncu source page, profiles/).
template <bool FAST>
__device__ __forceinline__ float zfeat_value(const Projection& p, const ZfLayout& L, int j, int num_freqs, float freq_factor) {
  if (j < L.n_raw) return zf_input(p, L, j);
  if (j < L.n_code) {
    const ZfCode c = zf_code(L, j);
    const float x = zf_input(p, L, c.i);
    if (FAST) {
      const float f_turns = freq_factor * (float)(1 << c.k) * 0.15915494309189535f;      // f / (2 pi)
      float t = fmaf(x, f_turns, c.cos ? 0.25f : 0.0f);
      t -= rintf(t);                                                                      // [-0.5, 0.5] turns
      return __sinf(t * 6.283185307179586f);
    }
    const float f = freq_factor * (float)(1 << c.k);
    const float ph = c.cos ? 1.57079637050628662109375f : 0.0f;   // float32(pi/2), code.py:26-27
    return sinf(fmaf(x, f, ph));                                   // sin(addcmul(phase, x, freq)): ATen fuses the multiply-add
  }
  return zf_dir(p, j - L.n_code);
}

// near * (1 - s) + far * s (nerf.py:119,151: separately rounded), or the linear-in-disparity variant (nerf.py:121,153)
__device__ __forceinline__ float lerp_depth(float near, float far, float s, int lindisp) {
  if (!lindisp) return __fadd_rn(__fmul_rn(near, __fsub_rn(1.0f, s)), __fmul_rn(far, s));
  float a = __fmul_rn(__fdiv_rn(1.0f, near), __fsub_rn(1.0f, s));
  float b = __fmul_rn(__fdiv_rn(1.0f, far), s);
  return __fdiv_rn(1.0f, __fadd_rn(a, b));
}
// sample_coarse (nerf.py:104-124) for one (ray, sample): z_steps + rand * step, then the lerp
__device__ __forceinline__ float coarse_depth(const float* __restrict__ ray, float step_k, float noise, float step, int lindisp) {
  return lerp_depth(ray[6], ray[7], __fadd_rn(step_k, __fmul_rn(noise, step)), lindisp);
}

// Fetch world point + direction `idx` (flattened (object, point)) from either point source.
__device__ __forceinline__ void fetch_point(const pnr_points& q, long long idx, float& px, float& py,
                                            float& pz, float& vx, float& vy, float& vz) {
  if (q.mode == 0) {
    const float* a = q.xyz + idx * 3;
    px = a[0]; py = a[1]; pz = a[2];
    if (q.dirs) { const float* d = q.dirs + idx * 3; vx = d[0]; vy = d[1]; vz = d[2]; }
    else { vx = vy = vz = 0.f; }
  } else {
    long long ray = idx / q.K;
    const float* r = q.rays + ray * 8;
    float zz = q.mode == 1 ? q.z[idx] : coarse_depth(r, q.steps[idx - ray * q.K], q.noise[idx], q.step, q.lindisp);
    vx = r[3]; vy = r[4]; vz = r[5];
    px = __fadd_rn(r[0], __fmul_rn(zz, vx));     // o + z * d, no FMA contraction (nerf.py:191)
    py = __fadd_rn(r[1], __fmul_rn(zz, vy));
    pz = __fadd_rn(r[2], __fmul_rn(zz, vz));
  }
}

}  // namespace pnr
