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

constexpr int kZFeat = 42;      // 39 positional-encoding values + 3 rotated view-direction values
constexpr int kHidden = 512;    // widest ResnetFC d_hidden the library runs (that of every shipped conf, conf/default*.conf)
// ResnetFC hidden widths the field and training paths run: the multiples of 64 up to kHidden
__host__ __device__ inline bool hidden_width_supported(int d_hidden) {
  return d_hidden >= 64 && d_hidden <= kHidden && d_hidden % 64 == 0;
}
#define PNR_HIDDEN_WIDTHS "64, 128, ..., 512 (multiples of 64)"

// Per-point camera-space quantities for one source view (models.py:168-230, encoder.py:94-98).
struct Projection {
  float xr, yr, zr;   // R x            (positional-encoding input, normalize_z=True)
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
  const float xc = o.xr + M[3], yc = o.yr + M[7], zc = o.zr + M[11];
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

// z-feature element j in [0,42): [x,y,z, sin/cos(f_k * x,y,z)..., R d]   code.py:30-42, models.py:183-209
__device__ __forceinline__ float zfeat_value(const Projection& p, int j, int num_freqs, float freq_factor) {
  const int n_pe = 3 + 6 * num_freqs;
  if (j < 3) return j == 0 ? p.xr : (j == 1 ? p.yr : p.zr);
  if (j < n_pe) {
    int q = j - 3;
    int k = q / 6;             // frequency index
    int r = q - k * 6;         // 0..2 sin(x,y,z), 3..5 cos(x,y,z)
    int d = r % 3;
    float x = d == 0 ? p.xr : (d == 1 ? p.yr : p.zr);
    float f = freq_factor * (float)(1 << k);
    float ph = r >= 3 ? 1.57079637050628662109375f : 0.0f;   // float32(pi/2), code.py:26-27
    return sinf(fmaf(x, f, ph));                             // sin(addcmul(phase, x, freq)): ATen fuses the multiply-add
  }
  int d = j - n_pe;
  return d == 0 ? p.dx : (d == 1 ? p.dy : p.dz);
}

// Same element for the bf16 tensor-core path, where the value is rounded to bf16 (2^-9 relative) right after: explicit
// range reduction in turns + the SFU sine (abs error < 1e-5 for |f x| < 128) instead of the ~40-instruction libm sinf,
// which was 45 % of the gather warps' issue slots in the fused kernel (ncu source page, profiles/).
__device__ __forceinline__ float zfeat_value_fast(const Projection& p, int j, int num_freqs, float freq_factor) {
  const int n_pe = 3 + 6 * num_freqs;
  if (j < 3) return j == 0 ? p.xr : (j == 1 ? p.yr : p.zr);
  if (j < n_pe) {
    const int q = j - 3, k = q / 6, r = q - k * 6, d = r % 3;
    const float x = d == 0 ? p.xr : (d == 1 ? p.yr : p.zr);
    const float f_turns = freq_factor * (float)(1 << k) * 0.15915494309189535f;      // f / (2 pi)
    float t = fmaf(x, f_turns, r >= 3 ? 0.25f : 0.0f);
    t -= rintf(t);                                                                    // [-0.5, 0.5] turns
    return __sinf(t * 6.283185307179586f);
  }
  const int d = j - n_pe;
  return d == 0 ? p.dx : (d == 1 ? p.dy : p.dz);
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
