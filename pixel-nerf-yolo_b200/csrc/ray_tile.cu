// F1: per-ray sampling, alpha compositing and inverse-CDF resampling (src/render/nerf.py).
// One warp owns one ray; the K-length recurrences (transmittance product, CDF sum) are warp-level
// prefix scans carried across 32-sample chunks.  Scans run in double and round to float per element,
// which is what torch.cumsum / torch.cumprod do on the CPU oracle (acc_type<float> = double).
#include "pnr_common.cuh"

namespace pnr {

constexpr int kWarpsPerBlock = 4;
constexpr int kMaxSortN = 512;   // padded (power of two) sort buffer per warp

__global__ void sample_coarse_kernel(const float* __restrict__ rays, const float* __restrict__ steps,
                                     const float* __restrict__ noise, float* __restrict__ z, int B, int Kc,
                                     float step, int lindisp) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * Kc) return;
  int b = (int)(i / Kc), k = (int)(i - (long long)b * Kc);
  z[i] = coarse_depth(rays + (size_t)b * 8, steps[k], noise[i], step, lindisp);   // z_steps += rand * step, lerp   nerf.py:117-121
}

template <typename T>
__device__ __forceinline__ T warp_incl_scan_mul(T v, int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    T o = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= d) v *= o;
  }
  return v;
}
template <typename T>
__device__ __forceinline__ T warp_incl_scan_add(T v, int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    T o = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= d) v += o;
  }
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  return v;
}

// nerf.py:184-188 + 229-255 for ray b, executed by one warp
__device__ __forceinline__ void composite_ray(const float4* __restrict__ rgb_sigma, const float* __restrict__ z,
                                              const float* __restrict__ rays, float* __restrict__ weights, float* __restrict__ rgb,
                                              float* __restrict__ depth, int b, int K, int white_bkgd, int lane) {
  const float far = rays[b * 8 + 7];
  const float* zr = z + (size_t)b * K;
  const float4* o = rgb_sigma + (size_t)b * K;
  double carry = 1.0;                      // running product of (1 - alpha + 1e-10), exclusive
  float acc_r = 0.f, acc_g = 0.f, acc_b = 0.f, acc_d = 0.f, acc_w = 0.f;
  for (int base = 0; base < K; base += 32) {
    const int i = base + lane;
    const bool valid = i < K;
    float zi = 0.f, alpha = 0.f;
    float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid) {
      zi = zr[i];
      float znext = (i + 1 < K) ? zr[i + 1] : far;          // delta_inf = far - z_last   nerf.py:187
      float delta = __fsub_rn(znext, zi);
      c = o[i];
      float sig = fmaxf(c.w, 0.0f);
      alpha = __fsub_rn(1.0f, expf(__fmul_rn(-delta, sig))); // 1 - exp(-delta * relu(sigma))
    }
    float a_shift = valid ? __fadd_rn(__fsub_rn(1.0f, alpha), 1e-10f) : 1.0f;
    double incl = warp_incl_scan_mul<double>((double)a_shift, lane);
    double excl = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) excl = 1.0;
    float T = (float)(carry * excl);       // cumprod([1, a_0, a_1, ...])[i], rounded per element
    carry = carry * __shfl_sync(0xffffffffu, incl, 31);
    float w = __fmul_rn(alpha, T);
    if (valid) {
      if (weights) weights[(size_t)b * K + i] = w;
      acc_r += w * c.x; acc_g += w * c.y; acc_b += w * c.z;
      acc_d += w * zi;  acc_w += w;
    }
  }
  acc_r = warp_sum(acc_r); acc_g = warp_sum(acc_g); acc_b = warp_sum(acc_b);
  acc_d = warp_sum(acc_d); acc_w = warp_sum(acc_w);
  if (lane == 0) {
    if (white_bkgd) {                      // rgb + 1 - pix_alpha                        nerf.py:247-250
      acc_r = __fsub_rn(__fadd_rn(acc_r, 1.0f), acc_w);
      acc_g = __fsub_rn(__fadd_rn(acc_g, 1.0f), acc_w);
      acc_b = __fsub_rn(__fadd_rn(acc_b, 1.0f), acc_w);
    }
    rgb[b * 3 + 0] = acc_r; rgb[b * 3 + 1] = acc_g; rgb[b * 3 + 2] = acc_b;
    depth[b] = acc_d;
  }
}
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
composite_kernel(const float4* __restrict__ rgb_sigma, const float* __restrict__ z,
                 const float* __restrict__ rays, float* __restrict__ weights, float* __restrict__ rgb,
                 float* __restrict__ depth, int B, int K, int white_bkgd) {
  const int b = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (b >= B) return;
  composite_ray(rgb_sigma, z, rays, weights, rgb, depth, b, K, white_bkgd, threadIdx.x & 31);
}

// In-warp bitonic sort of n (power of two, <= kMaxSortN) floats in shared memory, ascending.
__device__ __forceinline__ void warp_bitonic_sort(float* s, int n, int lane) {
  for (int k = 2; k <= n; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = lane; t < n / 2; t += 32) {
        // t-th compare-exchange pair of this stage
        int i = 2 * t - (t & (j - 1));
        int p = i + j;
        bool up = ((i & k) == 0);
        float a = s[i], c = s[p];
        if ((a > c) == up) { s[i] = c; s[p] = a; }
      }
      __syncwarp();
    }
  }
}

// nerf.py:126-167 + 300-301 for ray b, executed by one warp; cdf / srt: this warp's kMaxSortN-float scratch areas
__device__ __forceinline__ void resample_ray(const float* __restrict__ weights, const float* __restrict__ depth,
                                             const float* __restrict__ rays, const float* __restrict__ z_coarse,
                                             const float* __restrict__ u, const float* __restrict__ jitter,
                                             const float* __restrict__ gauss, float* __restrict__ z_out, int32_t* __restrict__ inds_out,
                                             float* __restrict__ z_fine_out, float* __restrict__ z_depth_out, int b, int Kc, int Kf,
                                             int Kfd, float depth_std, int lindisp, int n_pad, int lane, float* cdf, float* srt) {
  const float near = rays[b * 8 + 6], far = rays[b * 8 + 7];
  const int Ktot = Kc + Kf + Kfd;

  if (Kf > 0) {
    const float* w = weights + (size_t)b * Kc;
    // pdf = (w + 1e-5) / sum(w + 1e-5)                    nerf.py:136-137
    float part = 0.f;
    for (int i = lane; i < Kc; i += 32) part += __fadd_rn(w[i], 1e-5f);
    const float tot = warp_sum(part);
    // cdf = [0, cumsum(pdf)] : double running sum, rounded to float per element  nerf.py:138-139
    double carry = 0.0;
    if (lane == 0) cdf[0] = 0.0f;
    for (int base = 0; base < Kc; base += 32) {
      int i = base + lane;
      float pdf = (i < Kc) ? __fdiv_rn(__fadd_rn(w[i], 1e-5f), tot) : 0.0f;
      double incl = warp_incl_scan_add<double>((double)pdf, lane);
      if (i < Kc) cdf[i + 1] = (float)(carry + incl);
      carry += __shfl_sync(0xffffffffu, incl, 31);
    }
    __syncwarp();
    for (int j = lane; j < Kf; j += 32) {
      float uj = u[(size_t)b * Kf + j];
      // searchsorted(cdf, u, right=True): first index with cdf[idx] > u   nerf.py:144
      int lo = 0, hi = Kc + 1;
      while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (cdf[mid] <= uj) lo = mid + 1; else hi = mid;
      }
      float ind = fmaxf((float)lo - 1.0f, 0.0f);           // clamp_min(inds - 1, 0)       nerf.py:144-145
      float s = __fdiv_rn(__fadd_rn(ind, jitter[(size_t)b * Kf + j]), (float)Kc);   // nerf.py:147
      float zz = lerp_depth(near, far, s, lindisp);
      srt[Kc + j] = zz;
      if (inds_out) inds_out[(size_t)b * Kf + j] = (int32_t)ind;
      if (z_fine_out) z_fine_out[(size_t)b * Kf + j] = zz;
    }
  }
  if (Kfd > 0) {
    const float d = depth[b];
    for (int j = lane; j < Kfd; j += 32) {
      // depth + randn * depth_std, clamped to [near, far]   nerf.py:163-166
      float zz = __fadd_rn(d, __fmul_rn(gauss[(size_t)b * Kfd + j], depth_std));
      zz = fmaxf(fminf(zz, far), near);
      srt[Kc + Kf + j] = zz;
      if (z_depth_out) z_depth_out[(size_t)b * Kfd + j] = zz;
    }
  }
  for (int i = lane; i < Kc; i += 32) srt[i] = z_coarse[(size_t)b * Kc + i];
  for (int i = Ktot + lane; i < n_pad; i += 32) srt[i] = __int_as_float(0x7f800000);   // +inf padding
  __syncwarp();
  warp_bitonic_sort(srt, n_pad, lane);                     // torch.sort(cat(...))   nerf.py:300-301
  for (int i = lane; i < Ktot; i += 32) z_out[(size_t)b * Ktot + i] = srt[i];
}
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
sample_fine_kernel(const float* __restrict__ weights, const float* __restrict__ depth,
                   const float* __restrict__ rays, const float* __restrict__ z_coarse,
                   const float* __restrict__ u, const float* __restrict__ jitter,
                   const float* __restrict__ gauss, float* __restrict__ z_out, int32_t* __restrict__ inds_out,
                   float* __restrict__ z_fine_out, float* __restrict__ z_depth_out, int B, int Kc, int Kf,
                   int Kfd, float depth_std, int lindisp, int n_pad) {
  extern __shared__ float smem[];
  const int wid = threadIdx.x >> 5;
  const int b = blockIdx.x * kWarpsPerBlock + wid;
  if (b >= B) return;
  float* cdf = smem + (size_t)wid * (2 * kMaxSortN);       // Kc+1 entries
  resample_ray(weights, depth, rays, z_coarse, u, jitter, gauss, z_out, inds_out, z_fine_out, z_depth_out, b, Kc, Kf, Kfd, depth_std,
               lindisp, n_pad, threadIdx.x & 31, cdf, cdf + kMaxSortN);
}

// What pnr_render_forward runs between the two field launches, in one launch: the coarse depths are recomputed exactly as
// sample_coarse_kernel computes them (and stored for the merge), then composite_ray and resample_ray run back to back in the warp
// that owns the ray (its own global writes are visible to it after __syncwarp).
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
composite_resample_kernel(const float4* __restrict__ rgb_sigma, const float* __restrict__ rays, const float* __restrict__ steps,
                          const float* __restrict__ noise, const float* __restrict__ u, const float* __restrict__ jitter,
                          const float* __restrict__ gauss, float* __restrict__ z_coarse, float* __restrict__ weights,
                          float* __restrict__ rgb, float* __restrict__ depth, float* __restrict__ z_fine, int B, int Kc, int Kf, int Kfd,
                          float step, float depth_std, int white_bkgd, int lindisp, int n_pad) {
  extern __shared__ float smem[];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int b = blockIdx.x * kWarpsPerBlock + wid;
  if (b >= B) return;
  const float* ray = rays + (size_t)b * 8;
  for (int k = lane; k < Kc; k += 32) z_coarse[(size_t)b * Kc + k] = coarse_depth(ray, steps[k], noise[(size_t)b * Kc + k], step, lindisp);
  __syncwarp();
  composite_ray(rgb_sigma, z_coarse, rays, weights, rgb, depth, b, Kc, white_bkgd, lane);
  if (Kf + Kfd == 0) return;
  __syncwarp();
  float* cdf = smem + (size_t)wid * (2 * kMaxSortN);
  resample_ray(weights, depth, rays, z_coarse, u, jitter, gauss, z_fine, nullptr, nullptr, nullptr, b, Kc, Kf, Kfd, depth_std, lindisp,
               n_pad, lane, cdf, cdf + kMaxSortN);
}


// Backward of composite (nerf.py:184-188, 229-255), one warp per ray.  Given d rgb (B,3), d depth (B) and optionally
// d weights (B,K):   dw_i = d_rgb . c_i + d_depth z_i + d_weights_i - [white] sum(d_rgb)
//                    dalpha_i = dw_i T_i - (sum_{j>i} dw_j w_j) / (1 - alpha_i + 1e-10)        (w_j = alpha_j T_j)
//                    dsigma_i = dalpha_i delta_i (1 - alpha_i) [sigma_i > 0],   ddelta_i = dalpha_i relu(sigma_i) (1 - alpha_i)
//                    dz_i = w_i d_depth + ddelta_{i-1} - ddelta_i          (delta_i = z_{i+1} - z_i, last: far - z_K)
// alpha and T are recomputed exactly as composite_kernel does; the suffix sum runs in double.
// RAYS: also d far (the last interval is far - z_K) added into column 7 of d_rays; the instantiation without it is the kernel
// every training step runs.
template <bool RAYS>
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
composite_bwd_kernel(const float4* __restrict__ rgb_sigma, const float* __restrict__ z, const float* __restrict__ rays,
                     const float* __restrict__ d_rgb, const float* __restrict__ d_depth, const float* __restrict__ d_weights,
                     float4* __restrict__ d_rgb_sigma, float* __restrict__ d_z, float* __restrict__ d_rays, int B, int K,
                     int white_bkgd) {
  extern __shared__ float smem[];
  const int lane = threadIdx.x & 31;
  const int wid = threadIdx.x >> 5;
  const int b = blockIdx.x * kWarpsPerBlock + wid;
  if (b >= B) return;
  float* sT = smem + (size_t)wid * 3 * K;      // T_i
  float* sA = sT + K;                          // alpha_i
  float* sD = sA + K;                          // ddelta_i
  const float far = rays[b * 8 + 7];
  const float* zr = z + (size_t)b * K;
  const float4* o = rgb_sigma + (size_t)b * K;
  const float gr = d_rgb[b * 3 + 0], gg = d_rgb[b * 3 + 1], gb = d_rgb[b * 3 + 2];
  const float gd = d_depth ? d_depth[b] : 0.f;
  const float gwhite = white_bkgd ? (gr + gg + gb) : 0.f;
  double carry = 1.0;
  for (int base = 0; base < K; base += 32) {
    const int i = base + lane;
    const bool valid = i < K;
    float alpha = 0.f;
    if (valid) {
      const float zi = zr[i];
      const float znext = (i + 1 < K) ? zr[i + 1] : far;
      const float delta = __fsub_rn(znext, zi);
      const float sig = fmaxf(o[i].w, 0.0f);
      alpha = __fsub_rn(1.0f, expf(__fmul_rn(-delta, sig)));
    }
    const float a_shift = valid ? __fadd_rn(__fsub_rn(1.0f, alpha), 1e-10f) : 1.0f;
    const double incl = warp_incl_scan_mul<double>((double)a_shift, lane);
    double excl = __shfl_up_sync(0xffffffffu, incl, 1);
    if (lane == 0) excl = 1.0;
    if (valid) { sT[i] = (float)(carry * excl); sA[i] = alpha; }
    carry = carry * __shfl_sync(0xffffffffu, incl, 31);
  }
  __syncwarp();
  double suffix = 0.0;                          // sum_{j > current chunk} dw_j w_j
  const int n_chunks = (K + 31) / 32;
  for (int ch = n_chunks - 1; ch >= 0; --ch) {
    const int i = ch * 32 + lane;
    const bool valid = i < K;
    float dw = 0.f, w = 0.f, T = 0.f, alpha = 0.f, zi = 0.f, delta = 0.f;
    float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid) {
      c = o[i]; zi = zr[i]; T = sT[i]; alpha = sA[i];
      const float znext = (i + 1 < K) ? zr[i + 1] : far;
      delta = __fsub_rn(znext, zi);
      w = alpha * T;
      dw = gr * c.x + gg * c.y + gb * c.z + gd * zi - gwhite + (d_weights ? d_weights[(size_t)b * K + i] : 0.f);
    }
    // inclusive suffix scan of dw*w within the chunk (lanes above), then make it exclusive
    double v = (double)dw * (double)w;
    double incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const double t = __shfl_down_sync(0xffffffffu, incl, d);
      if (lane + d < 32) incl += t;
    }
    const double S = suffix + (incl - v);
    suffix += __shfl_sync(0xffffffffu, incl, 0);
    if (valid) {
      const float one_m = __fadd_rn(__fsub_rn(1.0f, alpha), 1e-10f);
      const float dalpha = dw * T - (float)(S / (double)one_m);
      const float keep = 1.0f - alpha;          // d alpha / d (delta * sigma) = exp(-delta sigma) = 1 - alpha
      const float sig = fmaxf(c.w, 0.0f);
      const float dsig = (c.w > 0.0f) ? dalpha * delta * keep : 0.0f;
      sD[i] = dalpha * sig * keep;
      d_rgb_sigma[(size_t)b * K + i] = make_float4(w * gr, w * gg, w * gb, dsig);
    }
  }
  if (d_z) {
    __syncwarp();
    for (int i = lane; i < K; i += 32) {
      const float w = sA[i] * sT[i];
      d_z[(size_t)b * K + i] = w * gd + (i > 0 ? sD[i - 1] : 0.f) - sD[i];
    }
  }
  if (RAYS && lane == ((K - 1) & 31)) d_rays[b * 8 + 7] += sD[K - 1];
}

// Backward of sample_fine_depth + cat + sort (nerf.py:156-167, 296-301) with respect to the coarse depth: the Kfd depth
// samples are z_j = clamp(depth + gauss_j * depth_std, near, far); sample j sits at the position of its value in the
// sorted row, and passes the gradient on unless it was clamped.  (sample_fine is fed detached weights, nerf.py:136,293.)
__global__ void sample_depth_bwd_kernel(const float* __restrict__ z_sorted, const float* __restrict__ d_z_sorted,
                                        const float* __restrict__ depth, const float* __restrict__ gauss,
                                        const float* __restrict__ rays, float* __restrict__ d_depth, int B, int K, int Kfd,
                                        float depth_std) {
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= B) return;
  const float near = rays[b * 8 + 6], far = rays[b * 8 + 7], d = depth[b];
  const float* zs = z_sorted + (size_t)b * K;
  float acc = 0.f;
  for (int j = lane; j < Kfd; j += 32) {
    const float raw = __fadd_rn(d, __fmul_rn(gauss[(size_t)b * Kfd + j], depth_std));
    if (!(raw > near && raw < far)) continue;                 // clamped (or NaN): no gradient
    int lo = 0, hi = K;                                       // first position with zs[pos] >= raw
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (zs[mid] < raw) lo = mid + 1; else hi = mid; }
    int rank = 0;                                             // equal depth samples occupy consecutive positions
    for (int jj = 0; jj < j; ++jj)
      if (__fadd_rn(d, __fmul_rn(gauss[(size_t)b * Kfd + jj], depth_std)) == raw) ++rank;
    const int pos = lo + rank;
    if (pos < K && zs[pos] == raw) acc += d_z_sorted[(size_t)b * K + pos];
  }
  acc = warp_sum(acc);
  if (lane == 0) d_depth[b] = acc;
}

// near / far gradients of the sample depths, one warp per ray.  Every sample is a function of the ray's bounds:
//   coarse (nerf.py:117-121) and importance (nerf.py:147-153) samples z = lerp_depth(near, far, s), with s = steps_k + noise / Kc
//   or s = (ind + jitter) / Kc (the bin is piecewise constant; the sampler reads detached weights, nerf.py:136,293);
//   depth samples (nerf.py:163-166) z = clamp(depth + gauss std, near, far) send their gradient to the bound they clamp at.
// z_sorted == nullptr: the coarse samples with their gradient d_z_coarse (B, Kc).  Otherwise the fine pass's merged row z_sorted
// (B, Kc + Kf + Kfd) and its gradient: each sample of the concatenation (coarse, importance, depth; nerf.py:300-301) is found at
// the position of its value, equal values taking consecutive positions in concatenation order; the coarse samples' share goes
// to d_z_coarse_out (B, Kc; overwritten, may be null), the unclamped depth samples' share to the depth
// (pnr_sample_fine_depth_backward).  d near / d far are added into columns 6 and 7 of d_rays (B, 8).
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
sample_bounds_bwd_kernel(const float* __restrict__ rays, const float* __restrict__ steps, const float* __restrict__ noise,
                         const float* __restrict__ d_z_coarse, const float* __restrict__ z_coarse, const float* __restrict__ z_sorted,
                         const float* __restrict__ d_z_sorted, const int32_t* __restrict__ inds, const float* __restrict__ jitter,
                         const float* __restrict__ depth, const float* __restrict__ gauss, float* __restrict__ d_rays,
                         float* __restrict__ d_z_coarse_out, int B, int Kc, int Kf, int Kfd, float step, float depth_std, int lindisp) {
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (b >= B) return;
  const float near = rays[b * 8 + 6], far = rays[b * 8 + 7];
  float dn = 0.f, df = 0.f;
  // z = near (1 - s) + far s, or 1 / ((1 - s) / near + s / far) with lindisp: dz/dnear = z^2 (1 - s) / near^2, dz/dfar = z^2 s / far^2
  auto bounds = [&](float s, float g) {
    if (!lindisp) { dn += g * (1.0f - s); df += g * s; return; }
    const float z = lerp_depth(near, far, s, 1);
    dn += g * z * z * (1.0f - s) / (near * near);
    df += g * z * z * s / (far * far);
  };
  if (!z_sorted) {
    for (int k = lane; k < Kc; k += 32) {
      const size_t i = (size_t)b * Kc + k;
      bounds(__fadd_rn(steps[k], __fmul_rn(noise[i], step)), d_z_coarse[i]);
    }
  } else {
    const int K = Kc + Kf + Kfd;
    const float* zs = z_sorted + (size_t)b * K;
    const float* dzs = d_z_sorted + (size_t)b * K;
    const float d = Kfd > 0 ? depth[b] : 0.f;
    auto fine_s = [&](int j) { return __fdiv_rn(__fadd_rn((float)inds[(size_t)b * Kf + j], jitter[(size_t)b * Kf + j]), (float)Kc); };
    auto depth_raw = [&](int j) { return __fadd_rn(d, __fmul_rn(gauss[(size_t)b * Kfd + j], depth_std)); };
    auto cat_value = [&](int c) {            // sample c of the concatenation, exactly as pnr_sample_fine computes it
      if (c < Kc) return z_coarse[(size_t)b * Kc + c];
      if (c < Kc + Kf) return lerp_depth(near, far, fine_s(c - Kc), lindisp);
      return fmaxf(fminf(depth_raw(c - Kc - Kf), far), near);
    };
    auto grad_at = [&](float v, int c) {     // gradient at the sorted position of sample c (value v)
      int lo = 0, hi = K;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (zs[mid] < v) lo = mid + 1; else hi = mid; }
      if (lo + 1 < K && zs[lo + 1] == v)
        for (int cc = 0; cc < c; ++cc) lo += cat_value(cc) == v;
      return (lo < K && zs[lo] == v) ? dzs[lo] : 0.f;
    };
    for (int k = lane; k < Kc; k += 32) {
      const float g = grad_at(z_coarse[(size_t)b * Kc + k], k);
      if (d_z_coarse_out) d_z_coarse_out[(size_t)b * Kc + k] = g;
    }
    for (int j = lane; j < Kf; j += 32) {
      const float s = fine_s(j);
      bounds(s, grad_at(lerp_depth(near, far, s, lindisp), Kc + j));
    }
    for (int j = lane; j < Kfd; j += 32) {
      const float raw = depth_raw(j);
      if (raw > near && raw < far) continue;                    // unclamped: the gradient goes to the depth
      const float g = grad_at(fmaxf(fminf(raw, far), near), Kc + Kf + j);
      if (raw <= near) dn += g;
      else if (raw >= far) df += g;
    }
  }
  dn = warp_sum(dn);
  df = warp_sum(df);
  if (lane == 0) { d_rays[b * 8 + 6] += dn; d_rays[b * 8 + 7] += df; }
}

// YoloRenderer.forward's per-ray reduction (src/render/yolo.py:96-114): raw field values (B, K, A*7) -> (B, A, 7) =
// [max_k p, sum_k(v * p) / (sum_k p + 1e-5)] with p = sigmoid(value 0 of the anchor).  One warp per (ray, anchor).
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
yolo_reduce_kernel(const float* __restrict__ out, float* __restrict__ res, long long n_pairs, int K, int A) {
  const int lane = threadIdx.x & 31;
  const long long pa = (long long)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (pa >= n_pairs) return;
  const long long b = pa / A;
  const int a = (int)(pa - b * A);
  const float* o = out + (size_t)b * K * A * 7 + a * 7;
  float sp = 0.f, mp = -1.0f, sv[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int k = lane; k < K; k += 32) {
    const float* v = o + (size_t)k * A * 7;
    const float p = 1.0f / (1.0f + expf(-v[0]));
    sp += p;
    mp = fmaxf(mp, p);
#pragma unroll
    for (int j = 0; j < 6; ++j) sv[j] += v[1 + j] * p;
  }
  sp = warp_sum(sp);
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) mp = fmaxf(mp, __shfl_xor_sync(0xffffffffu, mp, d));
#pragma unroll
  for (int j = 0; j < 6; ++j) sv[j] = warp_sum(sv[j]);
  if (lane == 0) {
    float* r = res + pa * 7;
    r[0] = mp;
#pragma unroll
    for (int j = 0; j < 6; ++j) r[1 + j] = __fdiv_rn(sv[j], __fadd_rn(sp, 1e-5f));
  }
}

// Backward of the reduction above (what autograd derives for src/render/yolo.py:96-114): d_res (pairs, 7) -> d_out (B, K, A*7).
//   r_0 = max_k p_k            -> d p_k  = d_res_0 [k == first argmax]          (torch.max's gradient goes to one index)
//   r_j = N_j / S, N_j = sum_k v_jk p_k, S = sum_k p_k + 1e-5
//                              -> d v_jk = d_res_j p_k / S ;  d p_k += sum_j d_res_j (v_jk - r_j) / S
//   p = sigmoid(o)             -> d o_k  = d p_k p_k (1 - p_k)
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
yolo_reduce_bwd_kernel(const float* __restrict__ out, const float* __restrict__ d_res, float* __restrict__ d_out, long long n_pairs,
                       int K, int A) {
  const int lane = threadIdx.x & 31;
  const long long pa = (long long)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
  if (pa >= n_pairs) return;
  const long long b = pa / A;
  const int a = (int)(pa - b * A);
  const float* o = out + (size_t)b * K * A * 7 + a * 7;
  float* go = d_out + (size_t)b * K * A * 7 + a * 7;
  float sp = 0.f, mp = -1.0f, sv[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  int arg = 0x7fffffff;
  for (int k = lane; k < K; k += 32) {
    const float* v = o + (size_t)k * A * 7;
    const float p = 1.0f / (1.0f + expf(-v[0]));
    sp += p;
    if (p > mp) { mp = p; arg = k; }
#pragma unroll
    for (int j = 0; j < 6; ++j) sv[j] += v[1 + j] * p;
  }
  sp = warp_sum(sp);
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {                    // (max, lowest index) reduction
    const float om = __shfl_xor_sync(0xffffffffu, mp, d);
    const int oa = __shfl_xor_sync(0xffffffffu, arg, d);
    if (om > mp || (om == mp && oa < arg)) { mp = om; arg = oa; }
  }
#pragma unroll
  for (int j = 0; j < 6; ++j) sv[j] = warp_sum(sv[j]);
  const float S = __fadd_rn(sp, 1e-5f);
  const float* gr = d_res + pa * 7;
  float g[7], r[6];
#pragma unroll
  for (int j = 0; j < 7; ++j) g[j] = gr[j];
#pragma unroll
  for (int j = 0; j < 6; ++j) r[j] = __fdiv_rn(sv[j], S);
  for (int k = lane; k < K; k += 32) {
    const float* v = o + (size_t)k * A * 7;
    float* gv = go + (size_t)k * A * 7;
    const float p = 1.0f / (1.0f + expf(-v[0]));
    float dp = (k == arg) ? g[0] : 0.f;
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      gv[1 + j] = g[1 + j] * p / S;
      dp += g[1 + j] * (v[1 + j] - r[j]) / S;
    }
    gv[0] = dp * p * (1.0f - p);
  }
}

}  // namespace pnr

using namespace pnr;

extern "C" int pnr_sample_coarse(const float* rays, const float* steps, const float* noise, float* z, int B,
                                 int Kc, int lindisp, void* stream) {
  reset_launch_count();
  PNR_REQUIRE(rays && steps && noise && z, PNR_ERR_ARG, "pnr_sample_coarse: null pointer");
  PNR_REQUIRE(B >= 0 && Kc > 0, PNR_ERR_ARG, "pnr_sample_coarse: bad shape B=%d Kc=%d", B, Kc);
  if (B == 0) return PNR_OK;
  long long n = (long long)B * Kc;
  float step = (float)(1.0 / (double)Kc);
  sample_coarse_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(rays, steps, noise, z, B,
                                                                                      Kc, step, lindisp);
  PNR_CHECK_LAUNCH("sample_coarse_kernel");
  return PNR_OK;
}

extern "C" int pnr_composite(const float* rgb_sigma, const float* z, const float* rays, float* weights,
                             float* rgb, float* depth, int B, int K, int white_bkgd, void* stream) {
  reset_launch_count();
  PNR_REQUIRE(rgb_sigma && z && rays && rgb && depth, PNR_ERR_ARG, "pnr_composite: null pointer");
  PNR_REQUIRE(B >= 0 && K > 0, PNR_ERR_ARG, "pnr_composite: bad shape B=%d K=%d", B, K);
  if (B == 0) return PNR_OK;
  composite_kernel<<<(B + kWarpsPerBlock - 1) / kWarpsPerBlock, kWarpsPerBlock * 32, 0, (cudaStream_t)stream>>>(
      (const float4*)rgb_sigma, z, rays, weights, rgb, depth, B, K, white_bkgd);
  PNR_CHECK_LAUNCH("composite_kernel");
  return PNR_OK;
}

extern "C" int pnr_sample_fine(const float* weights, const float* depth, const float* rays,
                               const float* z_coarse, const float* u, const float* jitter, const float* gauss,
                               float* z_out, int32_t* inds_out, float* z_fine_out, float* z_depth_out, int B,
                               int Kc, int Kf, int Kfd, float depth_std, int lindisp, void* stream) {
  reset_launch_count();
  PNR_REQUIRE(rays && z_coarse && z_out, PNR_ERR_ARG, "pnr_sample_fine: null pointer");
  PNR_REQUIRE(Kf == 0 || (weights && u && jitter), PNR_ERR_ARG, "pnr_sample_fine: importance inputs missing");
  PNR_REQUIRE(Kfd == 0 || (depth && gauss), PNR_ERR_ARG, "pnr_sample_fine: depth-sample inputs missing");
  PNR_REQUIRE(B >= 0 && Kc > 0 && Kf >= 0 && Kfd >= 0, PNR_ERR_ARG, "pnr_sample_fine: bad shape");
  int Ktot = Kc + Kf + Kfd;
  int n_pad = 32;
  while (n_pad < Ktot) n_pad <<= 1;
  PNR_REQUIRE(n_pad <= kMaxSortN && Kc + 1 <= kMaxSortN, PNR_ERR_UNSUPPORTED,
              "pnr_sample_fine: %d samples per ray exceeds the %d-sample tile", Ktot, kMaxSortN);
  if (B == 0) return PNR_OK;
  size_t smem = (size_t)kWarpsPerBlock * 2 * kMaxSortN * sizeof(float);
  sample_fine_kernel<<<(B + kWarpsPerBlock - 1) / kWarpsPerBlock, kWarpsPerBlock * 32, smem,
                       (cudaStream_t)stream>>>(weights, depth, rays, z_coarse, u, jitter, gauss, z_out, inds_out,
                                               z_fine_out, z_depth_out, B, Kc, Kf, Kfd, depth_std, lindisp, n_pad);
  PNR_CHECK_LAUNCH("sample_fine_kernel");
  return PNR_OK;
}

extern "C" int pnr_composite_resample(const float* rgb_sigma, const float* rays, const float* steps, const float* noise_coarse,
                                      const float* u, const float* jitter, const float* gauss, float* z_coarse_out,
                                      float* weights_coarse, float* rgb_coarse, float* depth_coarse, float* z_fine_out, int B, int Kc,
                                      int Kf, int Kfd, float depth_std, int white_bkgd, int lindisp, void* stream) {
  reset_launch_count();
  PNR_REQUIRE(rgb_sigma && rays && steps && noise_coarse && z_coarse_out && weights_coarse && rgb_coarse && depth_coarse, PNR_ERR_ARG,
              "pnr_composite_resample: null pointer");
  PNR_REQUIRE(B >= 0 && Kc > 0 && Kf >= 0 && Kfd >= 0, PNR_ERR_ARG, "pnr_composite_resample: bad shape");
  PNR_REQUIRE(Kf + Kfd == 0 || z_fine_out, PNR_ERR_ARG, "pnr_composite_resample: z_fine_out missing");
  PNR_REQUIRE((Kf == 0 || (u && jitter)) && (Kfd == 0 || gauss), PNR_ERR_ARG, "pnr_composite_resample: noise missing");
  if (B == 0) return PNR_OK;
  const int Ktot = Kc + Kf + Kfd;
  int n_pad = 32;
  while (n_pad < Ktot) n_pad <<= 1;
  PNR_REQUIRE(n_pad <= kMaxSortN && Kc + 1 <= kMaxSortN, PNR_ERR_UNSUPPORTED, "pnr_composite_resample: %d samples per ray exceed the %d-entry sort buffer",
              Ktot, kMaxSortN);
  const size_t smem = (size_t)kWarpsPerBlock * 2 * kMaxSortN * sizeof(float);
  composite_resample_kernel<<<(B + kWarpsPerBlock - 1) / kWarpsPerBlock, kWarpsPerBlock * 32, smem, (cudaStream_t)stream>>>(
      (const float4*)rgb_sigma, rays, steps, noise_coarse, u, jitter, gauss, z_coarse_out, weights_coarse, rgb_coarse, depth_coarse, z_fine_out,
      B, Kc, Kf, Kfd, (float)(1.0 / (double)Kc), depth_std, white_bkgd, lindisp, n_pad);
  PNR_CHECK_LAUNCH("composite_resample_kernel");
  return PNR_OK;
}

extern "C" int pnr_composite_backward(const float* rgb_sigma, const float* z, const float* rays, const float* d_rgb,
                                      const float* d_depth, const float* d_weights, float* d_rgb_sigma, float* d_z,
                                      int B, int K, int white_bkgd, void* stream) {
  return pnr_composite_backward_rays(rgb_sigma, z, rays, d_rgb, d_depth, d_weights, d_rgb_sigma, d_z, nullptr, B, K, white_bkgd,
                                     stream);
}

extern "C" int pnr_composite_backward_rays(const float* rgb_sigma, const float* z, const float* rays, const float* d_rgb,
                                           const float* d_depth, const float* d_weights, float* d_rgb_sigma, float* d_z,
                                           float* d_rays, int B, int K, int white_bkgd, void* stream) {
  reset_launch_count();
  PNR_REQUIRE(rgb_sigma && z && rays && d_rgb && d_rgb_sigma, PNR_ERR_ARG, "pnr_composite_backward: null pointer");
  PNR_REQUIRE(B >= 0 && K > 0 && K <= 1024, PNR_ERR_ARG, "pnr_composite_backward: bad shape B=%d K=%d", B, K);
  if (B == 0) return PNR_OK;
  const size_t smem = (size_t)kWarpsPerBlock * 3 * K * sizeof(float);
  const unsigned grid = (B + kWarpsPerBlock - 1) / kWarpsPerBlock;
  if (d_rays)
    composite_bwd_kernel<true><<<grid, kWarpsPerBlock * 32, smem, (cudaStream_t)stream>>>(
        (const float4*)rgb_sigma, z, rays, d_rgb, d_depth, d_weights, (float4*)d_rgb_sigma, d_z, d_rays, B, K, white_bkgd);
  else
    composite_bwd_kernel<false><<<grid, kWarpsPerBlock * 32, smem, (cudaStream_t)stream>>>(
        (const float4*)rgb_sigma, z, rays, d_rgb, d_depth, d_weights, (float4*)d_rgb_sigma, d_z, nullptr, B, K, white_bkgd);
  PNR_CHECK_LAUNCH("composite_bwd_kernel");
  return PNR_OK;
}

extern "C" int pnr_sample_bounds_backward(const float* rays, const float* steps, const float* noise_coarse, const float* d_z_coarse,
                                          const float* z_coarse, const float* z_sorted, const float* d_z_sorted, const int32_t* inds,
                                          const float* jitter, const float* depth, const float* gauss, float* d_rays,
                                          float* d_z_coarse_out, int B, int Kc, int Kf, int Kfd, float depth_std, int lindisp,
                                          void* stream) {
  reset_launch_count();
  PNR_REQUIRE(rays && d_rays, PNR_ERR_ARG, "pnr_sample_bounds_backward: null pointer");
  PNR_REQUIRE(B >= 0 && Kc > 0 && Kf >= 0 && Kfd >= 0, PNR_ERR_ARG, "pnr_sample_bounds_backward: bad shape");
  if (!z_sorted)
    PNR_REQUIRE(steps && noise_coarse && d_z_coarse, PNR_ERR_ARG, "pnr_sample_bounds_backward: coarse inputs missing");
  else
    PNR_REQUIRE(z_coarse && d_z_sorted && (Kf == 0 || (inds && jitter)) && (Kfd == 0 || (depth && gauss)), PNR_ERR_ARG,
                "pnr_sample_bounds_backward: fine-pass inputs missing");
  if (B == 0) return PNR_OK;
  sample_bounds_bwd_kernel<<<(B + kWarpsPerBlock - 1) / kWarpsPerBlock, kWarpsPerBlock * 32, 0, (cudaStream_t)stream>>>(
      rays, steps, noise_coarse, d_z_coarse, z_coarse, z_sorted, d_z_sorted, inds, jitter, depth, gauss, d_rays, d_z_coarse_out, B, Kc,
      z_sorted ? Kf : 0, z_sorted ? Kfd : 0, (float)(1.0 / (double)Kc), depth_std, lindisp);
  PNR_CHECK_LAUNCH("sample_bounds_bwd_kernel");
  return PNR_OK;
}

extern "C" int pnr_sample_fine_depth_backward(const float* z_sorted, const float* d_z_sorted, const float* depth,
                                              const float* gauss, const float* rays, float* d_depth, int B, int K,
                                              int Kfd, float depth_std, void* stream) {
  reset_launch_count();
  PNR_REQUIRE(z_sorted && d_z_sorted && depth && gauss && rays && d_depth, PNR_ERR_ARG,
              "pnr_sample_fine_depth_backward: null pointer");
  PNR_REQUIRE(B >= 0 && K > 0 && Kfd > 0 && Kfd <= K, PNR_ERR_ARG, "pnr_sample_fine_depth_backward: bad shape");
  if (B == 0) return PNR_OK;
  sample_depth_bwd_kernel<<<(B + 3) / 4, 128, 0, (cudaStream_t)stream>>>(z_sorted, d_z_sorted, depth, gauss, rays,
                                                                         d_depth, B, K, Kfd, depth_std);
  PNR_CHECK_LAUNCH("sample_depth_bwd_kernel");
  return PNR_OK;
}

extern "C" int pnr_yolo_reduce(const float* out, float* result, int B, int K, int num_anchors, void* stream) {
  reset_launch_count();
  PNR_REQUIRE(out && result, PNR_ERR_ARG, "pnr_yolo_reduce: null pointer");
  PNR_REQUIRE(B >= 0 && K > 0 && num_anchors > 0, PNR_ERR_ARG, "pnr_yolo_reduce: bad shape");
  if (B == 0) return PNR_OK;
  const long long n = (long long)B * num_anchors;
  yolo_reduce_kernel<<<(unsigned)((n + kWarpsPerBlock - 1) / kWarpsPerBlock), kWarpsPerBlock * 32, 0, (cudaStream_t)stream>>>(
      out, result, n, K, num_anchors);
  PNR_CHECK_LAUNCH("yolo_reduce_kernel");
  return PNR_OK;
}

extern "C" int pnr_yolo_reduce_backward(const float* out, const float* d_result, float* d_out, int B, int K, int num_anchors,
                                        void* stream) {
  reset_launch_count();
  PNR_REQUIRE(out && d_result && d_out, PNR_ERR_ARG, "pnr_yolo_reduce_backward: null pointer");
  PNR_REQUIRE(B >= 0 && K > 0 && num_anchors > 0, PNR_ERR_ARG, "pnr_yolo_reduce_backward: bad shape");
  if (B == 0) return PNR_OK;
  const long long n = (long long)B * num_anchors;
  yolo_reduce_bwd_kernel<<<(unsigned)((n + kWarpsPerBlock - 1) / kWarpsPerBlock), kWarpsPerBlock * 32, 0, (cudaStream_t)stream>>>(
      out, d_result, d_out, n, K, num_anchors);
  PNR_CHECK_LAUNCH("yolo_reduce_bwd_kernel");
  return PNR_OK;
}
