// Library-level entry points: version, thread-local error string, launch counter, field dispatch.
#include "pnr_common.cuh"
#include <string.h>
#include <mutex>
#include <nvtx3/nvToolsExt.h>

namespace pnr {
static thread_local char g_err[512] = "";
static thread_local int g_launches = 0;

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches += n; }
void reset_launch_count() { g_launches = 0; }

int validate_scene_points(const pnr_scene* sc, const pnr_points* q, const char* who);
size_t field_workspace_fp32(const pnr_scene* sc, const pnr_points* q, int d_in, int H);
int field_forward_fp32(const pnr_scene* sc, const pnr_points* q, const pnr_mlp_params* mp, float* out, void* ws,
                       size_t ws_bytes, int num_freqs, float freq_factor, int raw, cudaStream_t st);
size_t field_workspace_umma();
int field_forward_umma(const pnr_scene* sc, const pnr_points* q, const pnr_mlp_params* mp, const void* packed,
                       float* out, void* ws, size_t ws_bytes, int num_freqs, float freq_factor, int raw,
                       cudaStream_t st);
}  // namespace pnr

using namespace pnr;

extern "C" int pnr_version(void) { return PNR_ABI_VERSION; }
extern "C" const char* pnr_last_error(void) { return g_err; }
extern "C" int pnr_last_launch_count(void) { return g_launches; }

extern "C" int pnr_device_supported(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { set_error("no CUDA device"); return 0; }
  int major = 0, minor = 0;
  cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
  if (major != 10) { set_error("device is sm_%d%d; this library only has sm_100a code", major, minor); return 0; }
  return 1;
}

extern "C" size_t pnr_field_workspace_bytes(const pnr_scene* scene, const pnr_points* pts, int precision) {
  if (!scene || !pts) return 0;
  if (precision == PNR_PREC_FP32) return field_workspace_fp32(scene, pts, 64, kHidden);
  if (precision == PNR_PREC_BF16) return field_workspace_umma();
  return 0;
}

extern "C" int pnr_field_forward(const pnr_scene* scene, const pnr_points* pts, const pnr_mlp_params* params,
                                 const void* packed, float* out, void* workspace, size_t workspace_bytes,
                                 int precision, int num_freqs, float freq_factor, void* stream) {
  reset_launch_count();
  int rc = validate_scene_points(scene, pts, "pnr_field_forward");
  if (rc) return rc;
  PNR_REQUIRE(params && out, PNR_ERR_ARG, "pnr_field_forward: null params/out");
  cudaStream_t st = (cudaStream_t)stream;
  const int raw = (scene->flags & PNR_SCENE_RAW_OUTPUT) ? 1 : 0;
  if (precision == PNR_PREC_FP32) {
    PNR_REQUIRE(hidden_width_supported(params->d_hidden), PNR_ERR_UNSUPPORTED,
                "pnr_field_forward: d_hidden=%d (supported: " PNR_HIDDEN_WIDTHS ")", params->d_hidden);
    return field_forward_fp32(scene, pts, params, out, workspace, workspace_bytes, num_freqs, freq_factor, raw, st);
  }
  if (precision == PNR_PREC_BF16)
    return field_forward_umma(scene, pts, params, packed, out, workspace, workspace_bytes, num_freqs, freq_factor, raw, st);
  PNR_REQUIRE(false, PNR_ERR_ARG, "pnr_field_forward: unknown precision %d", precision);
}

// ---- NeRFRenderer.forward as ONE call (src/render/nerf.py:257-309) in FOUR launches, all enqueued on `stream`:
//   field (coarse; sample_coarse folded into its point fetch) -> composite + sample_fine + sample_fine_depth + sort -> field (fine)
//   -> composite.  Every buffer is the caller's.  Results are bit-identical to the stage entry points called one by one.
namespace {
constexpr int kMaxSplits = 4;
struct RenderLayout { size_t z_c, out_c, w_c, z_f, out_f, field_ws, field_ws_each, total; int splits; };

// Small batches (one 2 048-ray shard of a 128x128 image = 14 waves of super groups over the 74 CTA pairs) lose up to one wave per
// field launch to the tail.  Rendering the batch as independent slices on forked streams lets the tail of one slice's field
// kernel overlap the head of the next slice's.  Rays are independent, so the result does not depend on the slicing.
int resolve_splits(const pnr_render_args* a) {
  if (a->n_splits == 1 || a->scene->SB != 1) return 1;
  if (a->field_events[0] || a->field_events[1] || a->field_events[2] || a->field_events[3]) return 1;   // the hooks time whole launches
  if (a->n_splits > 1) return a->n_splits < kMaxSplits ? a->n_splits : kMaxSplits;
  const int NS = a->scene->NS > 0 ? a->scene->NS : 1;
  const long long pts_per_sg = (long long)(64 / NS) * (64 / (64 / NS));      // points one CTA pair retires per super group
  const long long waves = ((long long)a->B * a->n_coarse / pts_per_sg) / 74;
  return (a->B >= 512 && waves < 48) ? 2 : 1;
}
RenderLayout render_layout(const pnr_render_args* a) {
  const size_t Bt = (size_t)a->scene->SB * a->B;
  const size_t Kc = a->n_coarse, Kf = a->n_fine > 0 ? (size_t)a->n_coarse + a->n_fine : 0;
  auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
  RenderLayout L;
  L.splits = resolve_splits(a);
  size_t off = 0;
  L.z_c = off; off = al(off + Bt * Kc * sizeof(float));
  L.out_c = off; off = al(off + Bt * Kc * 4 * sizeof(float));
  L.w_c = off; off = al(off + Bt * Kc * sizeof(float));
  L.z_f = off; off = al(off + Bt * Kf * sizeof(float));
  L.out_f = off; off = al(off + Bt * Kf * 4 * sizeof(float));
  L.field_ws_each = al(pnr::field_workspace_umma());
  L.field_ws = off; off = off + (size_t)L.splits * L.field_ws_each;
  L.total = off;
  return L;
}

// forked streams + events, created once per device (the library's only persistent resources besides tensor maps)
struct ForkCtx { cudaStream_t side[kMaxSplits - 1]; cudaEvent_t fork, join[kMaxSplits - 1]; bool ok; };
ForkCtx* fork_ctx() {
  static std::mutex mu;
  static ForkCtx table[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  std::lock_guard<std::mutex> lock(mu);
  ForkCtx* c = &table[dev];
  if (!c->ok) {
    if (cudaEventCreateWithFlags(&c->fork, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    for (int i = 0; i < kMaxSplits - 1; ++i) {
      if (cudaStreamCreateWithFlags(&c->side[i], cudaStreamNonBlocking) != cudaSuccess) return nullptr;
      if (cudaEventCreateWithFlags(&c->join[i], cudaEventDisableTiming) != cudaSuccess) return nullptr;
    }
    c->ok = true;
  }
  return c;
}

struct NvtxRange {   // the reference's record_function labels (nerf.py:181,270; models.py:163; encoder.py:89; code.py:36; resnetfc.py:141)
  int n;
  explicit NvtxRange(const char* a, const char* b = nullptr, const char* c = nullptr, const char* d = nullptr) : n(0) {
    const char* names[4] = {a, b, c, d};
    for (int i = 0; i < 4; ++i) if (names[i]) { nvtxRangePushA(names[i]); ++n; }
  }
  ~NvtxRange() { for (int i = 0; i < n; ++i) nvtxRangePop(); }
};
}  // namespace

extern "C" size_t pnr_render_workspace_bytes(const pnr_render_args* a) {
  if (!a || !a->scene || a->B < 0 || a->n_coarse <= 0 || a->n_fine < 0) return 0;
  return render_layout(a).total;
}

// one slice [r0, r1) of the flattened ray batch, on stream `st`
static int render_slice(const pnr_render_args* a, const RenderLayout& L, long long r0, long long r1, int slot, cudaStream_t st,
                        int* launches_out) {
  const int kc = a->n_coarse, kf = a->n_fine - a->n_fine_depth, kfd = a->n_fine_depth;
  const bool fine = a->n_fine > 0;
  const int n = (int)(r1 - r0);
  uint8_t* ws = (uint8_t*)a->workspace;
  float* z_c = (float*)(ws + L.z_c) + r0 * kc;
  float* out_c = (float*)(ws + L.out_c) + r0 * kc * 4;
  float* w_c = a->weights_coarse ? a->weights_coarse + r0 * kc : (float*)(ws + L.w_c) + r0 * kc;
  uint8_t* fws = ws + L.field_ws + (size_t)slot * L.field_ws_each;
  const float* rays = a->rays + r0 * 8;
  void* stream = (void*)st;
  int launches = 0, rc;
#define RSTEP(call) do { rc = (call); if (rc) return rc; launches += pnr_last_launch_count(); } while (0)
  // launch 1: the coarse field; its sample depths are computed where they are needed (point mode 2: no sample_coarse launch)
  pnr_scene sc = *a->scene;           // SB == 1 whenever the batch is sliced; otherwise the slice is the whole batch
  pnr_points pts = {};
  const int b_obj = sc.SB == 1 ? n : a->B;
  pts.rays = rays; pts.mode = 2; pts.K = kc; pts.P = b_obj * kc; pts.total = (long long)n * kc;
  pts.steps = a->steps; pts.noise = a->noise_coarse + r0 * kc; pts.step = (float)(1.0 / (double)kc); pts.lindisp = a->lindisp;
  auto mark = [&](int i) { if (a->field_events[i]) cudaEventRecord((cudaEvent_t)a->field_events[i], st); };
  mark(0);
  {
    NvtxRange r("model_inference", "encoder_index", "positional_enc", "resnetfc_infer");
    RSTEP(pnr_field_forward(&sc, &pts, a->mlp_coarse, a->packed_coarse, out_c, fws, L.field_ws_each, PNR_PREC_BF16, a->num_freqs,
                            a->freq_factor, stream));
  }
  mark(1);
  // launch 2: composite of the coarse pass + sample_fine + sample_fine_depth + sort (nerf.py:229-255, 290-301)
  const int K = kc + a->n_fine;
  float* z_f = fine ? (float*)(ws + L.z_f) + r0 * K : nullptr;
  {
    NvtxRange r("renderer_composite");
    RSTEP(pnr_composite_resample(out_c, rays, a->steps, a->noise_coarse + r0 * kc, fine && kf > 0 ? a->noise_u + r0 * kf : nullptr,
                                 fine && kf > 0 ? a->noise_jitter + r0 * kf : nullptr, fine && kfd > 0 ? a->noise_gauss + r0 * kfd : nullptr,
                                 z_c, w_c, a->rgb_coarse + r0 * 3, a->depth_coarse + r0, z_f, n, kc, fine ? kf : 0, fine ? kfd : 0,
                                 a->depth_std, a->white_bkgd, a->lindisp, stream));
  }
  if (fine) {
    float* out_f = (float*)(ws + L.out_f) + r0 * K * 4;
    pnr_scene scf = a->scene_fine ? *a->scene_fine : *a->scene;
    pts.mode = 1; pts.z = z_f; pts.K = K; pts.P = b_obj * K; pts.total = (long long)n * K;
    const pnr_mlp_params* mf = a->mlp_fine ? a->mlp_fine : a->mlp_coarse;          // models.py:291: no fine network -> coarse
    const void* pf = a->mlp_fine ? a->packed_fine : a->packed_coarse;
    mark(2);
    {
      NvtxRange r("model_inference", "encoder_index", "positional_enc", "resnetfc_infer");
      RSTEP(pnr_field_forward(&scf, &pts, mf, pf, out_f, fws, L.field_ws_each, PNR_PREC_BF16, a->num_freqs, a->freq_factor, stream));
    }
    mark(3);
    NvtxRange r("renderer_composite");
    RSTEP(pnr_composite(out_f, z_f, rays, a->weights_fine ? a->weights_fine + r0 * K : nullptr, a->rgb_fine + r0 * 3,
                        a->depth_fine + r0, n, K, a->white_bkgd, stream));
  }
#undef RSTEP
  *launches_out += launches;
  return PNR_OK;
}

extern "C" int pnr_render_forward(const pnr_render_args* a, void* stream) {
  reset_launch_count();
  PNR_REQUIRE(a && a->scene && a->rays && a->steps && a->noise_coarse && a->mlp_coarse && a->packed_coarse, PNR_ERR_ARG,
              "pnr_render_forward: null pointer");
  PNR_REQUIRE(a->rgb_coarse && a->depth_coarse, PNR_ERR_ARG, "pnr_render_forward: coarse outputs missing");
  PNR_REQUIRE(a->precision == PNR_PREC_BF16, PNR_ERR_UNSUPPORTED, "pnr_render_forward: the single-call render is the bf16 tensor-core path");
  PNR_REQUIRE(a->B >= 0 && a->n_coarse > 0 && a->n_fine >= 0 && a->n_fine_depth >= 0 && a->n_fine_depth <= a->n_fine, PNR_ERR_ARG,
              "pnr_render_forward: bad sample counts");
  const int kf = a->n_fine - a->n_fine_depth, kfd = a->n_fine_depth;
  const bool fine = a->n_fine > 0;
  if (fine) {
    PNR_REQUIRE(a->rgb_fine && a->depth_fine, PNR_ERR_ARG, "pnr_render_forward: fine outputs missing");
    PNR_REQUIRE((kf == 0 || (a->noise_u && a->noise_jitter)) && (kfd == 0 || a->noise_gauss), PNR_ERR_ARG,
                "pnr_render_forward: fine-pass noise missing");
    PNR_REQUIRE(a->mlp_fine == nullptr || a->packed_fine, PNR_ERR_ARG, "pnr_render_forward: packed fine weights missing");
    PNR_REQUIRE(!a->scene_fine || (a->scene_fine->SB == a->scene->SB && a->scene_fine->NS == a->scene->NS), PNR_ERR_ARG,
                "pnr_render_forward: scene_fine and scene disagree on SB / NS");
  }
  const long long Bt_ll = (long long)a->scene->SB * a->B;
  PNR_REQUIRE(a->total_rays == Bt_ll, PNR_ERR_ARG,
              "pnr_render_forward: the ray buffers hold %lld rays but the scene has SB=%d objects x B=%d rays (encode() and the ray batch disagree?)",
              (long long)a->total_rays, a->scene->SB, a->B);
  const RenderLayout L = render_layout(a);
  PNR_REQUIRE(a->workspace && a->workspace_bytes >= L.total && ((uintptr_t)a->workspace & 255) == 0, PNR_ERR_ARG,
              "pnr_render_forward: workspace of pnr_render_workspace_bytes() = %zu bytes (256-byte aligned) required", L.total);
  PNR_REQUIRE(Bt_ll < (1LL << 31), PNR_ERR_ARG, "pnr_render_forward: too many rays");
  if (Bt_ll == 0) return PNR_OK;
  NvtxRange whole("renderer_forward");
  cudaStream_t st = (cudaStream_t)stream;
  int launches = 0, rc;
  if (L.splits <= 1) {
    rc = render_slice(a, L, 0, Bt_ll, 0, st, &launches);
    if (rc) return rc;
  } else {
    ForkCtx* fc = fork_ctx();
    PNR_REQUIRE(fc, PNR_ERR_CUDA, "pnr_render_forward: could not create the forked streams");
    PNR_REQUIRE(cudaEventRecord(fc->fork, st) == cudaSuccess, PNR_ERR_CUDA, "pnr_render_forward: cudaEventRecord(fork)");
    long long r0 = 0;
    for (int s = 0; s < L.splits; ++s) {
      long long r1 = s + 1 == L.splits ? Bt_ll : ((Bt_ll * (s + 1) / L.splits) + 31) / 32 * 32;
      if (r1 > Bt_ll) r1 = Bt_ll;
      cudaStream_t ss = s == 0 ? st : fc->side[s - 1];
      if (s > 0) cudaStreamWaitEvent(ss, fc->fork, 0);
      if (r1 > r0) { rc = render_slice(a, L, r0, r1, s, ss, &launches); if (rc) return rc; }
      if (s > 0) { cudaEventRecord(fc->join[s - 1], ss); cudaStreamWaitEvent(st, fc->join[s - 1], 0); }
      r0 = r1;
    }
    PNR_REQUIRE(cudaGetLastError() == cudaSuccess, PNR_ERR_CUDA, "pnr_render_forward: stream fork/join failed");
  }
  reset_launch_count();
  count_launch(launches);
  return PNR_OK;
}
