// Host side of the tcgen05 field path: packed-weight blob layout (bias tables + the CTA-pair weight stream of
// mlp_umma_pair.cu), pnr_mlp_pack*, and the dispatch of pnr_field_forward(PNR_PREC_BF16) to pair::field_pair_kernel.
// ResnetFC parameters: src/model/resnetfc.py:103-132; the op replaced: PixelNeRFNet.forward, src/model/models.py:153-318.
#include "pnr_common.cuh"
#include "umma.cuh"
#include <stdlib.h>

namespace pnr {
using namespace umma;

int validate_scene_points(const pnr_scene* sc, const pnr_points* q, const char* who);

constexpr uint32_t kPackMagic = 0x504e5233u; // "PNR3"
constexpr size_t kPackHeader = 1024;

struct Sched {
  int n_blocks;   // ResnetFC blocks
  int CL;         // block index before which the views are pooled (combine_layer); == n_blocks: no pooling (NS == 1 only)
  int n_linz;     // min(combine_layer, n_blocks)
  int KBz;        // d_latent / 64
};

// CTA-pair kernel (mlp_umma_pair.cu)
size_t pair_stream_bytes(const pnr_mlp_params* p, int proj);
int pair_stages(const pnr_mlp_params* p, int proj);
int pair_pack(const pnr_mlp_params* p, uint8_t* stream, int proj, cudaStream_t st);
size_t pair_workspace_bytes();
int field_forward_pair(const pnr_scene* sc, const pnr_points* q, const pnr_mlp_params* mp, const uint8_t* stream,
                       const float* bx, const float* bh, const float* bo, float* out, void* ws, size_t ws_bytes,
                       int num_freqs, float freq_factor, int raw, int proj, cudaStream_t st);

// blob = 1 KiB header | cumulative x biases (n_blocks + 1) x 512 | fc_0 biases n_blocks x 512 | lin_out bias (128) | pair stream
// The bias tables keep a 512-feature stride whatever d_hidden is; entries at and past d_hidden are zero (the padding to Hp).
// header: magic, d_in, d_latent, d_hidden, d_out, n_blocks, combine_layer, stages, Hp
struct PackOffsets { size_t bias_x, bias_h, bias_out, pair_stream, total; };
static PackOffsets pack_offsets(const Sched& s, const pnr_mlp_params* p, int proj = 0) {
  PackOffsets o;
  o.bias_x = kPackHeader;
  o.bias_h = o.bias_x + (size_t)(s.n_blocks + 1) * kHidden * sizeof(float);
  o.bias_out = o.bias_h + (size_t)s.n_blocks * kHidden * sizeof(float);
  o.pair_stream = (o.bias_out + 128 * sizeof(float) + 1023) & ~(size_t)1023;
  o.total = o.pair_stream + pair_stream_bytes(p, proj);
  return o;
}

__global__ void pack_bias_kernel(pnr_mlp_params mp, Sched sc, int n_stages, float* __restrict__ bias_x, float* __restrict__ bias_h,
                                 float* __restrict__ bias_out, uint32_t* __restrict__ header) {
  const int f = threadIdx.x;   // 512 threads
  const bool live = f < mp.d_hidden;               // padded features: every bias 0
  float cum = live ? mp.lin_in_b[f] + (sc.n_linz > 0 ? mp.linz_b[0][f] : 0.f) : 0.f;
  bias_x[f] = cum;
  for (int e = 1; e <= sc.n_blocks; ++e) {
    if (e - 1 == sc.CL) cum = 0.f;                 // the view-mean epilogue materialises the bias into TMEM
    if (live) cum += mp.fc1_b[e - 1][f] + (e < sc.n_linz ? mp.linz_b[e][f] : 0.f);
    bias_x[e * kHidden + f] = cum;
  }
  for (int b = 0; b < sc.n_blocks; ++b) bias_h[b * kHidden + f] = live ? mp.fc0_b[b][f] : 0.f;
  if (f < 128) bias_out[f] = f < mp.d_out ? mp.lin_out_b[f] : 0.f;
  if (f == 0) {
    header[0] = kPackMagic; header[1] = mp.d_in; header[2] = mp.d_latent; header[3] = mp.d_hidden;
    header[4] = mp.d_out; header[5] = mp.n_blocks; header[6] = mp.combine_layer; header[7] = n_stages;
    header[8] = mp.d_hidden <= 256 ? 256 : 512;
  }
}

static int make_sched(const pnr_mlp_params* p, Sched* s, const char* who) {
  PNR_REQUIRE(p, PNR_ERR_ARG, "%s: null params", who);
  PNR_REQUIRE(hidden_width_supported(p->d_hidden), PNR_ERR_UNSUPPORTED, "%s: d_hidden=%d (supported: " PNR_HIDDEN_WIDTHS ")", who,
              p->d_hidden);
  PNR_REQUIRE(p->d_in > 0 && p->d_in <= 64, PNR_ERR_UNSUPPORTED, "%s: d_in=%d must be in (0,64]", who, p->d_in);
  PNR_REQUIRE(p->d_latent > 0 && p->d_latent % 64 == 0, PNR_ERR_UNSUPPORTED, "%s: d_latent=%d must be a positive multiple of 64", who, p->d_latent);
  PNR_REQUIRE(p->n_blocks >= 1 && p->n_blocks <= 8, PNR_ERR_UNSUPPORTED, "%s: n_blocks=%d", who, p->n_blocks);
  PNR_REQUIRE(p->combine_layer >= 1 && p->combine_layer <= p->n_blocks, PNR_ERR_ARG,
              "%s: combine_layer=%d (pass min(combine_layer, n_blocks))", who, p->combine_layer);
  PNR_REQUIRE(p->combine_type == PNR_COMBINE_AVERAGE || p->combine_type == PNR_COMBINE_MAX, PNR_ERR_ARG,
              "%s: combine_type=%d", who, p->combine_type);
  PNR_REQUIRE(p->d_out >= 1 && p->d_out <= 32, PNR_ERR_UNSUPPORTED, "%s: d_out=%d", who, p->d_out);
  s->n_blocks = p->n_blocks; s->CL = p->combine_layer; s->n_linz = p->combine_layer; s->KBz = p->d_latent / 64;
  return PNR_OK;
}

size_t field_workspace_umma() { return pair_workspace_bytes(); }

int field_forward_umma(const pnr_scene* sc, const pnr_points* q, const pnr_mlp_params* mp, const void* packed,
                       float* out, void* ws, size_t ws_bytes, int num_freqs, float freq_factor, int raw,
                       cudaStream_t st) {
  Sched sch;
  int rc = make_sched(mp, &sch, "field_forward_umma");
  if (rc) return rc;
  PNR_REQUIRE(packed, PNR_ERR_ARG, "field_forward_umma: packed weights missing (call pnr_mlp_pack)");
  PNR_REQUIRE(((uintptr_t)packed & 1023) == 0, PNR_ERR_ARG, "field_forward_umma: packed blob must be 1024-byte aligned");
  PNR_REQUIRE(!sc->feat_fp32, PNR_ERR_ARG, "field_forward_umma: needs bf16 channels-last feature maps");
  const int proj = (sc->flags & PNR_SCENE_PROJECTED) ? 1 : 0;
  if (proj) {
    PNR_REQUIRE(sc->C == sch.n_linz * mp->d_hidden, PNR_ERR_ARG,
                "field_forward_umma: projected maps must have n_linz x d_hidden = %d x %d = %d channels (got %d)", sch.n_linz,
                mp->d_hidden, sch.n_linz * mp->d_hidden, sc->C);
    sch.KBz = mp->d_hidden / 64;         // blob from pnr_mlp_pack_projected: identity lin_z over d_hidden channels
  } else {
    PNR_REQUIRE(sc->C == mp->d_latent, PNR_ERR_ARG, "field_forward_umma: feature maps have %d channels, the MLP expects %d", sc->C, mp->d_latent);
  }
  PNR_REQUIRE(mp->d_in == 6 * num_freqs + 6, PNR_ERR_ARG, "field_forward_umma: d_in/num_freqs mismatch");
  PNR_REQUIRE(sc->NS >= 1 && sc->NS <= 8 && sc->NS != 7, PNR_ERR_UNSUPPORTED, "field_forward_umma: NS=%d source views", sc->NS);
  PNR_REQUIRE(mp->combine_layer < mp->n_blocks || sc->NS == 1, PNR_ERR_UNSUPPORTED,
              "field_forward_umma: combine_layer >= n_blocks never pools the views; only valid with one source view");
  if ((long long)sc->SB * q->P == 0) return PNR_OK;
  const PackOffsets po = pack_offsets(sch, mp, proj);
  const uint8_t* blob = (const uint8_t*)packed;
  return field_forward_pair(sc, q, mp, blob + po.pair_stream, (const float*)(blob + po.bias_x), (const float*)(blob + po.bias_h),
                            (const float*)(blob + po.bias_out), out, ws, ws_bytes, num_freqs, freq_factor, raw, proj, st);
}

}  // namespace pnr

using namespace pnr;

static size_t mlp_pack_bytes(const pnr_mlp_params* p, int proj) {
  Sched s;
  if (make_sched(p, &s, "pnr_mlp_pack_bytes")) return 0;
  if (proj) s.KBz = p->d_hidden / 64;
  return pack_offsets(s, p, proj).total;
}
extern "C" size_t pnr_mlp_pack_bytes(const pnr_mlp_params* p) { return mlp_pack_bytes(p, 0); }
extern "C" size_t pnr_mlp_pack_projected_bytes(const pnr_mlp_params* p) { return mlp_pack_bytes(p, 1); }

static int mlp_pack(const pnr_mlp_params* p, void* packed, int proj, void* stream) {
  reset_launch_count();
  Sched s;
  int rc = make_sched(p, &s, "pnr_mlp_pack");
  if (rc) return rc;
  if (proj) s.KBz = p->d_hidden / 64;
  PNR_REQUIRE(packed && ((uintptr_t)packed & 1023) == 0, PNR_ERR_ARG, "pnr_mlp_pack: packed must be non-null and 1024-byte aligned");
  PNR_REQUIRE(p->lin_in_w && p->lin_in_b && p->lin_out_w && p->lin_out_b, PNR_ERR_ARG, "pnr_mlp_pack: null lin_in/lin_out");
  for (int b = 0; b < p->n_blocks; ++b)
    PNR_REQUIRE(p->fc0_w[b] && p->fc0_b[b] && p->fc1_w[b] && p->fc1_b[b], PNR_ERR_ARG, "pnr_mlp_pack: null block %d", b);
  for (int b = 0; b < s.n_linz; ++b) PNR_REQUIRE(p->linz_w[b] && p->linz_b[b], PNR_ERR_ARG, "pnr_mlp_pack: null lin_z %d", b);
  const PackOffsets po = pack_offsets(s, p, proj);
  uint8_t* blob = (uint8_t*)packed;
  cudaStream_t st = (cudaStream_t)stream;
  rc = pair_pack(p, blob + po.pair_stream, proj, st);
  if (rc) return rc;
  pack_bias_kernel<<<1, kHidden, 0, st>>>(*p, s, pair_stages(p, proj), (float*)(blob + po.bias_x), (float*)(blob + po.bias_h),
                                          (float*)(blob + po.bias_out), (uint32_t*)blob);
  PNR_CHECK_LAUNCH("pack_bias_kernel");
  return PNR_OK;
}
extern "C" int pnr_mlp_pack(const pnr_mlp_params* p, void* packed, void* stream) { return mlp_pack(p, packed, 0, stream); }
extern "C" int pnr_mlp_pack_projected(const pnr_mlp_params* p, void* packed, void* stream) { return mlp_pack(p, packed, 1, stream); }
