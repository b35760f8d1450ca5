/*
 * pixelnerf_b200.h -- C ABI of the B200-native pixelNeRF-YOLO rendering hot path.
 *
 * The reference (kofinandi/pixel-nerf-yolo) is pure Python/PyTorch and has no FFI layer: the seam is
 * its class API (NeRFRenderer.forward src/render/nerf.py:257-309, PixelNeRFNet.encode/forward
 * src/model/models.py:92-318).  The drop-in Python classes in pixel-nerf-yolo_b200/ keep that API and
 * call the entry points below through ctypes; INTEGRATION.md shows the binding.  Each entry point
 * names the reference code it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (torch caching allocator) unless noted;
 *   - every call only enqueues work on `stream` (a cudaStream_t passed as void*), no host sync;
 *   - return value 0 = ok, negative = error; pnr_last_error() gives the thread-local message;
 *   - no global state, re-entrant, callable from several host threads on different devices
 *     (the reference's DataParallel runs one Python thread per GPU, src/render/nerf.py:373-377).
 */
#ifndef PIXELNERF_B200_H
#define PIXELNERF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PNR_ABI_VERSION 3

/* precision of the field function (PixelNeRFNet.forward) */
#define PNR_PREC_FP32 0 /* SIMT fp32 operands + fp32 accumulate: the <=1e-4 "accumulate-only" check build */
#define PNR_PREC_BF16 1 /* tcgen05 bf16 operands, fp32 accumulate in TMEM: the production path      */

/* error codes */
#define PNR_OK 0
#define PNR_ERR_ARG (-1)      /* bad shape / null pointer / unsupported option            */
#define PNR_ERR_CUDA (-2)     /* CUDA runtime error at enqueue time                        */
#define PNR_ERR_UNSUPPORTED (-3) /* valid reference option that this build does not cover */

/* State left behind by PixelNeRFNet.encode (src/model/models.py:92-151) plus the encoder output
 * (SpatialEncoder.latent / latent_scaling, src/model/encoder.py:138-172), re-laid out for the GPU:
 * feature maps are channels-last so one bilinear tap is one contiguous C-vector. */
typedef struct pnr_scene {
  const void* feat;    /* (SB*NS, Hl, Wl, C) channels-last; bf16 (feat_fp32=0) or fp32 (feat_fp32=1) */
  const float* poses;  /* (SB*NS, 3, 4) world->camera [R^T | -R^T t]   models.py:116-118           */
  const float* focal;  /* (SB*NS, 2) per view, fy already negated       models.py:126-137,225-227   */
  const float* center; /* (SB*NS, 2) per view principal point           models.py:139-148,228-230   */
  int32_t SB;          /* objects ("super batch")                                                   */
  int32_t NS;          /* source views per object                                                   */
  int32_t C;           /* latent channels (512 resnet34 x4 levels, 1792 YOLO backbone)              */
  int32_t Hl, Wl;      /* feature-map size                                                          */
  int32_t feat_fp32;   /* 0: bf16 maps, 1: fp32 maps                                                */
  float image_w, image_h;          /* PixelNeRFNet.image_shape  models.py:122-123                   */
  float lat_scale_x, lat_scale_y;  /* SpatialEncoder.latent_scaling  encoder.py:170-172             */
  int32_t flags;       /* PNR_SCENE_* bits                                                          */
} pnr_scene;

/* YOLO mode of PixelNeRFNet.forward (models.py:221-224, 254-264): the latent of a (point, view) row is zeroed where the
 * point's camera-space z is >= 0.  (The mode's other differences are data: poses are used as given and the focal
 * signs differ, models.py:119-120,136-137,220-222 -- the caller passes focal with the sign that makes
 * uv = -xy / z * focal + c come out right.) */
#define PNR_SCENE_MASK_NONNEG_Z 1
/* pnr_field_forward returns the raw lin_out values instead of [sigmoid(rgb), relu(sigma)] (models.py:309-310). */
#define PNR_SCENE_RAW_OUTPUT 2
/* `feat` holds the lin_z PRE-PROJECTIONS of the encoder output (pnr_project_features): n_linz x d_hidden channels (the
 * unpadded width, whatever width the packed network is padded to), slice b = latent . lin_z[b].weight^T.  pnr_field_forward
 * checks C == n_linz * d_hidden.  Bilinear interpolation and lin_z are both linear, so lin_z[b](gather(latent)) ==
 * gather(slice b) (+ bias); the kernel then accumulates the gathered slice with an identity weight instead of streaming a
 * d_latent-wide lin_z.  For wide latents (1 792-channel YOLO backbone maps) this removes 3/4 of the gather traffic and 45 % of
 * the weight stages.  Needs `packed` from pnr_mlp_pack_projected.  bf16 tcgen05 path only. */
#define PNR_SCENE_PROJECTED 4
/* Training path only (pnr_field_forward_train / pnr_field_backward): run the GEMMs on the tensor cores with TF32 operands
 * (10-bit mantissa) and fp32 accumulation instead of fp32 SIMT arithmetic: ~3x faster, gradients within ~5e-3 of autograd
 * instead of ~1e-4. */
#define PNR_SCENE_TRAIN_TF32 8
/* Training path only: the tcgen05 path -- bf16 operands (activations kept on a bf16 tape, 1 KiB per row and layer), fp32
 * accumulation in TMEM, cta_group::2 GEMMs for the forward layers, the input gradients and the weight gradients
 * (csrc/train_umma.cu).  Gradients within ~2e-2 of autograd (bf16 operand rounding).  C a multiple of 64. */
#define PNR_SCENE_TRAIN_BF16 16
/* z-feature layout: the non-latent part of each MLP input row, as PixelNeRFNet's switches shape it (models.py:16-90,
 * 183-209).  All bits clear is the layout of every shipped conf: [PE(R x) (3 + 6 num_freqs), R d (3)].  In general, with
 * x_rot = R x and x_cam = R x + t of the source view:
 *   u  = x_rot (x_cam with CAM_COORDS), or the one value -u_z with Z_ONLY;  u ++= R d with CODE_VIEWDIRS (unless NO_VIEWDIRS);
 *   zf = PE(u) = [u (unless NO_CODE_INPUT), sin(f_0 u), cos(f_0 u), sin(f_1 u), ...], or u itself with NO_CODE;
 *   zf ++= R d unless NO_VIEWDIRS or CODE_VIEWDIRS.
 * Its width is pnr_zfeat_width(flags, num_freqs); every field, gather and training entry point requires d_in to equal it. */
#define PNR_SCENE_ZF_NO_VIEWDIRS 32      /* use_viewdirs = False                                                       */
#define PNR_SCENE_ZF_CODE_VIEWDIRS 64    /* use_code_viewdirs = True: R d goes through the positional encoding          */
#define PNR_SCENE_ZF_CAM_COORDS 128      /* normalize_z = False: camera coordinates R x + t instead of R x             */
#define PNR_SCENE_ZF_Z_ONLY 256          /* use_xyz = False: the single coordinate -z                                  */
#define PNR_SCENE_ZF_NO_CODE 512         /* use_code = False: no positional encoding                                   */
#define PNR_SCENE_ZF_NO_CODE_INPUT 1024  /* code.include_input = False: the encoding drops its raw input columns        */

/* Where the query points of a field evaluation come from. */
typedef struct pnr_points {
  const float* xyz;   /* mode 0: (SB, P, 3) world points   (PixelNeRFNet.forward argument)          */
  const float* dirs;  /* mode 0: (SB, P, 3) view directions                                          */
  const float* rays;  /* mode 1: (SB*B, 8) [o, d, near, far]; point (b,k) = o + z[b,k] d             */
  const float* z;     /* mode 1: (SB*B, K) sample depths       (nerf.py:191,208-212)                 */
  int32_t mode;       /* 0 explicit points, 1 rays x depths, 2 rays x coarse depths computed on the fly      */
  int32_t P;          /* points per object (mode 1: B*K)                                             */
  int32_t K;          /* mode 1: samples per ray                                                     */
  int64_t total;      /* points the buffers above hold in all (xyz: total x 3, z: total); every entry point  */
                      /* requires total == scene->SB * P, so a scene encoded for more objects than the       */
                      /* caller's batch cannot run past the buffers                                           */
  /* mode 2: z[b,k] = sample_coarse (nerf.py:104-124) evaluated where it is needed -- bit-identical to pnr_sample_coarse, */
  /* no depth buffer and no separate launch: steps = linspace(0, 1 - 1/K, K), noise (SB*B, K) in [0,1), step = 1/K       */
  const float* steps; const float* noise; float step; int32_t lindisp;
} pnr_points;

/* ---- library ---------------------------------------------------------------------------------- */
int pnr_version(void);
const char* pnr_last_error(void);
/* 1 if the current device is sm_100 (the only target this library has code for). */
int pnr_device_supported(void);

/* ---- ray tile: sampling / compositing / resampling (src/render/nerf.py) ------------------------- */
/* sample_coarse, nerf.py:104-124.  steps = torch.linspace(0, 1-1/Kc, Kc) (passed in so that schedules
 * with non power-of-two Kc stay bit-exact), noise (B,Kc) in [0,1).  z (B,Kc). */
int pnr_sample_coarse(const float* rays, const float* steps, const float* noise, float* z,
                      int B, int Kc, int lindisp, void* stream);

/* composite, nerf.py:184-188 (deltas) + 229-255 (alpha, transmittance, weights, rgb, depth, white
 * background).  rgb_sigma (B,K,4) = model output [r,g,b,sigma]; weights may be NULL. */
int pnr_composite(const float* rgb_sigma, const float* z, const float* rays, float* weights,
                  float* rgb, float* depth, int B, int K, int white_bkgd, void* stream);

/* sample_fine (nerf.py:126-154) + sample_fine_depth (nerf.py:156-167) + cat/sort (nerf.py:300-301).
 * weights (B,Kc) and depth (B) are the coarse composite outputs; u, jitter (B,Kf) and gauss (B,Kfd)
 * the three noise draws.  z_out (B, Kc+Kf+Kfd) sorted ascending.  Optional debug outputs:
 * inds_out (B,Kf) int32 searchsorted bins, z_fine_out (B,Kf), z_depth_out (B,Kfd) (may be NULL). */
int pnr_sample_fine(const float* weights, const float* depth, const float* rays, const float* z_coarse,
                    const float* u, const float* jitter, const float* gauss, float* z_out,
                    int32_t* inds_out, float* z_fine_out, float* z_depth_out, int B, int Kc, int Kf,
                    int Kfd, float depth_std, int lindisp, void* stream);

/* composite of the coarse pass + the whole resampling step in ONE launch (what pnr_render_forward enqueues between the two field
 * launches): z_coarse is recomputed from (rays, steps, noise_coarse) exactly as pnr_sample_coarse does and written to z_coarse_out,
 * then pnr_composite and pnr_sample_fine run back to back in the same warp.  weights_coarse (B,Kc) is written (the importance
 * sampler reads it); with n_fine == 0 only the composite part runs. */
int pnr_composite_resample(const float* rgb_sigma, const float* rays, const float* steps, const float* noise_coarse, const float* u,
                           const float* jitter, const float* gauss, float* z_coarse_out, float* weights_coarse, float* rgb_coarse,
                           float* depth_coarse, float* z_fine_out, int B, int Kc, int Kf, int Kfd, float depth_std, int white_bkgd,
                           int lindisp, void* stream);

/* YoloRenderer.forward's per-ray reduction (src/render/yolo.py:96-114): raw field values out (B, K, A*7) ->
 * result (B, A, 7) = [max_k p, sum_k(v p) / (sum_k p + 1e-5)], p = sigmoid(first value of the anchor). */
int pnr_yolo_reduce(const float* out, float* result, int B, int K, int num_anchors, void* stream);

/* Backward of pnr_yolo_reduce (what autograd derives for yolo.py:96-114; torch.max sends its gradient to the first maximal
 * sample): out (B, K, A*7) raw field values, d_result (B, A, 7) -> d_out (B, K, A*7), overwritten. */
int pnr_yolo_reduce_backward(const float* out, const float* d_result, float* d_out, int B, int K, int num_anchors, void* stream);

/* ---- encode-side repack (SpatialEncoder.latent NCHW fp32 -> channels-last) ---------------------- */
/* src (N, C, H, W) fp32 -> dst (N, H, W, C) bf16 (to_fp32=0) or fp32 (to_fp32=1). */
int pnr_pack_features(const float* src, void* dst, int N, int C, int H, int W, int to_fp32, void* stream);

/* SpatialEncoder.forward's tail in one pass (src/model/encoder.py:159-168): every pyramid level (N, C_l, H_l, W_l) fp32 is
 * upsampled bilinearly (align_corners=True) to level 0's size, concatenated along channels and written channels-last:
 * dst (N, H_0, W_0, sum C_l) bf16 (to_fp32=0) or fp32.  `levels` is a HOST array of n_levels (<= 8) device pointers. */
int pnr_pyramid_pack(const float* const* levels, const int32_t* level_C, const int32_t* level_H, const int32_t* level_W,
                     int n_levels, int N, void* dst, int to_fp32, void* stream);

/* ---- ray generation (src/util/util.py:115-145 unproj_map, 240-278 gen_rays) --------------------------------- */
/* poses (N, 4, 4) camera-to-world -> rays [origin(3), dir(3), near, far].  pix_inds == NULL: all N*H*W pixels, rays
 * (N, H, W, 8), n_out = N*H*W.  Otherwise pix_inds (n_out) int64 flat indices into (N, H, W) (the trainer's ray
 * sampling, PixelNerfTrainer.py:100-117) and rays (n_out, 8). */
int pnr_gen_rays(const float* poses, const long long* pix_inds, float* rays, long long n_out, int N, int H, int W,
                 float fx, float fy, float cx, float cy, float z_near, float z_far, void* stream);

/* util.gen_rays_yolo (src/util/util.py:808-876): rays through the cell centres (+0.49) of a W x H detection grid for N
 * cameras given as world-to-camera extrinsics.  inv_intr (3,3) and inv_extr (N,4,4) are the inverses the reference computes with
 * torch.inverse (the caller does the same on the host side; a 3x3 / 4x4 inverse is not kernel work); rays (N, H, W, 8) =
 * [origin = inv_extr[:3,3], dir = inv_extr[:3,:3] . (inv_intr . [x+0.49, y+0.49, 1]) (NOT normalised), z_near, z_far]. */
int pnr_gen_rays_yolo(const float* inv_intr, const float* inv_extr, float* rays, int N, int H, int W, float z_near,
                      float z_far, void* stream);

/* ---- output side ------------------------------------------------------------------------------------------- */
/* eval/eval.py:283-290: rgb (B,3) -> rgb_u8 (B,3) = uint8(clamp(rgb,0,1)*255); depth (B) -> depth_norm (B) =
 * (depth - z_near) / (z_far - z_near).  Either output may be NULL. */
int pnr_image_output(const float* rgb, const float* depth, uint8_t* rgb_u8, float* depth_norm, long long B,
                     float z_near, float z_far, void* stream);
/* train/trainlib/PixelNerfTrainer.py:147-157 with src/model/loss.py:92-104 (MSELoss, or L1Loss when use_l1): adds
 * mean((rgb - gt)^2) (or mean |rgb - gt|) over n values to *loss (caller zeroes it) and, if d_rgb is non-NULL, writes
 * d loss / d rgb (n). */
int pnr_rgb_loss(const float* rgb, const float* gt, float* loss, float* d_rgb, long long n, int use_l1, void* stream);

/* ---- project + 4-tap gather + positional encoding, stand-alone ---------------------------------- */
/* models.py:168-230 + encoder.py:79-108 + code.py:30-42.  For every (object, view, point) row
 * r = (s*NS + v)*P + p writes latent_out[r, 0:C] (bf16 if out_fp32=0 else fp32) and zfeat_out[r, 0:W] fp32, the z-feature in
 * the layout of the scene's PNR_SCENE_ZF_* bits, W = pnr_zfeat_width(scene->flags, num_freqs) (default: [PE(R x) (39),
 * R d (3)] at 6 frequencies).  Either output may be NULL. */
int pnr_gather_encode(const pnr_scene* scene, const pnr_points* pts, void* latent_out, float* zfeat_out,
                      int out_fp32, int num_freqs, float freq_factor, void* stream);

/* Width of the z-feature (PixelNeRFNet's d_in) that the PNR_SCENE_ZF_* bits of `flags` give at num_freqs frequencies
 * (num_freqs is ignored with PNR_SCENE_ZF_NO_CODE).  Default layout: 6 * num_freqs + 6.  Host function, no device work. */
int pnr_zfeat_width(int flags, int num_freqs);

/* PositionalEncoding.forward as a stand-alone operator (src/model/code.py:30-42):
 * x (n, d) -> out (n, d * (2*num_freqs + include_input)) = [x, sin(f0 x), cos(f0 x), sin(f1 x), ...]. */
int pnr_positional_encoding(const float* x, float* out, long long n, int d, int num_freqs,
                            float freq_factor, int include_input, void* stream);

/* SpatialEncoder.index as a stand-alone operator (src/model/encoder.py:79-108), bilinear,
 * align_corners=True, zero padding.  uv (uv_views, P, 2) pixel coordinates with uv_views == 1 (broadcast)
 * or SB*NS; out (SB*NS, C, P) fp32 in the reference's layout.  Only feat, SB, NS, C, Hl, Wl, feat_fp32,
 * image_*, lat_scale_* of the scene are used. */
int pnr_index_features(const pnr_scene* scene, const float* uv, int uv_views, int P, float* out, void* stream);

/* ---- ResnetFC weights (src/model/resnetfc.py:103-132) ------------------------------------------- */
/* View pooling of ResnetFC (combine_type, resnetfc.py:172-174, util.combine_interleaved util.py:489-499): the NS source views of
 * a point are reduced before block combine_layer by their mean or by their elementwise max. */
#define PNR_COMBINE_AVERAGE 0
#define PNR_COMBINE_MAX 1

/* fp32 parameters of one ResnetFC in state_dict order; all device pointers. */
typedef struct pnr_mlp_params {
  const float* lin_in_w;  const float* lin_in_b;     /* (H, d_in), (H)                 */
  const float* lin_out_w; const float* lin_out_b;    /* (d_out, H), (d_out)            */
  const float* fc0_w[8];  const float* fc0_b[8];     /* blocks.i.fc_0  (H,H),(H)       */
  const float* fc1_w[8];  const float* fc1_b[8];     /* blocks.i.fc_1  (H,H),(H)       */
  const float* linz_w[8]; const float* linz_b[8];    /* lin_z.i  (H, d_latent),(H)     */
  /* combine_layer = min(combine_layer, n_blocks): the views are pooled before block combine_layer; combine_layer == n_blocks
   * never pools (the single-view network of conf/default.conf), which is only defined for NS == 1 */
  /* d_hidden: a multiple of 64 from 64 to 512 on every path; the tcgen05 inference path packs the network zero-padded to
   * 256 (d_hidden <= 256) or 512 features.  Other widths: PNR_ERR_UNSUPPORTED at the first pack or field call. */
  int32_t d_in, d_latent, d_hidden, d_out, n_blocks, combine_layer;
  int32_t combine_type;                              /* PNR_COMBINE_*; the packed weight stream does not depend on it */
} pnr_mlp_params;

/* Bytes of the packed bf16 weight stream + fp32 bias tables for the tcgen05 path. */
size_t pnr_mlp_pack_bytes(const pnr_mlp_params* p);
/* Build the packed blob (device, caller-allocated, 1024-byte aligned) from fp32 parameters.
 * A derived cache: rebuilt after load_state_dict / optimizer steps, never saved. */
int pnr_mlp_pack(const pnr_mlp_params* p, void* packed, void* stream);

/* Projected variant of the blob (see PNR_SCENE_PROJECTED): lin_z stages are identity matrices over d_hidden channels. */
size_t pnr_mlp_pack_projected_bytes(const pnr_mlp_params* p);
int pnr_mlp_pack_projected(const pnr_mlp_params* p, void* packed, void* stream);
/* feat (n_pixels, d_latent) fp32 channels-last encoder output -> out (n_pixels, n_linz * d_hidden) bf16, slice b =
 * feat . lin_z[b].weight^T (no bias; fp32 arithmetic, one rounding).  workspace: n_pixels * d_hidden floats. */
int pnr_project_features(const pnr_mlp_params* p, const float* feat, long long n_pixels, void* out, void* workspace,
                         size_t workspace_bytes, void* stream);

/* ---- field function: PixelNeRFNet.forward (src/model/models.py:153-318) -------------------------- */
/* out (SB*P, 4) fp32 = [sigmoid(rgb), relu(sigma)].  precision PNR_PREC_FP32 uses `params` and a
 * caller workspace of pnr_field_workspace_bytes(); PNR_PREC_BF16 uses `packed` (from pnr_mlp_pack)
 * and a small caller workspace (pnr_field_workspace_bytes(): 256 KiB of view-mean scratch per SM pair,
 * 16-byte aligned; its contents need not survive the call but two concurrent calls need two workspaces). */
size_t pnr_field_workspace_bytes(const pnr_scene* scene, const pnr_points* pts, int precision);
int pnr_field_forward(const pnr_scene* scene, const pnr_points* pts, const pnr_mlp_params* params,
                      const void* packed, float* out, void* workspace, size_t workspace_bytes,
                      int precision, int num_freqs, float freq_factor, void* stream);

/* ---- training step (BASELINE config 3): what loss.backward() does for the reference ------------------ */
/* Gradient accumulators laid out like the pointer part of pnr_mlp_params: fp32 device buffers the backward pass ADDS into;
 * the caller zeroes them, like optimizer.zero_grad(). */
typedef struct pnr_mlp_grads {
  float* lin_in_w;  float* lin_in_b;
  float* lin_out_w; float* lin_out_b;
  float* fc0_w[8];  float* fc0_b[8];
  float* fc1_w[8];  float* fc1_b[8];
  float* linz_w[8]; float* linz_b[8];
} pnr_mlp_grads;

/* PixelNeRFNet.forward in training mode: fp32 arithmetic, fp32 channels-last feature maps (feat_fp32=1), every
 * activation the backward pass needs is kept on the caller-owned `tape` (pnr_field_tape_bytes()).  With PNR_COMBINE_MAX
 * the tape also holds the winning view of every (point, feature) (one byte each): the backward pass sends the pooled
 * gradient to the first maximal view, as torch.max(dim) does. */
size_t pnr_field_tape_bytes(const pnr_scene* scene, const pnr_points* pts, const pnr_mlp_params* params);
int pnr_field_forward_train(const pnr_scene* scene, const pnr_points* pts, const pnr_mlp_params* params, float* out,
                            void* tape, size_t tape_bytes, int num_freqs, float freq_factor, void* stream);
/* Backward of the call above.  out / d_out (SB*P, d_out): activated outputs and their gradient.  Adds the parameter
 * gradients into `grads`; optionally adds into d_feat (fp32 channels-last, shape of scene->feat: the gradient that
 * autograd sends into SpatialEncoder.latent through F.grid_sample, encoder.py:101-107) and into d_xyz (SB*P, 3;
 * point mode 0) or d_z (SB*B*K; point mode 1, x = o + z d), which the caller zeroes.  Any of the three may be NULL. */
size_t pnr_field_backward_workspace_bytes(const pnr_scene* scene, const pnr_points* pts, const pnr_mlp_params* params);
int pnr_field_backward(const pnr_scene* scene, const pnr_points* pts, const pnr_mlp_params* params, const void* tape,
                       const float* out, const float* d_out, const pnr_mlp_grads* grads, float* d_feat, float* d_xyz,
                       float* d_z, void* workspace, size_t workspace_bytes, int num_freqs, float freq_factor,
                       void* stream);
/* Camera gradients of the field function: what autograd sends, for the reference, into the camera inputs of
 * PixelNeRFNet.encode / forward and of the renderers.  Optional outputs that pnr_field_backward_cameras ADDS into (the caller
 * zeroes them); NULL = not wanted.
 *   d_poses  (SB*NS, 3, 4): with respect to the world->camera matrices of scene->poses (R | t);
 *   d_focal  (SB*NS, 2)   : with respect to scene->focal, the per-view values the kernels read (fy sign convention and YOLO
 *                           negation already applied: uv = -xy / z * focal + center);
 *   d_center (SB*NS, 2)   : with respect to scene->center;
 *   d_dirs   (SB, P, 3)   : point mode 0: with respect to pts->dirs (used only by z-feature layouts with view directions);
 *   d_rays   (SB*B, 8)    : point mode 1: columns 0-5, origin and direction of pts->rays (points o + z d, view direction d).
 *                           Near and far reach the depths only through the samplers: pnr_sample_bounds_backward.
 * image_shape and latent_scaling are constants (buffers in the reference). */
typedef struct pnr_camera_grads {
  float* d_poses;
  float* d_focal;
  float* d_center;
  float* d_dirs;
  float* d_rays;
} pnr_camera_grads;
/* pnr_field_backward plus the camera gradients of `cams` (NULL, or all of its pointers NULL: exactly pnr_field_backward).
 * The gradient of the projection x_cam = R x + t, uv = -x_cam.xy / x_cam.z * focal + center, of the bilinear tap position
 * (a row whose latent is zeroed -- YOLO z >= 0 -- or whose taps all fall outside the map has none) and of the z-feature
 * inputs (R x, R x + t, -z, R d, raw or encoded) of every (object, view, point) row, summed over rows per view and over
 * views per point or ray. */
int pnr_field_backward_cameras(const pnr_scene* scene, const pnr_points* pts, const pnr_mlp_params* params, const void* tape,
                               const float* out, const float* d_out, const pnr_mlp_grads* grads, float* d_feat, float* d_xyz,
                               float* d_z, const pnr_camera_grads* cams, void* workspace, size_t workspace_bytes, int num_freqs,
                               float freq_factor, void* stream);
/* Backward of pnr_composite (nerf.py:184-188, 229-255): d_rgb (B,3), d_depth (B, may be NULL), d_weights (B,K, may be
 * NULL) -> d_rgb_sigma (B,K,4) and, if non-NULL, d_z (B,K) (both overwritten). */
int pnr_composite_backward(const float* rgb_sigma, const float* z, const float* rays, const float* d_rgb,
                           const float* d_depth, const float* d_weights, float* d_rgb_sigma, float* d_z, int B, int K,
                           int white_bkgd, void* stream);
/* pnr_composite_backward that also adds d far (the last interval is far - z_K, nerf.py:187) into column 7 of d_rays (B, 8)
 * when d_rays is non-NULL. */
int pnr_composite_backward_rays(const float* rgb_sigma, const float* z, const float* rays, const float* d_rgb,
                                const float* d_depth, const float* d_weights, float* d_rgb_sigma, float* d_z, float* d_rays,
                                int B, int K, int white_bkgd, void* stream);
/* Near / far gradients of the sample depths (nerf.py:104-167, 300-301), added into columns 6 and 7 of d_rays (B, 8).
 *   z_sorted == NULL, the coarse samples: z = near (1 - s) + far s (lindisp: 1 / ((1 - s) / near + s / far)) with
 *     s = steps_k + noise_coarse / Kc (as pnr_sample_coarse), given their gradient d_z_coarse (B, Kc).
 *   z_sorted != NULL, the fine pass: the merged row z_sorted (B, Kc+Kf+Kfd) of pnr_sample_fine and its gradient d_z_sorted.
 *     Each sample is found at the position of its value (equal values in concatenation order).  Importance samples have
 *     s = (inds + jitter) / Kc (inds (B, Kf) int32 from pnr_sample_fine's inds_out); depth samples clamped at near or far
 *     send their gradient there; the coarse samples' share is written to d_z_coarse_out (B, Kc; may be NULL).  The
 *     unclamped depth samples' share is pnr_sample_fine_depth_backward's. */
int pnr_sample_bounds_backward(const float* rays, const float* steps, const float* noise_coarse, const float* d_z_coarse,
                               const float* z_coarse, const float* z_sorted, const float* d_z_sorted, const int32_t* inds,
                               const float* jitter, const float* depth, const float* gauss, float* d_rays, float* d_z_coarse_out,
                               int B, int Kc, int Kf, int Kfd, float depth_std, int lindisp, void* stream);
/* Backward of sample_fine_depth + cat + sort (nerf.py:156-167, 296-301) with respect to the coarse depth:
 * d_depth[b] = sum of d_z_sorted over the positions of the unclamped depth samples (overwritten). */
int pnr_sample_fine_depth_backward(const float* z_sorted, const float* d_z_sorted, const float* depth,
                                   const float* gauss, const float* rays, float* d_depth, int B, int K, int Kfd,
                                   float depth_std, void* stream);

/* ---- the whole render in one call: NeRFRenderer.forward (src/render/nerf.py:257-309) ----------------------------- */
/* sample_coarse -> field (coarse MLP) -> composite -> sample_fine + sample_fine_depth + sort -> field (fine MLP) ->
 * composite, enqueued back to back on `stream` (bf16 tensor-core path).  rays (SB*B, 8); noise as for the stage calls;
 * outputs rgb (SB*B,3), depth (SB*B), optional weights (SB*B,K); fine outputs unused when n_fine == 0; mlp_fine may be
 * NULL (the coarse network renders the fine pass, models.py:291).  workspace: pnr_render_workspace_bytes(), 256-byte
 * aligned (sample depths, field values, view-mean scratch). */
typedef struct pnr_render_args {
  const pnr_scene* scene;
  const float* rays; int32_t B;                    /* rays per object */
  int64_t total_rays;                              /* rows of `rays` / the noise / output buffers; must equal scene->SB * B */
  const pnr_scene* scene_fine;                     /* scene of the fine pass if it differs (lin_z pre-projections of the fine
                                                      network, PNR_SCENE_PROJECTED); NULL = `scene` */
  int32_t n_splits;                                /* 0 = automatic.  > 1: the ray batch is rendered as that many independent
                                                      slices on forked streams, so that the tail wave of one field launch
                                                      overlaps the head of the next (matters for small batches, e.g. one
                                                      2 048-ray shard of an image; results are bit-identical, rays are
                                                      independent).  Only for scene->SB == 1. */
  const float* steps;                              /* linspace(0, 1 - 1/Kc, Kc), see pnr_sample_coarse */
  const float* noise_coarse; const float* noise_u; const float* noise_jitter; const float* noise_gauss;
  const pnr_mlp_params* mlp_coarse; const void* packed_coarse;
  const pnr_mlp_params* mlp_fine;   const void* packed_fine;
  int32_t n_coarse, n_fine, n_fine_depth;
  float depth_std;
  int32_t white_bkgd, lindisp, precision, num_freqs;
  float freq_factor;
  float* rgb_coarse; float* depth_coarse; float* weights_coarse;
  float* rgb_fine;   float* depth_fine;   float* weights_fine;
  void* workspace; size_t workspace_bytes;
  void* field_events[4];                           /* optional cudaEvent_t: recorded before / after the coarse and the fine
                                                      field-kernel launch (measurement hook of bench.py); NULL = none */
} pnr_render_args;
size_t pnr_render_workspace_bytes(const pnr_render_args* args);
int pnr_render_forward(const pnr_render_args* args, void* stream);

/* ResnetFC.forward as a stand-alone operator (src/model/resnetfc.py:134-186), fp32 arithmetic.
 * zx (rows, d_latent + d_in) fp32, rows ordered (object, view, point) with NS views and P points per
 * object (combine_inner_dims = (NS, P)); out (rows / NS, d_out) raw lin_out values. */
size_t pnr_resnetfc_workspace_bytes(const pnr_mlp_params* p, long long rows);
int pnr_resnetfc_forward(const pnr_mlp_params* p, const float* zx, long long rows, int NS, int P,
                         float* out, void* workspace, size_t workspace_bytes, void* stream);

/* Number of kernels the last pnr_* call on this thread launched (for bench.py's gpu_launches). */
int pnr_last_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* PIXELNERF_B200_H */
