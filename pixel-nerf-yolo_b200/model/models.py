"""PixelNeRFNet: drop-in for ``src/model/models.py`` whose ``forward`` is one fused sm_100a kernel.

``encode`` keeps the reference's bookkeeping (world->camera poses, focal sign flip, principal point,
``image_shape``; models.py:92-151) and runs the encoder trunk in PyTorch; ``forward`` hands
(points, view directions, scene) to ``pnr_field_forward`` which does projection, the 4-tap gather,
positional encoding, the ResnetFC with the view mean and the output activations (models.py:153-318).
"""
import os
import os.path as osp
import warnings

import torch

from .. import _lib
from .code import PositionalEncoding
from .model_util import make_encoder, make_mlp


class _FieldTrainFn(torch.autograd.Function):
    """PixelNeRFNet.forward with a backward pass (BASELINE config 3): ``pnr_field_forward_train`` keeps the
    activations on a tape, ``pnr_field_backward`` produces what autograd produces for the reference --
    gradients of the ResnetFC parameters, of the feature maps and of the sample depths / query points.  When a camera input
    requires grad (the per-view poses / focal / center tensors of ``_camera_tensors``, the view directions in point mode, the
    rays in ray mode), ``pnr_field_backward_cameras`` adds those gradients in the same pass."""

    @staticmethod
    def forward(ctx, net, mlp, mode, sb, feat, a, b, cam_poses, cam_focal, cam_center, *params):
        lib = _lib.load()
        dev = feat.device
        sc, keep = net._scene_for(feat, fp32_maps=True, cams=(cam_poses, cam_focal, cam_center) + net._camera_tensors()[3:])
        # mode "rays": a = rays (SB*B, 8), b = z (SB*B, K); mode "xyz": a = xyz (SB, P, 3), b = viewdirs (SB, P, 3)
        pts = _lib.points_rays(a, b, sb) if mode == "rays" else _lib.points_xyz(a, b)
        P = pts.P
        cp = mlp.c_params()
        out = torch.empty(sb, P, net.d_out, device=dev, dtype=torch.float32)
        tape = torch.empty(lib.pnr_field_tape_bytes(sc, pts, cp), dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            rc = lib.pnr_field_forward_train(sc, pts, cp, out.data_ptr(), tape.data_ptr(), tape.numel(),
                                             *net.code_args(), _lib.stream_ptr(dev))
        _lib.check(rc, "pnr_field_forward_train")
        net.last_launches = lib.pnr_last_launch_count()
        ctx.net, ctx.mlp, ctx.mode, ctx.sb, ctx.P = net, mlp, mode, sb, P
        ctx.keep = keep
        ctx.save_for_backward(feat, a, b, out, tape, *params)
        return out

    @staticmethod
    def backward(ctx, d_out):
        lib = _lib.load()
        feat, a, b, out, tape, *params = ctx.saved_tensors
        net, mlp, mode, sb, P = ctx.net, ctx.mlp, ctx.mode, ctx.sb, ctx.P
        dev = feat.device
        sc, _keep = net._scene_for(feat, fp32_maps=True, cams=ctx.keep)
        pts = _lib.points_rays(a, b, sb) if mode == "rays" else _lib.points_xyz(a, b)
        cp = mlp.c_params()
        flat = torch.zeros(sum(p.numel() for p in params), device=dev, dtype=torch.float32)      # one fill for all accumulators
        grads, off = [], 0
        for p in params:
            grads.append(flat[off:off + p.numel()].view_as(p))
            off += p.numel()
        need_feat, need_a, need_b = ctx.needs_input_grad[4], ctx.needs_input_grad[5], ctx.needs_input_grad[6]
        d_feat = torch.zeros_like(feat) if need_feat else None
        d_xyz = torch.zeros_like(a) if (mode == "xyz" and need_a) else None
        d_z = torch.zeros_like(b) if (mode == "rays" and need_b) else None
        # camera inputs: per-view poses / focal / center, view directions (point mode), rays (ray mode)
        zeros_if = lambda need, t: torch.zeros(t.shape, device=dev, dtype=torch.float32) if need else None
        d_poses, d_focal, d_center = (zeros_if(ctx.needs_input_grad[7 + i], t) for i, t in enumerate(ctx.keep[:3]))
        d_dirs = zeros_if(mode == "xyz" and need_b, b)
        d_rays = zeros_if(mode == "rays" and need_a, a)
        ws = torch.empty(lib.pnr_field_backward_workspace_bytes(sc, pts, cp), dtype=torch.uint8, device=dev)
        d_out = d_out.contiguous().float()
        args = (sc, pts, cp, tape.data_ptr(), out.data_ptr(), d_out.data_ptr(), mlp.c_grads(grads), _lib.ptr(d_feat),
                _lib.ptr(d_xyz), _lib.ptr(d_z))
        tail = (ws.data_ptr(), ws.numel(), *net.code_args(), _lib.stream_ptr(dev))
        cam_grads = (d_poses, d_focal, d_center, d_dirs, d_rays)
        with torch.cuda.device(dev):
            if any(t is not None for t in cam_grads):
                cg = _lib.CameraGrads(*(_lib.ptr(t) for t in cam_grads))
                rc = lib.pnr_field_backward_cameras(*args, cg, *tail)
            else:
                rc = lib.pnr_field_backward(*args, *tail)
        _lib.check(rc, "pnr_field_backward")
        net.last_bwd_launches = getattr(net, "last_bwd_launches", 0) + lib.pnr_last_launch_count()
        d_a = d_xyz if mode == "xyz" else d_rays
        d_b = d_dirs if mode == "xyz" else d_z
        return (None, None, None, None, d_feat, d_a, d_b, d_poses, d_focal, d_center, *grads)


class PixelNeRFNet(torch.nn.Module):
    TRAIN_PRECISIONS = ("fp32", "tf32", "bf16")

    def __init__(self, conf, stop_encoder_grad=False):
        super().__init__()
        self.encoder = make_encoder(conf["encoder"])
        self.use_encoder = conf.get_bool("use_encoder", True)
        self.use_xyz = conf.get_bool("use_xyz", False)
        assert self.use_encoder or self.use_xyz
        self.normalize_z = conf.get_bool("normalize_z", True)
        self.stop_encoder_grad = stop_encoder_grad
        self.use_code = conf.get_bool("use_code", False)
        self.use_code_viewdirs = conf.get_bool("use_code_viewdirs", True)
        self.use_viewdirs = conf.get_bool("use_viewdirs", False)
        self.use_global_encoder = conf.get_bool("use_global_encoder", False)
        # The fused kernels implement every switch that shapes the z-feature (the non-latent part of each MLP input row:
        # use_xyz, normalize_z, use_code, code.include_input, use_viewdirs, use_code_viewdirs; PNR_SCENE_ZF_* bits) and both
        # view-pooling modes of ResnetFC: combine_type average / max before block combine_layer, or no pooling at all
        # (combine_layer >= n_blocks, the single-view conf/default.conf network; one source view only).  Not built: the
        # network without pixel-aligned features (use_encoder = False), the global encoder, and z-features wider than the
        # one K = 64 slab of lin_in.
        unsupported = []
        if not self.use_encoder: unsupported.append("use_encoder=False")
        if self.use_global_encoder: unsupported.append("use_global_encoder=True")
        if unsupported:
            raise NotImplementedError("PixelNeRFNet (B200 path) does not build: " + ", ".join(unsupported))

        d_latent = self.encoder.latent_size
        # z-feature width and encoder exactly as models.py:16-90 (no `code` module, and no code.* state, without use_code)
        d_in = 3 if self.use_xyz else 1
        if self.use_viewdirs and self.use_code_viewdirs:
            d_in += 3
        if self.use_code and d_in > 0:
            self.code = PositionalEncoding.from_conf(conf["code"], d_in=d_in)
            d_in = self.code.d_out
        if self.use_viewdirs and not self.use_code_viewdirs:
            d_in += 3
        if d_in > 64:
            raise NotImplementedError(
                f"PixelNeRFNet (B200 path): these switches give a z-feature of d_in={d_in} values; the fused kernels take at "
                f"most 64 (one K = 64 slab of lin_in)")
        self.zf_flags = ((0 if self.use_viewdirs else _lib.SCENE_ZF_NO_VIEWDIRS)
                         | (_lib.SCENE_ZF_CODE_VIEWDIRS if self.use_viewdirs and self.use_code_viewdirs else 0)
                         | (0 if self.normalize_z else _lib.SCENE_ZF_CAM_COORDS)
                         | (0 if self.use_xyz else _lib.SCENE_ZF_Z_ONLY)
                         | (0 if self.use_code else _lib.SCENE_ZF_NO_CODE)
                         | (_lib.SCENE_ZF_NO_CODE_INPUT if self.use_code and not self.code.include_input else 0))
        self.latent_size = self.encoder.latent_size
        self.mlp_coarse = make_mlp(conf["mlp_coarse"], d_in, d_latent)
        self.mlp_fine = make_mlp(conf["mlp_fine"], d_in, d_latent, allow_empty=True)
        self.register_buffer("poses", torch.empty(1, 3, 4), persistent=False)
        self.register_buffer("image_shape", torch.empty(2), persistent=False)
        # YOLO head (models.py:75-81): raw per-anchor values, poses/focal used as given, latent masked where z >= 0
        self.yolo = conf.get_bool("mlp_coarse.yolo", False)
        self.d_in = d_in
        if not self.yolo:
            self.d_out = conf.get_int("mlp_coarse.d_out", 4)
            if self.d_out != 4:
                raise NotImplementedError("PixelNeRFNet (B200 path): d_out must be 4 (rgb + sigma) outside YOLO mode")
        else:
            self.d_out = conf.get_int("mlp_coarse.d_out", 7) * conf.get_int("mlp_coarse.num_anchors_per_scale", 3)
            if self.d_out > 32:
                raise NotImplementedError("PixelNeRFNet (B200 path): YOLO head wider than 32 outputs is not built")
        self.d_latent = d_latent
        self.register_buffer("focal", torch.empty(1, 2), persistent=False)
        self.register_buffer("c", torch.empty(1, 2), persistent=False)
        self.num_objs = 0
        self.num_views_per_obj = 1
        # "bf16": tcgen05 tensor-core path (production).  "fp32": SIMT fp32 check path.
        self.precision = "bf16"
        # Latents wider than the hidden width (1 792-channel YOLO maps): gather lin_z PRE-PROJECTIONS of the maps instead of
        # streaming the wide lin_z through the kernel (PNR_SCENE_PROJECTED).  None = automatic (d_latent > 512).
        self.project_wide_latent = None
        # arithmetic of the training path's GEMMs: "fp32" (SIMT, gradients equal autograd up to summation order), "tf32"
        # (mma.sync tensor cores, fp32 accumulate) or "bf16" (tcgen05 cta_group::2 GEMMs over a bf16 tape, fp32 accumulate in
        # TMEM: the fast path, gradients within ~2e-2 of autograd)
        self.train_precision = "fp32"
        self.fp32_chunk_points = 50000
        self._cam_cache = None
        self._cam_gen = 0            # bumped by set_cameras (encode): part of render_state_key()
        self._field_ws = None        # persistent view-mean scratch of the tcgen05 field kernel

    # ------------------------------------------------------------------------------------------------
    def encode(self, images, poses, focal, z_bounds=None, c=None):
        """images (SB, NS, 3, H, W) or (NS, 3, H, W); poses camera-to-world (.., 4, 4); focal / c in any of
        the reference's formats (models.py:92-151)."""
        self.num_objs = images.size(0)
        if len(images.shape) == 5:
            assert len(poses.shape) == 4
            assert poses.size(1) == images.size(1)
            self.num_views_per_obj = images.size(1)
            images = images.reshape(-1, *images.shape[2:])
            poses = poses.reshape(-1, 4, 4)
        else:
            self.num_views_per_obj = 1
        self._check_views()
        self.encoder(images, return_latent=False)
        self.set_cameras(poses, focal, (images.shape[-1], images.shape[-2]), c)

    def _check_views(self):
        for mlp in (self.mlp_coarse, self.mlp_fine):
            if mlp is not None:
                mlp.check_views(self.num_views_per_obj)

    def set_cameras(self, poses, focal, image_wh, c=None):
        """The camera half of ``encode`` (models.py:116-148) without running the encoder trunk."""
        if not self.yolo:
            rot = poses[:, :3, :3].transpose(1, 2)
            trans = -torch.bmm(rot, poses[:, :3, 3:])
            self.poses = torch.cat((rot, trans), dim=-1).float()
        else:
            self.poses = poses[:, :3, :4].float()            # models.py:119-120: already world -> camera
        self.image_shape[0] = image_wh[0]
        self.image_shape[1] = image_wh[1]
        if len(focal.shape) == 0:
            focal = focal[None, None].repeat((1, 2))
        elif len(focal.shape) == 1:
            focal = focal.unsqueeze(-1).repeat((1, 2))
        else:
            focal = focal.clone()
        self.focal = focal.float().to(self.poses.device)
        if not self.yolo:
            self.focal[..., 1] *= -1.0                       # models.py:136-137
        if c is None:
            c = (self.image_shape * 0.5).unsqueeze(0)
        elif len(c.shape) == 0:
            c = c[None, None].repeat((1, 2))
        elif len(c.shape) == 1:
            c = c.unsqueeze(-1).repeat((1, 2))
        self.c = c.float().to(self.poses.device)
        self._cam_cache = None
        self._cam_gen += 1

    # ------------------------------------------------------------------------------------------------
    def _scene(self, fp32_maps: bool):
        """pnr_scene view of the encoded state (+ the tensors that must stay alive during the call)."""
        return self._scene_for(self.encoder.packed_latent(fp32=fp32_maps), fp32_maps)

    def _camera_tensors(self):
        """(poses (SB*NS, 3, 4), focal (SB*NS, 2), center (SB*NS, 2), image w, image h, latent scaling x, y): the per-view
        camera values the kernels read, computed from ``set_cameras``'s state once per encode.  They stay in torch's graph, so
        gradients of the per-view tensors reach the caller's camera-to-world poses and intrinsics as in the reference; a cache
        built without that graph (under no_grad) is rebuilt when a camera input requires grad."""
        cache = self._cam_cache
        stale = cache is not None and torch.is_grad_enabled() and any(
            src.requires_grad and not t.requires_grad for src, t in zip((self.poses, self.focal, self.c), cache[:3]))
        if cache is None or stale:
            n_views = self.poses.shape[0]
            NS = self.num_views_per_obj
            SB = n_views // NS
            dev = self.poses.device

            def per_view(t):     # (1|SB, 2) -> (SB*NS, 2): repeat_interleave over views (models.py:225-230)
                t = t.to(dev).float()
                if t.shape[0] == 1:
                    return t.expand(n_views, 2).contiguous()
                if t.shape[0] == SB:
                    return t.unsqueeze(1).expand(SB, NS, 2).reshape(n_views, 2).contiguous()
                if t.shape[0] == n_views:
                    return t.contiguous()
                raise AssertionError(f"focal/c has {t.shape[0]} rows for {SB} objects x {NS} views")
            # the kernels compute uv = -xy / z * focal + c (models.py:220); YOLO mode is uv = +xy / z * focal + c (:222)
            focal_k = -self.focal if self.yolo else self.focal
            self._cam_cache = (self.poses.contiguous(), per_view(focal_k), per_view(self.c),
                               float(self.image_shape[0]), float(self.image_shape[1]),
                               float(self.encoder.latent_scaling[0]), float(self.encoder.latent_scaling[1]))
        return self._cam_cache

    def _scene_for(self, feat, fp32_maps: bool, cams=None):
        """pnr_scene over an explicit channels-last feature tensor (the training path passes the autograd-tracked
        fp32 copy); ``cams`` re-uses the camera tensors captured at forward time."""
        n_views = self.poses.shape[0]
        NS = self.num_views_per_obj
        self._check_views()
        SB = n_views // NS
        poses, focal, center, iw, ih, lsx, lsy = cams if cams is not None else self._camera_tensors()
        assert feat.shape[0] == n_views, "encoder.latent and poses disagree on the number of views"
        sc = _lib.Scene()
        sc.feat, sc.poses, sc.focal, sc.center = feat.data_ptr(), poses.data_ptr(), focal.data_ptr(), center.data_ptr()
        sc.SB, sc.NS, sc.C, sc.Hl, sc.Wl = SB, NS, feat.shape[3], feat.shape[1], feat.shape[2]
        sc.feat_fp32 = int(fp32_maps)
        sc.flags = ((_lib.SCENE_MASK_NONNEG_Z | _lib.SCENE_RAW_OUTPUT) if self.yolo else 0) | self.zf_flags
        if fp32_maps and self.train_precision == "tf32":
            sc.flags |= _lib.SCENE_TRAIN_TF32            # read by the training entry points only
        elif fp32_maps and self.train_precision == "bf16":
            sc.flags |= _lib.SCENE_TRAIN_BF16
        sc.image_w, sc.image_h, sc.lat_scale_x, sc.lat_scale_y = iw, ih, lsx, lsy
        return sc, (poses, focal, center, iw, ih, lsx, lsy)

    def code_args(self):
        """(num_freqs, freq_factor) of the z-feature's positional encoding for the C entry points; (0, 0.0) without one."""
        if not self.use_code:
            return 0, 0.0
        return self.code.num_freqs, float(self.code.freq_factor)

    def projects_latent(self) -> bool:
        """True when the tcgen05 path gathers lin_z PRE-PROJECTIONS of the maps (PNR_SCENE_PROJECTED): automatic for latents
        wider than the hidden width (1 792-channel YOLO maps), or forced with ``project_wide_latent``."""
        proj = self.project_wide_latent
        if proj is None:
            proj = self.mlp_coarse.d_latent > self.mlp_coarse.d_hidden
        return bool(proj)

    def _scene_bf16(self, mlp, proj: bool):
        """pnr_scene of the tcgen05 path for one network: plain bf16 maps, or that network's lin_z pre-projections."""
        if proj:
            feat = mlp.project_features(self.encoder.packed_latent(fp32=True), self.encoder.generation)
            sc, keep = self._scene_for(feat, fp32_maps=False)
            sc.flags |= _lib.SCENE_PROJECTED
            return sc, (keep, feat)
        return self._scene(fp32_maps=False)

    def render_scenes(self):
        """(coarse scene, fine scene or None, keep-alives) for ``pnr_render_forward``: the two passes only differ when the
        maps are pre-projected through each network's own lin_z."""
        proj = self.projects_latent()
        sc_c, keep_c = self._scene_bf16(self.mlp_coarse, proj)
        if proj and self.mlp_fine is not None:
            sc_f, keep_f = self._scene_bf16(self.mlp_fine, proj)
            return sc_c, sc_f, (keep_c, keep_f)
        return sc_c, None, (keep_c,)

    def render_state_key(self):
        """Everything a prepared ``pnr_render_args`` depends on: encoded maps, cameras, weights, precision switches.  Explicit
        generation counters (not pointer identity, which the caching allocator re-issues)."""
        mf = self.mlp_fine
        return (self.encoder.generation, self._cam_gen, self.num_views_per_obj, self.projects_latent(), self.precision,
                self.mlp_coarse._param_key(), None if mf is None else mf._param_key())

    def _mlp(self, coarse):
        return self.mlp_coarse if (coarse or self.mlp_fine is None) else self.mlp_fine

    def _run_field(self, pts: "_lib.Points", SB: int, P: int, coarse: bool, keep) -> torch.Tensor:
        dev = self.poses.device
        _lib.require_device(dev)
        lib = _lib.load()
        mlp = self._mlp(coarse)
        out = torch.empty(SB, P, self.d_out, device=dev, dtype=torch.float32)
        if P == 0:
            return out
        launches = 0
        with torch.cuda.device(dev):
            if self.precision == "bf16":
                proj = self.projects_latent()
                sc, keep2 = self._scene_bf16(mlp, proj)
                ws_bytes = lib.pnr_field_workspace_bytes(sc, pts, _lib.PREC_BF16)
                ws = self._field_ws
                if ws is None or ws.numel() < max(ws_bytes, 16) or ws.device != dev:
                    ws = self._field_ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=dev)
                rc = lib.pnr_field_forward(sc, pts, mlp.c_params(), mlp.packed(projected=proj).data_ptr(), out.data_ptr(),
                                           ws.data_ptr(), ws_bytes, _lib.PREC_BF16, *self.code_args(),
                                           _lib.stream_ptr(dev))
                _lib.check(rc, "pnr_field_forward(bf16)")
                launches = lib.pnr_last_launch_count()
            elif self.precision == "fp32":
                sc, keep2 = self._scene(fp32_maps=True)
                cp = mlp.c_params()
                ws_bytes = lib.pnr_field_workspace_bytes(sc, pts, _lib.PREC_FP32)
                ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
                rc = lib.pnr_field_forward(sc, pts, cp, None, out.data_ptr(), ws.data_ptr(), ws_bytes,
                                           _lib.PREC_FP32, *self.code_args(),
                                           _lib.stream_ptr(dev))
                _lib.check(rc, "pnr_field_forward(fp32)")
                launches = lib.pnr_last_launch_count()
            else:
                raise ValueError(f"precision must be 'bf16' or 'fp32', got {self.precision!r}")
        self.last_launches = launches
        return out

    def forward(self, xyz, coarse=True, viewdirs=None, far=False):
        """(r, g, b, sigma) at world points xyz (SB, B, 3) given view directions (SB, B, 3) -> (SB, B, 4).  viewdirs may be
        None when the network does not use them (use_viewdirs = False)."""
        SB, B, _ = xyz.shape
        if self.use_viewdirs:
            assert viewdirs is not None
        _lib.require_cuda(xyz, "xyz")
        if viewdirs is not None:
            viewdirs = viewdirs.reshape(SB, B, 3).contiguous().float()
        if self._wants_grad(coarse, xyz, viewdirs):
            assert SB * self.num_views_per_obj == self.poses.shape[0], "call encode() first"
            mlp = self._mlp(coarse)
            return _FieldTrainFn.apply(self, mlp, "xyz", SB, self._train_feat(), xyz.contiguous().float(), viewdirs,
                                       *self._camera_tensors()[:3], *mlp.ordered_params())
        xyz = xyz.detach().contiguous().float()
        viewdirs = None if viewdirs is None else viewdirs.detach()
        assert SB * self.num_views_per_obj == self.poses.shape[0], "call encode() first"
        outs = []
        step = B if self.precision == "bf16" else max(1, self.fp32_chunk_points // max(SB * self.num_views_per_obj, 1))
        for b0 in range(0, max(B, 1), max(step, 1)):
            xs = xyz[:, b0:b0 + step].contiguous()
            ds = None if viewdirs is None else viewdirs[:, b0:b0 + step].contiguous()
            pts = _lib.points_xyz(xs, ds)
            outs.append(self._run_field(pts, SB, xs.shape[1], coarse, (xs, ds)))
        return outs[0] if len(outs) == 1 else torch.cat(outs, dim=1)

    def _wants_grad(self, coarse, *tensors):
        """True when this call must record a backward pass.  The reference simply runs under autograd, whatever the module's
        train/eval mode: so does this -- gradient mode on and anything on the path requiring grad (query points / depths,
        the network's parameters, the encoder's maps unless ``stop_encoder_grad``, the cameras of ``encode``: poses, focal, c;
        the caller passes its own camera inputs, view directions or rays).  Inference callers wrap the call in
        ``torch.no_grad()`` as the reference's eval scripts do (eval/eval.py:262, trainer.py vis/eval steps)."""
        if not torch.is_grad_enabled():
            return False
        want = any(t is not None and t.requires_grad for t in tensors + (self.poses, self.focal, self.c))
        want = want or any(p.requires_grad for p in self._mlp(coarse).parameters())
        if not want and not self.stop_encoder_grad:
            lat = self.encoder._latent
            want = lat is not None and lat.requires_grad
        return want

    def _train_feat(self):
        """fp32 channels-last view of encoder.latent that autograd can differentiate through (a permute + copy in
        torch: plumbing; models.py:242-243 detaches it when stop_encoder_grad is set)."""
        lat = self.encoder.latent
        if self.stop_encoder_grad:
            lat = lat.detach()
        return lat.float().permute(0, 2, 3, 1).contiguous()

    def fused_render_ready(self) -> bool:
        """True when NeRFRenderer can hand the whole forward to ``pnr_render_forward`` (one C call): bf16 tensor-core path,
        NeRF head."""
        return self.precision == "bf16" and not self.yolo

    def field_from_rays(self, rays, z, coarse=True, sb=1):
        """Renderer fast path: evaluate the field at o + z*d for rays (SB*B, 8), z (SB*B, K) without ever
        materialising the points (nerf.py:191-222 folded into the kernel's point fetch).  -> (SB*B, K, 4)."""
        Bt, K = z.shape
        assert Bt % sb == 0
        Bp = Bt // sb
        rays = rays.contiguous().float()
        z = z.contiguous().float()
        if self._wants_grad(coarse, z, rays):
            mlp = self._mlp(coarse)
            return _FieldTrainFn.apply(self, mlp, "rays", sb, self._train_feat(), rays, z, *self._camera_tensors()[:3],
                                       *mlp.ordered_params()).reshape(Bt, K, self.d_out)
        if self.precision == "bf16":
            pts = _lib.points_rays(rays, z, sb)
            return self._run_field(pts, sb, Bp * K, coarse, (rays, z)).reshape(Bt, K, self.d_out)
        # fp32 check path: bound the workspace by chunking rays (results do not depend on the chunking)
        step = max(1, self.fp32_chunk_points // max(K * self.num_views_per_obj * sb, 1))
        outs = []
        r3, z3 = rays.reshape(sb, Bp, 8), z.reshape(sb, Bp, K)
        for b0 in range(0, Bp, step):
            rc, zc = r3[:, b0:b0 + step].contiguous(), z3[:, b0:b0 + step].contiguous()
            n = rc.shape[1]
            pts = _lib.points_rays(rc.reshape(-1, 8), zc.reshape(-1, K), sb)
            outs.append(self._run_field(pts, sb, n * K, coarse, (rc, zc)).reshape(sb, n, K, self.d_out))
        return torch.cat(outs, dim=1).reshape(Bt, K, self.d_out)

    # ------------------------------------------------------------------------------------------------
    def load_weights(self, args, opt_init=False, strict=True, device=None):
        """checkpoints/<name>/pixel_nerf_{init,latest} (models.py:320-349)."""
        if opt_init and not args.resume:
            return
        ckpt_name = "pixel_nerf_init" if opt_init or not args.resume else "pixel_nerf_latest"
        model_path = "%s/%s/%s" % (args.checkpoints_path, args.name, ckpt_name)
        if device is None:
            device = self.poses.device
        if os.path.exists(model_path):
            print("Load", model_path)
            self.load_state_dict(torch.load(model_path, map_location=device), strict=strict)
        elif not opt_init:
            warnings.warn(("WARNING: {} does not exist, not loaded!! Model will be re-initialized.\n"
                           "If you are trying to load a pretrained model, STOP since it's not in the right place. "
                           "If training, unless you are startin a new experiment, please remember to pass --resume."
                           ).format(model_path))
        return self

    def save_weights(self, args, opt_init=False, epochNum=""):
        """models.py:351-370."""
        from shutil import copyfile
        ckpt_name = "pixel_nerf_init" if opt_init else "pixel_nerf_latest"
        backup_name = "pixel_nerf_init_backup" if opt_init else "pixel_nerf_backup" + epochNum
        ckpt_path = osp.join(args.checkpoints_path, args.name, ckpt_name)
        ckpt_backup_path = osp.join(args.checkpoints_path, args.name, backup_name)
        if osp.exists(ckpt_path):
            copyfile(ckpt_path, ckpt_backup_path)
        if epochNum == "":
            torch.save(self.state_dict(), ckpt_path)
        return self
