"""NeRFRenderer: drop-in for ``src/render/nerf.py`` on the sm_100a ray-tile kernels.

One ``forward`` = sample_coarse -> field (coarse MLP) -> composite -> sample_fine + sample_fine_depth +
sort -> field (fine MLP) -> composite, i.e. nerf.py:257-309, with every stage a CUDA kernel of the C-ABI
library and the sample positions never materialised (the field kernel computes o + z*d itself).
Random numbers are drawn with the same four torch calls, in the same order, as the reference
(nerf.py:117,141,147,164), so a run seeded like the reference consumes the generator identically;
``noise_override`` lets tests feed identical noise to the CPU oracle.
"""
import torch

from .. import _lib
from ..conf import DotMap


class _CoarseFn(torch.autograd.Function):
    """sample_coarse (nerf.py:104-124, yolo.py:15-27) with the gradient autograd derives for the reference's near and far
    (``pnr_sample_bounds_backward``).  Used when the rays require grad; otherwise the depths are drawn without a graph."""

    @staticmethod
    def forward(ctx, rays, noise, steps, lindisp):
        lib = _lib.load()
        B, Kc = noise.shape
        dev = rays.device
        noise = noise.contiguous()
        z = torch.empty(B, Kc, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            rc = lib.pnr_sample_coarse(rays.data_ptr(), steps.data_ptr(), noise.data_ptr(), z.data_ptr(), B, Kc, int(lindisp),
                                       _lib.stream_ptr(dev))
        _lib.check(rc, "pnr_sample_coarse")
        ctx.lindisp = int(lindisp)
        ctx.save_for_backward(rays, noise, steps)
        return z

    @staticmethod
    def backward(ctx, d_z):
        lib = _lib.load()
        rays, noise, steps = ctx.saved_tensors
        B, Kc = noise.shape
        dev = rays.device
        d_rays = torch.zeros_like(rays)
        d_z = d_z.contiguous().float()
        with torch.cuda.device(dev):
            rc = lib.pnr_sample_bounds_backward(rays.data_ptr(), steps.data_ptr(), noise.data_ptr(), d_z.data_ptr(), None, None,
                                                None, None, None, None, None, d_rays.data_ptr(), None, B, Kc, 0, 0, 0.0,
                                                ctx.lindisp, _lib.stream_ptr(dev))
        _lib.check(rc, "pnr_sample_bounds_backward")
        return d_rays, None, None, None


class _CompositeFn(torch.autograd.Function):
    """composite (nerf.py:184-188, 229-255) with the backward pass autograd derives for the reference."""

    @staticmethod
    def forward(ctx, out, z, rays, white_bkgd):
        lib = _lib.load()
        B, K = z.shape
        dev = z.device
        out, z = out.contiguous(), z.contiguous()
        w = torch.empty(B, K, device=dev, dtype=torch.float32)
        rgb = torch.empty(B, 3, device=dev, dtype=torch.float32)
        depth = torch.empty(B, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            rc = lib.pnr_composite(out.data_ptr(), z.data_ptr(), rays.data_ptr(), w.data_ptr(), rgb.data_ptr(),
                                   depth.data_ptr(), B, K, int(bool(white_bkgd)), _lib.stream_ptr(dev))
        _lib.check(rc, "pnr_composite")
        ctx.white = int(bool(white_bkgd))
        ctx.save_for_backward(out, z, rays)
        return w, rgb, depth

    @staticmethod
    def backward(ctx, d_w, d_rgb, d_depth):
        lib = _lib.load()
        out, z, rays = ctx.saved_tensors
        B, K = z.shape
        dev = z.device
        c = lambda t: None if t is None else t.contiguous().float()
        d_w, d_rgb, d_depth = c(d_w), c(d_rgb), c(d_depth)
        if d_rgb is None:
            d_rgb = torch.zeros(B, 3, device=dev)
        d_out = torch.empty_like(out)
        d_z = torch.empty_like(z) if ctx.needs_input_grad[1] else None
        d_rays = torch.zeros_like(rays) if ctx.needs_input_grad[2] else None      # far: the last interval is far - z_K
        with torch.cuda.device(dev):
            rc = lib.pnr_composite_backward_rays(out.data_ptr(), z.data_ptr(), rays.data_ptr(), d_rgb.data_ptr(),
                                                 _lib.ptr(d_depth), _lib.ptr(d_w), d_out.data_ptr(), _lib.ptr(d_z),
                                                 _lib.ptr(d_rays), B, K, ctx.white, _lib.stream_ptr(dev))
        _lib.check(rc, "pnr_composite_backward")
        return d_out, d_z, d_rays, None


class _ResampleFn(torch.autograd.Function):
    """sample_fine + sample_fine_depth + cat + sort (nerf.py:126-167, 290-301).  The coarse depth carries a gradient to the
    depth samples; when the rays require grad, the merged row also sends gradient to the coarse depths it contains and, from the
    importance samples and the clamped depth samples, to near / far (the importance sampler is fed detached weights,
    nerf.py:136, 293)."""

    @staticmethod
    def forward(ctx, depth, weights, rays, z_coarse, u, jitter, gauss, kf, kfd, depth_std, lindisp):
        lib = _lib.load()
        B, Kc = z_coarse.shape
        dev = rays.device
        z_out = torch.empty(B, Kc + kf + kfd, device=dev, dtype=torch.float32)
        c = lambda t: None if t is None else t.contiguous().data_ptr()
        depth = depth.contiguous()
        bounds = ctx.needs_input_grad[2] or ctx.needs_input_grad[3]
        inds = torch.empty(B, kf, device=dev, dtype=torch.int32) if bounds and kf > 0 else None
        with torch.cuda.device(dev):
            rc = lib.pnr_sample_fine(c(weights), depth.data_ptr(), rays.data_ptr(), z_coarse.data_ptr(), c(u), c(jitter),
                                     c(gauss), z_out.data_ptr(), _lib.ptr(inds), None, None, B, Kc, kf, kfd, float(depth_std),
                                     int(lindisp), _lib.stream_ptr(dev))
        _lib.check(rc, "pnr_sample_fine")
        ctx.kf, ctx.kfd, ctx.depth_std, ctx.lindisp = kf, kfd, float(depth_std), int(lindisp)
        cont = lambda t: None if t is None else t.contiguous()
        ctx.save_for_backward(z_out, depth, cont(gauss), rays, *((z_coarse, inds, cont(jitter)) if bounds else ()))
        return z_out

    @staticmethod
    def backward(ctx, d_z):
        lib = _lib.load()
        z_out, depth, gauss, rays, *bounds = ctx.saved_tensors
        B, K = z_out.shape
        dev = rays.device
        d_z = d_z.contiguous().float()
        d_depth = d_rays = d_zc = None
        with torch.cuda.device(dev):
            if ctx.kfd > 0 and ctx.needs_input_grad[0]:
                d_depth = torch.empty_like(depth)
                rc = lib.pnr_sample_fine_depth_backward(z_out.data_ptr(), d_z.data_ptr(), depth.data_ptr(), gauss.data_ptr(),
                                                        rays.data_ptr(), d_depth.data_ptr(), B, K, ctx.kfd, ctx.depth_std,
                                                        _lib.stream_ptr(dev))
                _lib.check(rc, "pnr_sample_fine_depth_backward")
            if bounds:
                z_coarse, inds, jitter = bounds
                Kc = z_coarse.shape[1]
                d_rays = torch.zeros_like(rays)
                d_zc = torch.empty_like(z_coarse)
                rc = lib.pnr_sample_bounds_backward(rays.data_ptr(), None, None, None, z_coarse.data_ptr(), z_out.data_ptr(),
                                                    d_z.data_ptr(), _lib.ptr(inds), _lib.ptr(jitter), depth.data_ptr(),
                                                    _lib.ptr(gauss), d_rays.data_ptr(), d_zc.data_ptr(), B, Kc, ctx.kf, ctx.kfd,
                                                    ctx.depth_std, ctx.lindisp, _lib.stream_ptr(dev))
                _lib.check(rc, "pnr_sample_bounds_backward")
        needs = ctx.needs_input_grad
        return (d_depth, None, d_rays if needs[2] else None, d_zc if needs[3] else None) + (None,) * 7


class _RenderWrapper(torch.nn.Module):
    """nerf.py:21-48: binds a network to a renderer; call signature ``(rays, want_weights=False)``."""

    def __init__(self, net, renderer, simple_output):
        super().__init__()
        self.net = net
        self.renderer = renderer
        self.simple_output = simple_output

    def forward(self, rays, want_weights=False):
        if rays.shape[0] == 0:
            return (torch.zeros(0, 3, device=rays.device), torch.zeros(0, device=rays.device))
        outputs = self.renderer(self.net, rays, want_weights=want_weights and not self.simple_output)
        if self.simple_output:
            lvl = outputs.fine if self.renderer.using_fine else outputs.coarse
            return lvl.rgb, lvl.depth
        return outputs.toDict()


class NeRFRenderer(torch.nn.Module):
    def __init__(self, n_coarse=128, n_fine=0, n_fine_depth=0, noise_std=0.0, depth_std=0.01,
                 eval_batch_size=100000, white_bkgd=False, lindisp=False, sched=None):
        super().__init__()
        self.n_coarse = n_coarse
        self.n_fine = n_fine
        self.n_fine_depth = n_fine_depth
        self.noise_std = noise_std
        self.depth_std = depth_std
        self.eval_batch_size = eval_batch_size     # kept for API compatibility; the fused path never chunks
        self.white_bkgd = white_bkgd
        self.lindisp = lindisp
        if lindisp:
            print("Using linear displacement rays")
        self.using_fine = n_fine > 0
        self.sched = sched
        if sched is not None and len(sched) == 0:
            self.sched = None
        self.register_buffer("iter_idx", torch.tensor(0, dtype=torch.long), persistent=True)
        self.register_buffer("last_sched", torch.tensor(0, dtype=torch.long), persistent=True)
        self.noise_override = None      # optional dict(coarse, fine_u, fine_jitter, depth) of device tensors
        self.n_splits = 0               # pnr_render_args.n_splits: 0 = automatic slicing of small batches over forked streams
        self._steps_cache = {}
        self._ws_cache = {}             # device -> persistent workspace of the single-call render
        self._plan = {}                 # device -> (key, pnr_render_args, keep-alives) of the last single-call render
        self.field_events = None        # optional 4 torch.cuda.Event (timing on): recorded around the two field-kernel launches
        self.last_launches = 0          # kernels launched by the last forward (bench.py's gpu_launches)

    # ---- stage wrappers (public so the parity tests can drive each reference method) -------------------
    def _steps(self, device):
        """linspace(0, 1 - 1/Kc, Kc) computed on the CPU (same bits as the oracle's) and kept on the device per (Kc, device)."""
        key = (self.n_coarse, str(device))
        t = self._steps_cache.get(key)
        if t is None:
            step = 1.0 / self.n_coarse
            t = torch.linspace(0, 1 - step, self.n_coarse).to(device)
            self._steps_cache[key] = t
        return t

    def sample_coarse(self, rays, noise=None):
        """nerf.py:104-124.  rays (B, 8) -> z (B, Kc)."""
        lib = _lib.load()
        B = rays.shape[0]
        dev = rays.device
        if noise is None:
            noise = torch.rand(B, self.n_coarse, device=dev, dtype=torch.float32)
        z = torch.empty(B, self.n_coarse, device=dev, dtype=torch.float32)
        steps = self._steps(dev)
        with torch.cuda.device(dev):
            rc = lib.pnr_sample_coarse(rays.data_ptr(), steps.data_ptr(), noise.contiguous().data_ptr(), z.data_ptr(),
                                       B, self.n_coarse, int(self.lindisp), _lib.stream_ptr(dev))
        _lib.check(rc, "pnr_sample_coarse")
        self.last_launches += lib.pnr_last_launch_count()
        return z

    def composite_values(self, out, z, rays, want_weights=True):
        """nerf.py:184-188,229-255 given the field values ``out`` (B, K, 4)."""
        lib = _lib.load()
        B, K = z.shape
        dev = z.device
        w = torch.empty(B, K, device=dev, dtype=torch.float32) if want_weights else None
        rgb = torch.empty(B, 3, device=dev, dtype=torch.float32)
        depth = torch.empty(B, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            rc = lib.pnr_composite(out.contiguous().data_ptr(), z.data_ptr(), rays.data_ptr(), _lib.ptr(w), rgb.data_ptr(),
                                   depth.data_ptr(), B, K, int(bool(self.white_bkgd)), _lib.stream_ptr(dev))
        _lib.check(rc, "pnr_composite")
        self.last_launches += lib.pnr_last_launch_count()
        return w, rgb, depth

    def resample(self, rays, z_coarse, weights, depth, u=None, jitter=None, gauss=None, debug=False):
        """sample_fine + sample_fine_depth + cat + sort (nerf.py:126-167, 290-301) -> z (B, Kc + n_fine)."""
        lib = _lib.load()
        B = rays.shape[0]
        dev = rays.device
        kf, kfd = self.n_fine - self.n_fine_depth, self.n_fine_depth
        if kf > 0:
            if u is None:
                u = torch.rand(B, kf, dtype=torch.float32, device=dev)
            if jitter is None:
                jitter = torch.rand_like(u)
        if kfd > 0 and gauss is None:
            gauss = torch.randn(B, kfd, dtype=torch.float32, device=dev)
        z_out = torch.empty(B, self.n_coarse + kf + kfd, device=dev, dtype=torch.float32)
        dbg = None
        if debug:
            dbg = (torch.empty(B, kf, device=dev, dtype=torch.int32), torch.empty(B, kf, device=dev),
                   torch.empty(B, kfd, device=dev))
        c = lambda t: None if t is None else t.contiguous().data_ptr()
        with torch.cuda.device(dev):
            rc = lib.pnr_sample_fine(c(weights), c(depth), rays.data_ptr(), z_coarse.data_ptr(), c(u), c(jitter), c(gauss),
                                     z_out.data_ptr(), c(dbg[0]) if dbg else None, c(dbg[1]) if dbg else None,
                                     c(dbg[2]) if dbg else None, B, self.n_coarse, kf, kfd, float(self.depth_std),
                                     int(self.lindisp), _lib.stream_ptr(dev))
        _lib.check(rc, "pnr_sample_fine")
        self.last_launches += lib.pnr_last_launch_count()
        return (z_out, dbg) if debug else z_out

    def _field(self, model, rays, z, coarse, sb):
        if not hasattr(model, "field_from_rays"):
            raise TypeError("NeRFRenderer (B200 path) renders pixel_nerf_yolo_b200.model.PixelNeRFNet instances "
                            "only: the per-point model call of the reference is fused into one kernel and there "
                            "is no generic-callable fallback")
        out = model.field_from_rays(rays, z, coarse=coarse, sb=sb)
        self.last_launches += getattr(model, "last_launches", 0)
        return out

    # ---- nerf.py:257-309 -----------------------------------------------------------------------------
    def forward(self, model, rays, want_weights=False):
        if self.sched is not None and self.last_sched.item() > 0:
            self.n_coarse = self.sched[1][self.last_sched.item() - 1]
            self.n_fine = self.sched[2][self.last_sched.item() - 1]
        assert len(rays.shape) == 3
        _lib.require_cuda(rays, "rays")
        _lib.require_device(rays.device)
        if self.training and self.noise_std > 0.0:
            raise NotImplementedError("NeRFRenderer (B200 path): noise_std > 0 is not built (no shipped conf uses it)")
        self.last_launches = 0
        sb = rays.shape[0]
        if hasattr(model, "num_views_per_obj") and hasattr(model, "poses") and rays.shape[1] > 0:
            # the kernels take the object count from the encoded scene: a ray batch for a different number of objects would run
            # past the ray / output buffers
            assert sb * model.num_views_per_obj == model.poses.shape[0], (
                f"rays hold {sb} object(s) but encode() saw {model.poses.shape[0] // max(model.num_views_per_obj, 1)}")
        rays = rays.reshape(-1, 8).contiguous().float()
        nz = self.noise_override or {}
        if torch.is_grad_enabled() and hasattr(model, "_wants_grad") and (
                model._wants_grad(True, rays) or (self.using_fine and model._wants_grad(False))):
            return self._forward_train(model, rays, sb, want_weights, nz)
        if getattr(model, "fused_render_ready", lambda: False)() and rays.shape[0] > 0:
            return self._forward_single_call(model, rays, sb, want_weights, nz)
        with torch.no_grad():
            z_coarse = self.sample_coarse(rays, nz.get("coarse"))
            out_c = self._field(model, rays, z_coarse, True, sb)
            need_w = want_weights or (self.using_fine and self.n_fine - self.n_fine_depth > 0)
            coarse = self.composite_values(out_c, z_coarse, rays, want_weights=need_w)
            outputs = DotMap(coarse=self._format_outputs(coarse, sb, want_weights))
            if self.using_fine:
                z_all = self.resample(rays, z_coarse, coarse[0], coarse[2], nz.get("fine_u"), nz.get("fine_jitter"),
                                      nz.get("depth"))
                out_f = self._field(model, rays, z_all, False, sb)
                fine = self.composite_values(out_f, z_all, rays, want_weights=want_weights)
                outputs.fine = self._format_outputs(fine, sb, want_weights)
        return outputs

    def _forward_single_call(self, model, rays, sb, want_weights, nz):
        """Inference: the whole of nerf.py:257-309 as ONE C-ABI call (``pnr_render_forward``).  Noise is drawn with the
        reference's four torch calls in the reference's order (nerf.py:117,141,147,164).  The argument block (scene, packed
        weights, sample counts, workspace) is prepared once per (model state, batch shape) and re-used: per call only the
        ray / noise / output pointers change."""
        import ctypes as C
        lib = _lib.load()
        dev = rays.device
        Bt = rays.shape[0]
        kc, kf, kfd = self.n_coarse, self.n_fine - self.n_fine_depth, self.n_fine_depth
        fine = self.using_fine and self.n_fine > 0
        with torch.no_grad():
            noise_c = nz.get("coarse")
            if noise_c is None:
                noise_c = torch.rand(Bt, kc, device=dev, dtype=torch.float32)
            u = jitter = gauss = None
            if fine:
                u, jitter, gauss = nz.get("fine_u"), nz.get("fine_jitter"), nz.get("depth")
                if kf > 0:
                    if u is None:
                        u = torch.rand(Bt, kf, dtype=torch.float32, device=dev)
                    if jitter is None:
                        jitter = torch.rand_like(u)
                if kfd > 0 and gauss is None:
                    gauss = torch.randn(Bt, kfd, dtype=torch.float32, device=dev)
            cont = lambda t: None if t is None else t.contiguous()
            noise_c, u, jitter, gauss = cont(noise_c), cont(u), cont(jitter), cont(gauss)
            key = (str(dev), Bt, sb, kc, self.n_fine if fine else 0, kfd if fine else 0, float(self.depth_std), bool(self.white_bkgd),
                   bool(self.lindisp), int(self.n_splits), self.field_events is not None, model.render_state_key())
            plan = self._plan.get(key[0])
            if plan is not None and plan[0] != key:
                plan = None
            if plan is None:
                a = _lib.RenderArgs()
                sc_c, sc_f, keep = model.render_scenes()
                a.scene = C.pointer(sc_c)
                if sc_f is not None:
                    a.scene_fine = C.pointer(sc_f)
                a.B, a.total_rays = Bt // sb, Bt
                steps = self._steps(dev)
                a.steps = steps.data_ptr()
                mc, mf = model.mlp_coarse, model.mlp_fine
                proj = model.projects_latent()
                cpc, pk_c = mc.c_params(), mc.packed(projected=proj)
                a.mlp_coarse, a.packed_coarse = C.pointer(cpc), pk_c.data_ptr()
                cpf = pk_f = None
                if mf is not None:
                    cpf, pk_f = mf.c_params(), mf.packed(projected=proj)
                    a.mlp_fine, a.packed_fine = C.pointer(cpf), pk_f.data_ptr()
                a.n_coarse, a.n_fine, a.n_fine_depth = kc, (self.n_fine if fine else 0), (kfd if fine else 0)
                a.depth_std, a.white_bkgd, a.lindisp = float(self.depth_std), int(bool(self.white_bkgd)), int(bool(self.lindisp))
                a.precision, (a.num_freqs, a.freq_factor) = _lib.PREC_BF16, model.code_args()
                a.n_splits = 1 if self.field_events is not None else int(self.n_splits)
                nbytes = lib.pnr_render_workspace_bytes(a)
                ws = self._ws_cache.get(key[0])                # one persistent workspace per (renderer, device)
                if ws is None or ws.numel() < nbytes:
                    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
                    self._ws_cache[key[0]] = ws
                a.workspace, a.workspace_bytes = ws.data_ptr(), nbytes
                plan = (key, a, (sc_c, sc_f, keep, steps, cpc, cpf, pk_c, pk_f, ws))
                self._plan[key[0]] = plan
            a = plan[1]
            a.rays, a.noise_coarse = rays.data_ptr(), noise_c.data_ptr()
            a.noise_u, a.noise_jitter, a.noise_gauss = _lib.ptr(u), _lib.ptr(jitter), _lib.ptr(gauss)
            f32 = dict(device=dev, dtype=torch.float32)
            rgb_c, depth_c = torch.empty(Bt, 3, **f32), torch.empty(Bt, **f32)
            w_c = torch.empty(Bt, kc, **f32) if want_weights else None
            a.rgb_coarse, a.depth_coarse, a.weights_coarse = rgb_c.data_ptr(), depth_c.data_ptr(), _lib.ptr(w_c)
            rgb_f = depth_f = w_f = None
            if fine:
                rgb_f, depth_f = torch.empty(Bt, 3, **f32), torch.empty(Bt, **f32)
                w_f = torch.empty(Bt, kc + self.n_fine, **f32) if want_weights else None
                a.rgb_fine, a.depth_fine, a.weights_fine = rgb_f.data_ptr(), depth_f.data_ptr(), _lib.ptr(w_f)
            for i in range(4):
                a.field_events[i] = None
            if self.field_events is not None:            # measurement hook (bench.py): events must exist before C records them
                for i, ev in enumerate(self.field_events[:4 if fine else 2]):
                    ev.record()
                    a.field_events[i] = ev.cuda_event
            with torch.cuda.device(dev):
                rc = lib.pnr_render_forward(a, _lib.stream_ptr(dev))
            _lib.check(rc, "pnr_render_forward")
            self.last_launches = lib.pnr_last_launch_count()
            outputs = DotMap(coarse=self._format_outputs((w_c, rgb_c, depth_c), sb, want_weights))
            if fine:
                outputs.fine = self._format_outputs((w_f, rgb_f, depth_f), sb, want_weights)
        return outputs

    def _forward_train(self, model, rays, sb, want_weights, nz):
        """The same sequence recorded for backward (PixelNerfTrainer.calc_losses -> loss.backward(), config 3):
        every stage is an autograd.Function over the C-ABI forward/backward kernels.  Rays that require grad get what autograd
        gives the reference's: origin and direction from the field, near and far from the samplers and the last interval."""
        dev = rays.device
        B = rays.shape[0]
        if rays.requires_grad:
            noise = nz.get("coarse")
            if noise is None:
                noise = torch.rand(B, self.n_coarse, device=dev, dtype=torch.float32)
            z_coarse = _CoarseFn.apply(rays, noise, self._steps(dev), self.lindisp)
            self.last_launches += _lib.last_launch_count()
        else:
            with torch.no_grad():
                z_coarse = self.sample_coarse(rays, nz.get("coarse"))
        out_c = self._field(model, rays, z_coarse, True, sb)
        w_c, rgb_c, depth_c = _CompositeFn.apply(out_c, z_coarse, rays, self.white_bkgd)
        outputs = DotMap(coarse=self._format_outputs((w_c, rgb_c, depth_c), sb, want_weights))
        if self.using_fine:
            kf, kfd = self.n_fine - self.n_fine_depth, self.n_fine_depth
            u, jitter, gauss = nz.get("fine_u"), nz.get("fine_jitter"), nz.get("depth")
            if kf > 0:
                if u is None:
                    u = torch.rand(B, kf, dtype=torch.float32, device=dev)
                if jitter is None:
                    jitter = torch.rand_like(u)
            if kfd > 0 and gauss is None:
                gauss = torch.randn(B, kfd, dtype=torch.float32, device=dev)
            z_all = _ResampleFn.apply(depth_c, w_c.detach(), rays, z_coarse, u, jitter, gauss, kf, kfd, self.depth_std,
                                      self.lindisp)
            out_f = self._field(model, rays, z_all, False, sb)
            w_f, rgb_f, depth_f = _CompositeFn.apply(out_f, z_all, rays, self.white_bkgd)
            outputs.fine = self._format_outputs((w_f, rgb_f, depth_f), sb, want_weights)
        return outputs

    def _format_outputs(self, rendered, sb, want_weights=False):
        weights, rgb, depth = rendered
        if sb > 0:
            rgb = rgb.reshape(sb, -1, 3)
            depth = depth.reshape(sb, -1)
            if weights is not None:
                weights = weights.reshape(sb, -1, weights.shape[-1])
        ret = DotMap(rgb=rgb, depth=depth)
        if want_weights:
            ret.weights = weights
        return ret

    def sched_step(self, steps=1):
        """nerf.py:324-344."""
        if self.sched is None:
            return
        self.iter_idx += steps
        while self.last_sched.item() < len(self.sched[0]) and self.iter_idx.item() >= self.sched[0][self.last_sched.item()]:
            self.n_coarse = self.sched[1][self.last_sched.item()]
            self.n_fine = self.sched[2][self.last_sched.item()]
            print("INFO: NeRF sampling resolution changed on schedule ==> c", self.n_coarse, "f", self.n_fine)
            self.last_sched += 1

    @classmethod
    def from_conf(cls, conf, white_bkgd=False, lindisp=False, eval_batch_size=100000):
        return cls(conf.get_int("n_coarse", 128), conf.get_int("n_fine", 0), n_fine_depth=conf.get_int("n_fine_depth", 0),
                   noise_std=conf.get_float("noise_std", 0.0), depth_std=conf.get_float("depth_std", 0.01),
                   white_bkgd=conf.get_float("white_bkgd", white_bkgd), lindisp=lindisp,
                   eval_batch_size=conf.get_int("eval_batch_size", eval_batch_size), sched=conf.get_list("sched", None))

    def bind_parallel(self, net, gpus=None, simple_output=False):
        """nerf.py:360-377.  With several GPUs the rays are sharded across devices with the weights and the
        encoded scene replicated once (not per call, as DataParallel does); see ``dist.ShardedRenderer``."""
        wrapped = _RenderWrapper(net, self, simple_output=simple_output)
        if gpus is not None and len(gpus) > 1:
            from ..dist import MultiDeviceRenderer
            print("Using multi-GPU", gpus)
            wrapped = MultiDeviceRenderer(wrapped, gpus)
        return wrapped
