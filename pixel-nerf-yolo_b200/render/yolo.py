"""YoloRenderer: drop-in for ``src/render/yolo.py`` -- the fork's multi-view detection head (SURVEY.md section 8f row 3).

One ``forward`` = sample_coarse (yolo.py:15-27) -> field in YOLO mode (raw per-anchor values, models.py:119-120,
220-224, 254-264, 309-310: the same fused sm_100a kernel as the NeRF path with d_out = anchors x 7, the z >= 0 latent
mask and no output activation) -> per-ray reduction (yolo.py:96-114, ``pnr_yolo_reduce``).  With gradients enabled and a
network that requires them the same sequence records its backward pass (the reference's YoloTrainer back-propagates the
detection loss through it, train/trainlib/YoloTrainer.py:140-190).
"""
import torch

from .. import _lib


class _YoloReduceFn(torch.autograd.Function):
    """The per-ray reduction (yolo.py:96-114) with the backward pass autograd derives for the reference
    (``pnr_yolo_reduce`` / ``pnr_yolo_reduce_backward``)."""

    @staticmethod
    def forward(ctx, out, B, K, A):
        lib = _lib.load()
        dev = out.device
        out = out.contiguous()
        res = torch.empty(B, A, 7, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            rc = lib.pnr_yolo_reduce(out.data_ptr(), res.data_ptr(), B, K, A, _lib.stream_ptr(dev))
        _lib.check(rc, "pnr_yolo_reduce")
        ctx.dims = (B, K, A)
        ctx.save_for_backward(out)
        return res

    @staticmethod
    def backward(ctx, d_res):
        lib = _lib.load()
        (out,) = ctx.saved_tensors
        B, K, A = ctx.dims
        d_out = torch.empty_like(out)
        d_res = d_res.contiguous().float()
        with torch.cuda.device(out.device):
            rc = lib.pnr_yolo_reduce_backward(out.data_ptr(), d_res.data_ptr(), d_out.data_ptr(), B, K, A, _lib.stream_ptr(out.device))
        _lib.check(rc, "pnr_yolo_reduce_backward")
        return d_out, None, None, None


class YoloRenderer(torch.nn.Module):
    def __init__(self, n_coarse, eval_batch_size, num_scales, num_anchors_per_scale):
        super().__init__()
        self.net = None
        self.n_coarse = n_coarse
        self.eval_batch_size = eval_batch_size        # kept for API compatibility; the fused path never chunks
        self.num_scales = num_scales
        self.num_anchors_per_scale = num_anchors_per_scale
        self.noise_override = None                    # optional (B, n_coarse) U[0,1) tensor (parity tests)
        self.last_launches = 0

    def bind_net(self, net):
        self.net = net

    def sample_coarse(self, ray_batch, noise=None):
        """yolo.py:15-27 (identical to NeRFRenderer.sample_coarse without lindisp)."""
        lib = _lib.load()
        B = ray_batch.shape[0]
        dev = ray_batch.device
        if noise is None:
            noise = torch.rand(B, self.n_coarse, device=dev, dtype=torch.float32)
        z = torch.empty(B, self.n_coarse, device=dev, dtype=torch.float32)
        step = 1.0 / self.n_coarse
        steps = torch.linspace(0, 1 - step, self.n_coarse).to(dev)
        with torch.cuda.device(dev):
            rc = lib.pnr_sample_coarse(ray_batch.data_ptr(), steps.data_ptr(), noise.contiguous().data_ptr(), z.data_ptr(), B,
                                       self.n_coarse, 0, _lib.stream_ptr(dev))
        _lib.check(rc, "pnr_sample_coarse")
        self.last_launches += lib.pnr_last_launch_count()
        return z

    @classmethod
    def from_conf(cls, conf):
        return cls(conf.get_int("renderer.n_coarse", 128), conf.get_int("renderer.eval_batch_size", 1024),
                   conf.get_int("model.mlp_coarse.num_scales", 1), conf.get_int("model.mlp_coarse.num_anchors_per_scale", 3))

    def forward(self, rays):
        """rays (..., 8) -> (B, num_anchors_per_scale, 7) = [max probability, probability-weighted box values]."""
        if self.net is None:
            raise RuntimeError("YoloRenderer: call bind_net()/bind_parallel() first")
        if not getattr(self.net, "yolo", False) or not hasattr(self.net, "field_from_rays"):
            raise TypeError("YoloRenderer (B200 path) renders pixel_nerf_yolo_b200 PixelNeRFNet instances in YOLO mode only")
        _lib.require_cuda(rays, "rays")
        _lib.require_device(rays.device)
        self.last_launches = 0
        rays = rays.reshape(-1, 8).contiguous().float()
        B, A = rays.shape[0], self.num_anchors_per_scale
        dev = rays.device
        res = torch.empty(B, A, 7, device=dev, dtype=torch.float32)
        if B == 0:
            return res
        if torch.is_grad_enabled() and self.net._wants_grad(True, rays):
            # training (YoloTrainer.calc_losses -> loss.backward(), train/trainlib/YoloTrainer.py:140-190): the field records its
            # backward pass (pnr_field_forward_train / pnr_field_backward), the reduction has its own; rays that require grad
            # also get their near / far gradient through the coarse sampler
            if rays.requires_grad:
                from .nerf import _CoarseFn
                noise = self.noise_override
                if noise is None:
                    noise = torch.rand(B, self.n_coarse, device=dev, dtype=torch.float32)
                steps = torch.linspace(0, 1 - 1.0 / self.n_coarse, self.n_coarse).to(dev)
                z = _CoarseFn.apply(rays, noise, steps, False)
            else:
                with torch.no_grad():
                    z = self.sample_coarse(rays, self.noise_override)
            out = self.net.field_from_rays(rays, z, coarse=True, sb=1)              # (B, K, A*7) raw, autograd-tracked
            assert out.shape[-1] == A * 7, f"model d_out {out.shape[-1]} != {A} anchors x 7"
            return _YoloReduceFn.apply(out, B, self.n_coarse, A)
        with torch.no_grad():
            z = self.sample_coarse(rays, self.noise_override)
            out = self.net.field_from_rays(rays, z, coarse=True, sb=1)              # (B, K, A*7) raw
            self.last_launches += getattr(self.net, "last_launches", 0)
            assert out.shape[-1] == A * 7, f"model d_out {out.shape[-1]} != {A} anchors x 7"
            lib = _lib.load()
            with torch.cuda.device(dev):
                rc = lib.pnr_yolo_reduce(out.contiguous().data_ptr(), res.data_ptr(), B, self.n_coarse, A, _lib.stream_ptr(dev))
            _lib.check(rc, "pnr_yolo_reduce")
            self.last_launches += lib.pnr_last_launch_count()
        return res

    def bind_parallel(self, net, gpus=None):
        self.net = net
        if gpus is not None and len(gpus) > 1:
            raise NotImplementedError("YoloRenderer (B200 path): shard rays with dist.ShardedRenderer-style slicing; "
                                      "DataParallel is not used")
        return self
