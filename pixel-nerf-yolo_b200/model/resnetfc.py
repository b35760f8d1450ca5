"""ResnetFC / ResnetBlockFC parameter containers with the reference's names, shapes and initialisers
(``src/model/resnetfc.py``).  The modules hold the fp32 master weights (what checkpoints store); the
arithmetic runs in the CUDA library: fused with the feature gather inside ``PixelNeRFNet.forward``
(tcgen05 bf16 or SIMT fp32), or stand-alone through ``ResnetFC.forward`` (SIMT fp32)."""
import torch
from torch import nn

from .. import _lib


class ResnetBlockFC(nn.Module):
    def __init__(self, size_in, size_out=None, size_h=None, beta=0.0):
        super().__init__()
        size_out = size_in if size_out is None else size_out
        size_h = min(size_in, size_out) if size_h is None else size_h
        if size_in != size_out or size_h != size_in:
            raise NotImplementedError("ResnetBlockFC: only square blocks (size_in == size_h == size_out) are built")
        if beta > 0:
            raise NotImplementedError("ResnetBlockFC: softplus activation (beta > 0) is not built; ReLU only")
        self.size_in, self.size_h, self.size_out = size_in, size_h, size_out
        self.fc_0 = nn.Linear(size_in, size_h)
        self.fc_1 = nn.Linear(size_h, size_out)
        nn.init.constant_(self.fc_0.bias, 0.0)
        nn.init.kaiming_normal_(self.fc_0.weight, a=0, mode="fan_in")
        nn.init.constant_(self.fc_1.bias, 0.0)
        nn.init.zeros_(self.fc_1.weight)
        self.shortcut = None

    def forward(self, x):
        raise NotImplementedError("ResnetBlockFC is evaluated inside the fused ResnetFC kernels; call ResnetFC")


class ResnetFC(nn.Module):
    def __init__(self, d_in, d_out, n_blocks=5, d_latent=0, d_hidden=128, beta=0.0, combine_layer=1000,
                 combine_type="average", use_spade=False):
        super().__init__()
        if combine_type not in _lib.COMBINE_TYPES:
            raise NotImplementedError(f"ResnetFC: combine_type={combine_type!r} is not built (average or max)")
        if combine_type != "average" and combine_layer >= n_blocks:
            # a network that never pools its views has no pooling step for the mode to select; only the reference's default
            # ("average") is accepted there, so that a conf naming a mode it cannot apply is not silently ignored
            raise NotImplementedError(f"ResnetFC: combine_type={combine_type!r} needs combine_layer < n_blocks "
                                      f"(combine_layer={combine_layer}, n_blocks={n_blocks}: the views are never pooled)")
        if use_spade:
            raise NotImplementedError("ResnetFC: use_spade is not built")
        if beta > 0:
            raise NotImplementedError("ResnetFC: softplus activation (beta > 0) is not built; ReLU only")
        if d_in <= 0 or d_latent <= 0:
            raise NotImplementedError("ResnetFC: needs d_in > 0 and d_latent > 0 (pixel-aligned features)")
        self.lin_in = nn.Linear(d_in, d_hidden)
        nn.init.constant_(self.lin_in.bias, 0.0)
        nn.init.kaiming_normal_(self.lin_in.weight, a=0, mode="fan_in")
        self.lin_out = nn.Linear(d_hidden, d_out)
        nn.init.constant_(self.lin_out.bias, 0.0)
        nn.init.kaiming_normal_(self.lin_out.weight, a=0, mode="fan_in")
        self.n_blocks, self.d_latent, self.d_in, self.d_out, self.d_hidden = n_blocks, d_latent, d_in, d_out, d_hidden
        self.combine_layer, self.combine_type, self.use_spade = combine_layer, combine_type, use_spade
        self.blocks = nn.ModuleList([ResnetBlockFC(d_hidden, beta=beta) for _ in range(n_blocks)])
        n_lin_z = min(combine_layer, n_blocks)
        self.lin_z = nn.ModuleList([nn.Linear(d_latent, d_hidden) for _ in range(n_lin_z)])
        for lz in self.lin_z:
            nn.init.constant_(lz.bias, 0.0)
            nn.init.kaiming_normal_(lz.weight, a=0, mode="fan_in")
        self.activation = nn.ReLU()
        self._packed = None
        self._packed_key = None
        self._generation = 0

    # ---- C-ABI views of the parameters --------------------------------------------------------------
    def c_params(self) -> "_lib.MlpParams":
        p = _lib.MlpParams()
        f = lambda t: t.detach().contiguous().data_ptr()
        p.lin_in_w, p.lin_in_b = f(self.lin_in.weight), f(self.lin_in.bias)
        p.lin_out_w, p.lin_out_b = f(self.lin_out.weight), f(self.lin_out.bias)
        for i, blk in enumerate(self.blocks):
            p.fc0_w[i], p.fc0_b[i] = f(blk.fc_0.weight), f(blk.fc_0.bias)
            p.fc1_w[i], p.fc1_b[i] = f(blk.fc_1.weight), f(blk.fc_1.bias)
        for i, lz in enumerate(self.lin_z):
            p.linz_w[i], p.linz_b[i] = f(lz.weight), f(lz.bias)
        p.d_in, p.d_latent, p.d_hidden, p.d_out = self.d_in, self.d_latent, self.d_hidden, self.d_out
        p.n_blocks, p.combine_layer = self.n_blocks, min(self.combine_layer, self.n_blocks)
        p.combine_type = _lib.COMBINE_TYPES[self.combine_type]
        return p

    def pools_views(self) -> bool:
        """False for a network whose combine_layer is at or past its last block (conf/default.conf): it never pools the source
        views, so it is only defined for one view per object."""
        return self.combine_layer < self.n_blocks

    def check_views(self, num_views: int) -> None:
        if num_views > 1 and not self.pools_views():
            raise NotImplementedError(f"ResnetFC: combine_layer={self.combine_layer} >= n_blocks={self.n_blocks} never pools the "
                                      f"source views; it is only defined for one view per object (got {num_views})")

    def ordered_params(self):
        """Parameters in the fixed order the training-path autograd function passes them (and returns grads)."""
        ps = [self.lin_in.weight, self.lin_in.bias, self.lin_out.weight, self.lin_out.bias]
        for blk in self.blocks:
            ps += [blk.fc_0.weight, blk.fc_0.bias, blk.fc_1.weight, blk.fc_1.bias]
        for lz in self.lin_z:
            ps += [lz.weight, lz.bias]
        return ps

    def c_grads(self, grads):
        """pnr_mlp_grads over a list of fp32 accumulators in ``ordered_params`` order."""
        g = _lib.MlpGrads()
        it = iter(t.data_ptr() for t in grads)
        g.lin_in_w, g.lin_in_b, g.lin_out_w, g.lin_out_b = next(it), next(it), next(it), next(it)
        for i in range(len(self.blocks)):
            g.fc0_w[i], g.fc0_b[i], g.fc1_w[i], g.fc1_b[i] = next(it), next(it), next(it), next(it)
        for i in range(len(self.lin_z)):
            g.linz_w[i], g.linz_b[i] = next(it), next(it)
        return g

    def _param_key(self):
        """Identity of the current weights: every derived cache (packed bf16 stream, lin_z pre-projections, render plans) is
        keyed on it.  In-place updates through ``p.data`` do not bump ``p._version``: call ``invalidate()`` after those."""
        return (self._generation,) + tuple((q.data_ptr(), q._version) for q in self.parameters())

    def invalidate(self):
        """Drop every cache derived from the parameters (call after editing weights behind autograd's back, e.g. ``p.data``)."""
        self._generation += 1
        self._packed = None
        self._packed_proj = None
        self._projected = None

    def _load_from_state_dict(self, *args, **kwargs):
        super()._load_from_state_dict(*args, **kwargs)
        self._generation += 1

    def packed(self, projected: bool = False) -> torch.Tensor:
        """bf16 tcgen05 weight stream + bias tables: a derived cache, rebuilt whenever a parameter changed
        (optimizer step, load_state_dict, .to()); never part of the state_dict.  ``projected``: the variant for
        pre-projected feature maps (identity lin_z stages, ``PNR_SCENE_PROJECTED``)."""
        if projected:
            return self._packed_projected()
        key = self._param_key()
        if self._packed is None or self._packed_key != key:
            dev = self.lin_in.weight.device
            _lib.require_cuda(self.lin_in.weight, "ResnetFC parameters")
            _lib.require_device(dev)
            lib = _lib.load()
            cp = self.c_params()
            nbytes = lib.pnr_mlp_pack_bytes(cp)
            if nbytes == 0:
                _lib.check(-3, "pnr_mlp_pack_bytes")
            buf = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
            off = (-buf.data_ptr()) % 1024
            blob = buf[off:off + nbytes]
            with torch.cuda.device(dev):
                _lib.check(lib.pnr_mlp_pack(cp, blob.data_ptr(), _lib.stream_ptr(dev)), "pnr_mlp_pack")
            self._packed, self._packed_key = blob, key
        return self._packed

    def _packed_projected(self) -> torch.Tensor:
        key = self._param_key()
        hit = getattr(self, "_packed_proj", None)
        if hit is None or hit[0] != key:
            dev = self.lin_in.weight.device
            _lib.require_cuda(self.lin_in.weight, "ResnetFC parameters")
            _lib.require_device(dev)
            lib = _lib.load()
            cp = self.c_params()
            nbytes = lib.pnr_mlp_pack_projected_bytes(cp)
            if nbytes == 0:
                _lib.check(-3, "pnr_mlp_pack_projected_bytes")
            buf = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
            off = (-buf.data_ptr()) % 1024
            blob = buf[off:off + nbytes]
            with torch.cuda.device(dev):
                _lib.check(lib.pnr_mlp_pack_projected(cp, blob.data_ptr(), _lib.stream_ptr(dev)), "pnr_mlp_pack_projected")
            self._packed_proj = (key, blob)
        return self._packed_proj[1]

    def project_features(self, feat_fp32_nhwc: torch.Tensor, feat_gen: int = 0) -> torch.Tensor:
        """(N, Hl, Wl, d_latent) fp32 channels-last encoder output -> (N, Hl, Wl, n_lin_z * d_hidden) bf16: slice b is the map
        pushed through ``lin_z[b]`` (no bias).  Cached per (parameters, map): recomputed after an optimizer step or encode."""
        key = (self._param_key(), feat_fp32_nhwc.data_ptr(), feat_fp32_nhwc._version, tuple(feat_fp32_nhwc.shape), feat_gen)
        hit = getattr(self, "_projected", None)
        if hit is None or hit[0] != key:
            lib = _lib.load()
            dev = feat_fp32_nhwc.device
            n, h, w, c = feat_fp32_nhwc.shape
            assert c == self.d_latent
            out = torch.empty(n, h, w, len(self.lin_z) * self.d_hidden, device=dev, dtype=torch.bfloat16)
            ws = torch.empty(n * h * w * self.d_hidden * 4, dtype=torch.uint8, device=dev)
            with torch.cuda.device(dev):
                rc = lib.pnr_project_features(self.c_params(), feat_fp32_nhwc.data_ptr(), n * h * w, out.data_ptr(), ws.data_ptr(),
                                              ws.numel(), _lib.stream_ptr(dev))
            _lib.check(rc, "pnr_project_features")
            self._projected = (key, out)
        return self._projected[1]

    def forward(self, zx, combine_inner_dims=(1,), combine_index=None, dim_size=None):
        """Stand-alone operator, fp32 SIMT kernels: zx (..., d_latent + d_in) rows ordered
        (object, view, point) -> raw lin_out values (rows / NS, d_out)."""
        assert zx.size(-1) == self.d_latent + self.d_in
        if combine_index is not None:
            raise NotImplementedError("ResnetFC: combine_index (frustum culling) is not built")
        rows = zx.numel() // zx.size(-1)
        if len(combine_inner_dims) == 1:
            ns, pts = 1, max(rows, 1)
        else:
            ns, pts = int(combine_inner_dims[0]), int(combine_inner_dims[1])
        self.check_views(ns)
        _lib.require_cuda(zx, "ResnetFC input")
        _lib.require_device(zx.device)
        zx2 = zx.reshape(-1, zx.size(-1)).contiguous().float()
        lib = _lib.load()
        cp = self.c_params()
        out = torch.empty(rows // ns, self.d_out, device=zx.device, dtype=torch.float32)
        ws = torch.empty(lib.pnr_resnetfc_workspace_bytes(cp, rows), dtype=torch.uint8, device=zx.device)
        with torch.cuda.device(zx.device):
            rc = lib.pnr_resnetfc_forward(cp, zx2.data_ptr(), rows, ns, pts, out.data_ptr(), ws.data_ptr(),
                                          ws.numel(), _lib.stream_ptr(zx.device))
        _lib.check(rc, "pnr_resnetfc_forward")
        return out

    @classmethod
    def from_conf(cls, conf, d_in, **kwargs):
        if not conf.get_bool("yolo", False):
            d_out = conf.get_int("d_out", 4)
        else:
            d_out = conf.get_int("d_out", 7) * conf.get_int("num_anchors_per_scale", 3)
        return cls(d_in, d_out=d_out, n_blocks=conf.get_int("n_blocks", 5), d_hidden=conf.get_int("d_hidden", 128),
                   beta=conf.get_float("beta", 0.0), combine_layer=conf.get_int("combine_layer", 1000),
                   combine_type=conf.get_string("combine_type", "average"), use_spade=conf.get_bool("use_spade", False),
                   **kwargs)
