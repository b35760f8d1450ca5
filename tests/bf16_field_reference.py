"""The arithmetic of the tcgen05 inference kernel (``pair::field_pair_kernel``, csrc/mlp_umma_pair.cu), restated on the CPU.

The golden-pinned oracle (oracle/pixelnerf_oracle.py) is the reference BEHAVIOUR: fp32 everywhere.  The fused kernel is
defined to round some operands to bf16, and that rounding moves its output by up to ~1e-2 from the oracle.  A bound that
loose cannot see a kernel that skips one MMA or reads one bias slot wrong (DESIGN.md section 2).  This module restates
what the kernel computes, so that the kernel can be held to a bound set by fp32 summation order alone (``TIGHT``).

* the feature maps are read as bf16 (``pnr_pack_features``), blended in fp32 and the blended latent is rounded to bf16 once;
* every trunk Linear (lin_in, lin_z, fc_0, fc_1) multiplies bf16 operands with bf16 weights and accumulates in fp32, and the
  residual stream stays fp32 (``O.field_forward(..., emulate_bf16=True)``);
* lin_out multiplies bf16 relu(x) with bf16 weights (the emulation keeps its weights fp32);
* view pooling is the mean or the elementwise max (tests/pooling_oracle.py);
* with pre-projected wide latents (``PNR_SCENE_PROJECTED``) the maps go through lin_z[b] in fp32 (``pnr_project_features``),
  are rounded to bf16, blended, rounded again, and added to x with an identity weight, which is exact; the lin_z bias is
  part of the kernel's cumulative bias table and is added in fp32.

``rounding=False`` switches every rounding off: the result is then the oracle's (bit for bit for streamed latents).

The bound is on the root mean square of the error over the points, not on the worst element.  The kernel accumulates in a
different order than the CPU, so the fp32 value before a bf16 rounding differs in its last bits, and one activation in a
few ten thousand rounds to the other bf16 neighbour.  A point has 512 features x NS views x ~12 layers of them, so such
flips are not rare: each moves some points by up to ~1e-3 (measured on a B200: worst element 1.5e-3 with average pooling,
5.6e-3 with max pooling; nudging every weight by one fp32 ulp on the CPU gives the same), while the mean square stays near
1e-4.  A structural fault (one skipped MMA, a wrong bias slot) moves every point, so it moves the mean square.
"""
import contextlib
import functools
from typing import Dict, Optional

import torch

import pooling_oracle as PO
from oracle import pixelnerf_oracle as O

# Bound on the RMS over points of kernel - field_forward_bf16: rgb absolute, sigma relative to 1 + |sigma|
# (tests/test_gpu_field_coverage.py, whose docstring has the measured numbers).  Max pooling passes the rounding flips of the
# one winning view through where the mean averages NS of them: its bound is MAX_POOL_FACTOR x TIGHT.
TIGHT = 6e-4
MAX_POOL_FACTOR = 2.0


def tight_bound(combine_type: str) -> float:
    return TIGHT * (MAX_POOL_FACTOR if combine_type == "max" else 1.0)


def bf16(t: torch.Tensor) -> torch.Tensor:
    """Round to the nearest bf16 (ties to even), kept in fp32."""
    return t.bfloat16().float()


def errors(out: torch.Tensor, ref: torch.Tensor):
    """(max |rgb error|, max |sigma error| / (1 + |sigma|)) of two (..., 4) field outputs."""
    out, ref = out.detach().cpu().float(), ref.detach().cpu().float()
    e_rgb = (out[..., :3] - ref[..., :3]).abs().max().item()
    e_sig = ((out[..., 3] - ref[..., 3]).abs() / (1 + ref[..., 3].abs())).max().item()
    return e_rgb, e_sig


def rms_errors(out: torch.Tensor, ref: torch.Tensor):
    """(RMS rgb error, RMS sigma error relative to 1 + |sigma|) over all points of two (..., 4) field outputs."""
    out, ref = out.detach().cpu().double(), ref.detach().cpu().double()
    e_rgb = (out[..., :3] - ref[..., :3]).pow(2).mean().sqrt().item()
    e_sig = ((out[..., 3] - ref[..., 3]) / (1 + ref[..., 3].abs())).pow(2).mean().sqrt().item()
    return e_rgb, e_sig


def project_maps(latent: torch.Tensor, mlp: Dict[str, torch.Tensor], n_linz: int, rounding: bool = True) -> torch.Tensor:
    """(V, C, Hl, Wl) fp32 maps -> (V, n_linz * 512, Hl, Wl): slice b is the map pushed through lin_z[b] (no bias) in fp32,
    rounded to bf16 (the maps ``ResnetFC.project_features`` gives the kernel)."""
    V, C, Hl, Wl = latent.shape
    rows = latent.permute(0, 2, 3, 1).reshape(-1, C)
    slices = [rows @ mlp[f"lin_z.{b}.weight"].t() for b in range(n_linz)]
    out = torch.cat(slices, dim=-1)
    if rounding:
        out = bf16(out)
    return out.reshape(V, Hl, Wl, -1).permute(0, 3, 1, 2).contiguous()


def _resnetfc_projected(p: Dict[str, torch.Tensor], zx: torch.Tensor, d_latent: int, n_blocks: int, combine_layer: int,
                        inner_dims, emulate_bf16: bool = False, *, combine_type: str) -> torch.Tensor:
    """pooling_oracle.resnetfc_forward with lin_z[b](z) replaced by an identity-weight Linear over the gathered pre-projection
    slice b (+ lin_z[b]'s bias): ``zx`` carries n_linz x 512 blended projected channels in place of the latent.  The identity
    product of the bf16-rounded slice is exact, as the kernel's is."""
    hidden = p["lin_in.weight"].shape[0]
    q = {k: v for k, v in p.items() if not k.endswith(".weight") or not k.startswith("lin_z.")}
    for b in range(min(combine_layer, n_blocks)):
        q[f"lin_z.{b}.weight"] = torch.eye(hidden, d_latent).roll(b * hidden, dims=1)
    return PO.resnetfc_forward(q, zx, d_latent, n_blocks, combine_layer, inner_dims, emulate_bf16=emulate_bf16,
                               combine_type=combine_type)


@contextlib.contextmanager
def _resnetfc(fn):
    saved = O.resnetfc_forward
    O.resnetfc_forward = fn
    try:
        yield
    finally:
        O.resnetfc_forward = saved


def field_forward_bf16(scene: O.Scene, mlp: Dict[str, torch.Tensor], xyz: torch.Tensor, dirs: torch.Tensor, *,
                       n_blocks: int = 5, combine_layer: int = 3, combine_type: str = "average", yolo: bool = False,
                       projected: Optional[bool] = None, rounding: bool = True) -> torch.Tensor:
    """What the tcgen05 field kernel computes for ``O.field_forward(scene, mlp, xyz, dirs, ...)``.

    ``projected``: the maps are gathered as lin_z pre-projections (None: as ``PixelNeRFNet.projects_latent`` decides, i.e.
    for latents wider than the hidden width).  ``combine_layer`` may exceed ``n_blocks`` (a network that never pools)."""
    C = scene.latent.shape[1]
    hidden = mlp["lin_in.weight"].shape[0]
    if projected is None:
        projected = C > hidden
    p = dict(mlp)
    if rounding:
        p["lin_out.weight"] = bf16(p["lin_out.weight"])
    kw = dict(n_blocks=n_blocks, combine_layer=combine_layer, yolo=yolo, emulate_bf16=rounding)
    if projected:
        n_linz = min(combine_layer, n_blocks)
        sc = O.Scene(**{**scene.__dict__, "latent": project_maps(scene.latent, mlp, n_linz, rounding)})
        with _resnetfc(functools.partial(_resnetfc_projected, combine_type=combine_type)):
            return O.field_forward(sc, p, xyz, dirs, **kw)
    sc = O.Scene(**{**scene.__dict__, "latent": bf16(scene.latent) if rounding else scene.latent})
    # the blended latent is rounded to bf16 once: emulate_bf16 rounds every Linear's input, and lin_z[b] all read the same z
    with PO.combine_type(combine_type):
        return O.field_forward(sc, p, xyz, dirs, **kw)
