"""PixelNeRFNet.forward with the six z-feature switches, on the CPU, for the z-feature tests.

``oracle.pixelnerf_oracle.field_forward`` is pinned to the golden vectors of the shipped confs and builds the default z-feature
only.  ``field_forward`` here is the same computation with the z-feature of any switch combination (models.py:183-209):

    zf = x_rot if normalize_z else x_cam                       (rows, 3)   x_rot = R x, x_cam = R x + t
    zf = zf if use_xyz else -zf[..., 2:3]                      (rows, 1)
    if use_code and not use_code_viewdirs: zf = PE(zf)
    if use_viewdirs:                       zf = cat(zf, R d)
    if use_code and use_code_viewdirs:     zf = PE(zf)

with PE the oracle's ``positional_encoding`` (``include_input`` = code.include_input).  Everything else is the oracle's own
code: projection, ``bilinear_index``, ``resnetfc_forward`` (looked up at call time, so ``pooling_oracle.combine_type`` and
``bf16_field_reference`` still substitute theirs), the output activations.  With the default switches the result equals
``O.field_forward`` bit for bit (tests/test_oracle_zfeature.py).

``switched(...)`` makes ``O.field_forward`` this function for the duration of a ``with`` block, so that the oracle's callers
(``O.render``, ``bf16_field_reference.field_forward_bf16``) run the switched network.
"""
import contextlib
import functools
from typing import Dict, Optional

import torch

from oracle import pixelnerf_oracle as O

DEFAULT = dict(use_viewdirs=True, use_code_viewdirs=False, normalize_z=True, use_xyz=True, use_code=True, include_input=True)
_field_forward = O.field_forward


def zfeature(x_rot: torch.Tensor, x_cam: torch.Tensor, vd: Optional[torch.Tensor], *, num_freqs: int = 6,
             freq_factor: float = 1.5, use_viewdirs: bool = True, use_code_viewdirs: bool = False, normalize_z: bool = True,
             use_xyz: bool = True, use_code: bool = True, include_input: bool = True) -> torch.Tensor:
    """x_rot, x_cam (V, P, 3), vd (V*P, 3) rotated view directions -> z-feature rows (V*P, d_in)."""
    zf = x_rot if normalize_z else x_cam                                    # models.py:183-188
    zf = zf.reshape(-1, 3) if use_xyz else -zf[..., 2:3].reshape(-1, 1)
    code = lambda t: O.positional_encoding(t, num_freqs, freq_factor, include_input)
    if use_code and not use_code_viewdirs:
        zf = code(zf)                                                       # models.py:190-195
    if use_viewdirs:
        assert vd is not None
        zf = torch.cat((zf, vd), dim=1)                                     # models.py:201-209
    if use_code and use_code_viewdirs:
        zf = code(zf)
    return zf


def field_forward(scene: O.Scene, mlp: Dict[str, torch.Tensor], xyz: torch.Tensor, viewdirs: Optional[torch.Tensor], *,
                  num_freqs: int = 6, freq_factor: float = 1.5, n_blocks: int = 5, combine_layer: int = 3,
                  padding: str = "zeros", return_raw: bool = False, yolo: bool = False, emulate_bf16: bool = False,
                  **switches) -> torch.Tensor:
    """``O.field_forward`` with the z-feature of ``switches`` (the keywords of ``zfeature``, defaults = DEFAULT)."""
    SB, P, _ = xyz.shape
    NS = scene.num_views
    R = scene.poses[:, None, :3, :3]
    rep = lambda t: t.unsqueeze(1).expand(-1, NS, *t.shape[1:]).reshape(-1, *t.shape[1:])  # util.py:60-67
    x_w = rep(xyz)                                                          # (SB*NS, P, 3)
    x_rot = torch.matmul(R, x_w.unsqueeze(-1))[..., 0]                      # models.py:169-171
    x_cam = x_rot + scene.poses[:, None, :3, 3]                             # models.py:172
    vd = None
    if viewdirs is not None:
        vd = rep(viewdirs.reshape(SB, P, 3, 1))
        vd = torch.matmul(R, vd).reshape(-1, 3)                             # models.py:201-206
    zf = zfeature(x_rot, x_cam, vd, num_freqs=num_freqs, freq_factor=freq_factor, **{**DEFAULT, **switches})
    if not yolo:
        uv = -x_cam[:, :, :2] / x_cam[:, :, 2:]                             # models.py:220
    else:
        uv = x_cam[:, :, :2] / x_cam[:, :, 2:]                              # models.py:222
    foc = scene.focal.unsqueeze(1)
    cc = scene.c.unsqueeze(1)
    if foc.shape[0] > 1:                                                    # models.py:225-227
        foc = rep(foc)
    if cc.shape[0] > 1:                                                     # models.py:228-230
        cc = rep(cc)
    uv = uv * foc + cc
    lat = O.bilinear_index(scene.latent, uv, scene.latent_scaling, scene.image_shape, padding)
    C = lat.shape[1]
    lat = lat.transpose(1, 2).reshape(-1, C)                                # models.py:244-246
    if yolo:                                                                # models.py:223, 254-264
        nonneg = (x_cam[:, :, 2:] >= 0).reshape(-1, 1)
        lat = torch.where(nonneg | lat.isnan(), torch.zeros_like(lat), lat)
    mlp_in = torch.cat((lat, zf), dim=-1)                                   # models.py:276
    out = O.resnetfc_forward(mlp, mlp_in, C, n_blocks, combine_layer, (NS, P), emulate_bf16=emulate_bf16)
    out = out.reshape(-1, P, out.shape[-1])
    if return_raw or yolo:                                                  # models.py:309-310
        return out.reshape(SB, P, -1)
    rgb = O._f64(torch.sigmoid, out[..., :3])                               # models.py:312-317
    sigma = torch.relu(out[..., 3:4])
    return torch.cat((rgb, sigma), dim=-1).reshape(SB, P, -1)


@contextlib.contextmanager
def switched(**zkw):
    """``O.field_forward`` is ``field_forward`` with ``zkw`` (switches, num_freqs, freq_factor) inside the block."""
    O.field_forward = functools.partial(field_forward, **zkw)
    try:
        yield
    finally:
        O.field_forward = _field_forward
