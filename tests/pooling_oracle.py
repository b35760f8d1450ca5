"""Both view-pooling modes of ResnetFC for the CPU oracle.

``oracle/pixelnerf_oracle.py`` restates ResnetFC.forward (src/model/resnetfc.py:134-186) for ``combine_type = "average"`` and
is pinned by outputs of the reference itself (tests/golden/).  The reference's other mode, ``"max"``, pools the views of a
point with ``util.combine_interleaved`` (src/util/util.py:489-499) as ``torch.max(t, dim=1)[0]``.  The reference is not
available to produce goldens for it, so this restatement is pinned two ways instead: for ``"average"`` it equals the oracle
bit for bit, and its max pooling and autograd equal a direct ``torch.max`` restatement (tests/test_oracle_pooling.py).

``with combine_type("max"):`` routes the oracle's ``field_forward`` / ``render`` / ``yolo_render`` through this ResnetFC.
"""
import contextlib
import functools
from typing import Dict, Optional, Tuple

import torch

from oracle import pixelnerf_oracle as O


def combine_interleaved(t: torch.Tensor, inner_dims: Tuple[int, ...], agg_type: str = "average") -> torch.Tensor:
    """util.py:489-499: (B * prod(inner_dims), ...) -> (B * prod(inner_dims[1:]), ...), reduced over inner_dims[0]."""
    if len(inner_dims) == 1 and inner_dims[0] == 1:
        return t
    t = t.reshape(-1, *inner_dims, *t.shape[1:])
    if agg_type == "average":
        return torch.mean(t, dim=1)
    if agg_type == "max":
        return torch.max(t, dim=1)[0]
    raise NotImplementedError(agg_type)


def resnetfc_forward(p: Dict[str, torch.Tensor], zx: torch.Tensor, d_latent: int, n_blocks: int, combine_layer: int,
                     inner_dims: Tuple[int, int], emulate_bf16: bool = False, combine_type: str = "average",
                     record: Optional[dict] = None) -> torch.Tensor:
    """oracle.resnetfc_forward with the pooling mode as an argument.  ``record``: if given, receives the pre-pooling
    activations as record["x_views"] (objects, NS, points, H), for tests that need to know how close two views come."""
    if emulate_bf16:
        def lin(x, w, b, trunk=True):
            return torch.nn.functional.linear(O._bf16_ste(x), O._bf16_ste(w), b) if trunk else torch.nn.functional.linear(x, w, b)
    else:
        def lin(x, w, b, trunk=True):
            return torch.nn.functional.linear(x, w, b)
    z = zx[..., :d_latent]
    x = zx[..., d_latent:]
    x = lin(x, p["lin_in.weight"], p["lin_in.bias"])                        # resnetfc.py:149
    for b in range(n_blocks):
        if b == combine_layer:                                              # resnetfc.py:154,172-174
            ns, pts = inner_dims
            if record is not None:
                record["x_views"] = x.detach().reshape(-1, ns, pts, x.shape[-1])
            x = combine_interleaved(x.reshape(-1, x.shape[-1]), (ns, pts), combine_type).reshape(-1, x.shape[-1])
        if d_latent > 0 and b < combine_layer:
            x = x + lin(z, p[f"lin_z.{b}.weight"], p[f"lin_z.{b}.bias"])    # resnetfc.py:176-182
        net = lin(torch.relu(x), p[f"blocks.{b}.fc_0.weight"], p[f"blocks.{b}.fc_0.bias"])
        dx = lin(torch.relu(net), p[f"blocks.{b}.fc_1.weight"], p[f"blocks.{b}.fc_1.bias"])
        x = x + dx                                                          # resnetfc.py:53-62
    xr = O._bf16_ste(torch.relu(x)) if emulate_bf16 else torch.relu(x)
    return lin(xr, p["lin_out.weight"], p["lin_out.bias"], trunk=False)     # resnetfc.py:185


@contextlib.contextmanager
def combine_type(mode: str, record: Optional[dict] = None):
    """Inside the block, every ResnetFC evaluation of the oracle pools the views with ``mode``."""
    saved = O.resnetfc_forward
    O.resnetfc_forward = functools.partial(resnetfc_forward, combine_type=mode, record=record)
    try:
        yield
    finally:
        O.resnetfc_forward = saved
