"""Hand-offs at the edges of the field kernel's work unit (`-m gpu`): the start of a tile (x tile 0 is handed to its epilogue in
the middle of the first lin_z layer; the gather writes the next tile's z-features as soon as lin_in has read the current ones,
before the latent tile is free), the end of a pre-combine tile (view pooling, then the next tile's lin_in) and the step from the
pre-combine to the post-combine phase, across consecutive super groups of one CTA pair.

Every case runs at least three super groups per CTA pair with a partial last super group, so pairs run three and four super
groups (odd and even counts) and every barrier parity wraps.  A column's arithmetic does not depend on where it sits, so the big
launch must equal, bit for bit, the same points evaluated in launches of under one wave each; a strided subset is held to the
bounds of tests/test_gpu_field_coverage.py (1e-2 against the fp32 oracle, the tight RMS bound against the bf16 reference).

Matrix: NS in {1, 2, 3, 8} x hidden tiles MT in {1, 2} (d_hidden 256 / 512) x latents {512 channels in one pass, 576 streamed in
two passes, 1792 pre-projected}; plus the unpooled single-view network and max pooling at both MT.
"""
import math

import pytest
import torch

import helpers as H
from test_gpu_hidden_width import Net, _check, _points

pytestmark = pytest.mark.gpu

LATENTS = [(512, False), (576, False), (1792, True)]
CASES = [(ns, d_hidden, C, project, 5, 3, "average") for ns in (1, 2, 3, 8) for d_hidden in (256, 512) for C, project in LATENTS]
CASES += [(1, d_hidden, 512, False, 5, 5, "average") for d_hidden in (256, 512)]        # unpooled: G = 1, lin_out after the tiles
CASES += [(8, d_hidden, 512, False, 5, 3, "max") for d_hidden in (256, 512)]


@pytest.fixture(scope="module")
def lib():
    from pixel_nerf_yolo_b200 import _lib
    assert torch.cuda.is_available()
    _lib.require_device(torch.device("cuda", 0))
    return _lib.load()


@pytest.mark.parametrize("ns,d_hidden,C,project,n_blocks,combine_layer,combine_type", CASES)
def test_work_unit_boundaries(lib, ns, d_hidden, C, project, n_blocks, combine_layer, combine_type):
    pp = 64 // ns
    g = 64 // pp                                         # tile pairs per super group
    per_sg = 2 * g * pp                                  # points of one super group (one object)
    n_pairs = torch.cuda.get_device_properties(0).multi_processor_count // 2
    P = 3 * n_pairs * per_sg + per_sg // 2 + 1           # 3 * n_pairs + 1 super groups, the last one partial
    scene = H.make_scene_dict(num_objs=1, num_views=ns, C=C)
    m = Net(scene, d_hidden, n_blocks=n_blocks, combine_layer=combine_layer, combine_type=combine_type, project=project)
    assert m.projected == project
    xyz, dirs = _points(P, 1100 + 10 * ns + d_hidden // 64 + C, 1)
    big = m(xyz, dirs)
    step = n_pairs * per_sg // 2                         # about half a wave of super groups
    for a in range(0, P, step):
        part = m(xyz[:, a:a + step].contiguous(), dirs[:, a:a + step].contiguous())
        assert torch.equal(big[:, a:a + step], part), (a, (big[:, a:a + step] - part).abs().max().item())
    stride = math.ceil(P / 512)
    xs, ds = xyz[:, ::stride].contiguous(), dirs[:, ::stride].contiguous()
    case = f"boundaries NS={ns} C={C} projected={project} ({n_blocks}, {combine_layer}) {combine_type} P={P}"
    ref = _check(case, m, big[:, ::stride], xs, ds)
    assert ref[..., 3].max() > 0.5 and ref[..., :3].std() > 0.01
