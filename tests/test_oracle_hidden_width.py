"""CPU pins of tests/bf16_field_reference.py at ResnetFC hidden widths other than 512 (no GPU needed).

The tcgen05 field kernel runs d_hidden <= 256 as a network zero-padded to 256 features (one 256-feature tile) and wider ones
padded to 512.  The padding contributes exact zeros, so the kernel's arithmetic at width h is the reference's at width h:

* with every rounding off the reference is the oracle, bit for bit with streamed latents and both pooling modes, and within
  fp32 summation order with pre-projected wide latents (the projection reassociates lin_z);
* the tight RMS bound still has teeth at the narrow widths: one skipped 128 x 16 MMA slab inside the live features, or 16
  missing lin_z k-columns, moves the reference's RMS by more than twice the bound.
"""
import pytest
import torch

import bf16_field_reference as BR
import helpers as H
import pixel_nerf_yolo_b200.synth as synth
import pooling_oracle as PO
from oracle import pixelnerf_oracle as O

WIDTHS = (64, 128, 256, 384)


def _points(P, seed, num_objs=1):
    g = torch.Generator().manual_seed(seed)
    xyz = (torch.rand(num_objs, P, 3, generator=g) - 0.5) * 0.9
    dirs = torch.nn.functional.normalize(torch.randn(num_objs, P, 3, generator=g), dim=-1)
    return xyz, dirs


def _case(d_hidden, ns=3, C=512, P=96, num_objs=1, n_blocks=5, combine_layer=3):
    scene = H.make_scene_dict(num_views=ns, num_objs=num_objs, C=C)
    mlp = synth.mlp_state(1, d_latent=C, d_hidden=d_hidden, n_blocks=n_blocks, combine_layer=combine_layer)
    xyz, dirs = _points(P, 40 + ns + d_hidden, num_objs)
    return H.oracle_scene(scene), mlp, xyz, dirs


@pytest.mark.parametrize("combine_type", ["average", "max"])
@pytest.mark.parametrize("d_hidden", WIDTHS)
def test_without_rounding_is_the_oracle(d_hidden, combine_type):
    sc, mlp, xyz, dirs = _case(d_hidden, num_objs=2)
    assert mlp["lin_in.weight"].shape[0] == d_hidden
    got = BR.field_forward_bf16(sc, mlp, xyz, dirs, combine_type=combine_type, projected=False, rounding=False)
    with PO.combine_type(combine_type):
        ref = O.field_forward(sc, mlp, xyz, dirs)
    assert torch.equal(got, ref)
    assert ref[..., 3].max() > 0.5 and ref[..., :3].std() > 0.01          # the comparison is not vacuous


@pytest.mark.parametrize("d_hidden", WIDTHS)
def test_unpooled_network_without_rounding_is_the_oracle(d_hidden):
    """The single-view network of conf/default.conf (3 blocks, lin_z before each, no pooling)."""
    sc, mlp, xyz, dirs = _case(d_hidden, ns=1, n_blocks=3, combine_layer=1000)
    kw = dict(n_blocks=3, combine_layer=1000)
    got = BR.field_forward_bf16(sc, mlp, xyz, dirs, projected=False, rounding=False, **kw)
    assert torch.equal(got, O.field_forward(sc, mlp, xyz, dirs, **kw))


@pytest.mark.parametrize("combine_type", ["average", "max"])
@pytest.mark.parametrize("d_hidden", WIDTHS)
def test_projected_latent(d_hidden, combine_type):
    """Pre-projected maps hold n_linz x d_hidden channels; without rounding the projection only reassociates lin_z.  A
    network narrower than its latent gathers pre-projections by default (PixelNeRFNet.projects_latent), the 512-channel maps of
    the default encoder included."""
    sc, mlp, xyz, dirs = _case(d_hidden, C=1792 if d_hidden == 384 else 512)
    with PO.combine_type(combine_type):
        ref = O.field_forward(sc, mlp, xyz, dirs)
    maps = BR.project_maps(sc.latent, mlp, 3)
    assert maps.shape[1] == 3 * d_hidden
    exact = BR.field_forward_bf16(sc, mlp, xyz, dirs, combine_type=combine_type, rounding=False)
    assert max(BR.errors(exact, ref)) < 2e-5
    got = BR.field_forward_bf16(sc, mlp, xyz, dirs, combine_type=combine_type)
    e = BR.errors(got, ref)                          # the bf16 tolerance of the other tests, 1.5x on sigma for max pooling
    assert e[0] < 1e-2 and e[1] < (1.5e-2 if combine_type == "max" else 1e-2), e
    assert not torch.equal(got, BR.field_forward_bf16(sc, mlp, xyz, dirs, combine_type=combine_type, projected=False))


# ------------------------------------------------------------------------------------------------ the bound has teeth
def _faults(mlp, d_hidden):
    """Faults of the size of one kernel mistake inside the live features: one 128-row x 16-k MMA slab of blocks.2.fc_0 (the
    last k-columns of the last live 128 rows), and 16 k-columns of lin_z.1."""
    slab = dict(mlp)
    w = slab["blocks.2.fc_0.weight"].clone()
    w[max(0, d_hidden - 128):d_hidden, d_hidden - 16:d_hidden] = 0
    slab["blocks.2.fc_0.weight"] = w
    linz = dict(mlp)
    w = linz["lin_z.1.weight"].clone()
    w[:, 64:80] = 0
    linz["lin_z.1.weight"] = w
    return {"skipped MMA slab": slab, "lin_z k-columns": linz}


@pytest.mark.parametrize("combine_type", ["average", "max"])
@pytest.mark.parametrize("ns", [3, 8])
@pytest.mark.parametrize("d_hidden", [128, 256])
def test_tight_bound_sees_one_mma_fault(d_hidden, ns, combine_type):
    sc, mlp, xyz, dirs = _case(d_hidden, ns=ns, P=400)
    bound = BR.tight_bound(combine_type)
    ref = BR.field_forward_bf16(sc, mlp, xyz, dirs, combine_type=combine_type)
    for name, bad in _faults(mlp, d_hidden).items():
        e = BR.rms_errors(BR.field_forward_bf16(sc, bad, xyz, dirs, combine_type=combine_type), ref)
        print(f"d_hidden={d_hidden} NS={ns} {combine_type} {name}: RMS moves rgb {e[0]:.2e} sigma {e[1]:.2e} (bound {bound:.1e})")
        assert max(e) > 2 * bound, (name, e)
