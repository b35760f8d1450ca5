"""CPU pins of tests/bf16_field_reference.py, the restatement of the tcgen05 field kernel's bf16 arithmetic (no GPU needed).

* With every rounding off it is the oracle: bit for bit for average pooling, and pooling_oracle's restatement for max.
* On inputs the kernel's roundings leave unchanged (bf16-representable maps and lin_out weights) it is the training tests'
  bf16-operand emulation, ``O.field_forward(..., emulate_bf16=True)``, bit for bit.
* Its tight bound ``TIGHT`` (on the RMS error over points) has teeth: faults of the size of one skipped MMA move it by more
  than twice the bound, with either pooling mode.
"""
import pytest
import torch

import bf16_field_reference as BR
import helpers as H
import pixel_nerf_yolo_b200.synth as synth
import pooling_oracle as PO
from oracle import pixelnerf_oracle as O


def _points(P, seed, num_objs=1):
    g = torch.Generator().manual_seed(seed)
    xyz = (torch.rand(num_objs, P, 3, generator=g) - 0.5) * 0.9
    dirs = torch.nn.functional.normalize(torch.randn(num_objs, P, 3, generator=g), dim=-1)
    return xyz, dirs


def _case(ns, n_blocks=5, combine_layer=3, C=512, P=96, num_objs=1):
    scene = H.make_scene_dict(num_views=ns, num_objs=num_objs, C=C)
    mlp = synth.mlp_state(1, d_latent=C, n_blocks=n_blocks, combine_layer=combine_layer)
    xyz, dirs = _points(P, 40 + ns, num_objs)
    return H.oracle_scene(scene), mlp, xyz, dirs


@pytest.mark.parametrize("ns,n_blocks,combine_layer", [(1, 3, 3), (3, 5, 3), (8, 4, 2), (2, 8, 7)])
def test_without_rounding_is_the_oracle(ns, n_blocks, combine_layer):
    sc, mlp, xyz, dirs = _case(ns, n_blocks, combine_layer, num_objs=2)
    kw = dict(n_blocks=n_blocks, combine_layer=combine_layer)
    got = BR.field_forward_bf16(sc, mlp, xyz, dirs, rounding=False, **kw)
    assert torch.equal(got, O.field_forward(sc, mlp, xyz, dirs, **kw))
    if ns > 1:
        got = BR.field_forward_bf16(sc, mlp, xyz, dirs, rounding=False, combine_type="max", **kw)
        with PO.combine_type("max"):
            assert torch.equal(got, O.field_forward(sc, mlp, xyz, dirs, **kw))


def test_without_rounding_yolo_is_the_oracle():
    sc, mlp, xyz, dirs = _case(3)
    mlp = synth.mlp_state(31, d_out=28)
    sc = O.encode_cameras(sc.latent, torch.linalg.inv(H.make_scene_dict()["poses"][0]), torch.tensor(131.25), (128, 128),
                          num_views=3, yolo=True)
    got = BR.field_forward_bf16(sc, mlp, xyz, dirs, yolo=True, rounding=False)
    assert torch.equal(got, O.field_forward(sc, mlp, xyz, dirs, yolo=True))


@pytest.mark.parametrize("combine_type", ["average", "max"])
def test_on_representable_inputs_is_the_emulation(combine_type):
    """The only roundings the bf16-operand emulation does not do are those of the maps and of lin_out's weights."""
    sc, mlp, xyz, dirs = _case(3)
    sc.latent = BR.bf16(sc.latent)
    mlp = dict(mlp, **{"lin_out.weight": BR.bf16(mlp["lin_out.weight"])})
    got = BR.field_forward_bf16(sc, mlp, xyz, dirs, combine_type=combine_type)
    with PO.combine_type(combine_type):
        assert torch.equal(got, O.field_forward(sc, mlp, xyz, dirs, emulate_bf16=True))


def test_rounding_is_not_the_emulation():
    """...and on the synthetic fp32 maps those two roundings do move the output (by about as much as a kernel fault)."""
    sc, mlp, xyz, dirs = _case(3, P=200)
    e = BR.errors(BR.field_forward_bf16(sc, mlp, xyz, dirs), O.field_forward(sc, mlp, xyz, dirs, emulate_bf16=True))
    assert max(e) > 5e-4, e


@pytest.mark.parametrize("combine_type", ["average", "max"])
def test_projected_latent(combine_type):
    """Pre-projected wide maps: without rounding the projection only reassociates lin_z (fp32 summation order); with it, the
    result stays within the bf16 tolerance of the oracle."""
    C = 1792
    sc, mlp, xyz, dirs = _case(3, C=C)
    with PO.combine_type(combine_type):
        ref = O.field_forward(sc, mlp, xyz, dirs)
    exact = BR.field_forward_bf16(sc, mlp, xyz, dirs, combine_type=combine_type, rounding=False)
    assert max(BR.errors(exact, ref)) < 2e-5
    got = BR.field_forward_bf16(sc, mlp, xyz, dirs, combine_type=combine_type)
    assert max(BR.errors(got, ref)) < 1e-2
    # the projected arithmetic is not the streamed one: they round different things
    streamed = BR.field_forward_bf16(sc, mlp, xyz, dirs, combine_type=combine_type, projected=False)
    assert not torch.equal(got, streamed)


# ------------------------------------------------------------------------------------------------ the bound has teeth
def _faults(mlp):
    """Faults of the size of one kernel mistake, applied to the weights the reference is given."""
    slab = dict(mlp)                       # one 128-row x 16-k MMA slab of blocks.2.fc_0 skipped (one CTA's half of one MMA)
    w = slab["blocks.2.fc_0.weight"].clone()
    w[128:256, 496:512] = 0
    slab["blocks.2.fc_0.weight"] = w
    linz = dict(mlp)                       # 16 k-columns of lin_z.1 missing
    w = linz["lin_z.1.weight"].clone()
    w[:, 64:80] = 0
    linz["lin_z.1.weight"] = w
    return {"skipped MMA slab": slab, "lin_z k-columns": linz}


@pytest.fixture(scope="module")
def teeth_cases():
    cases = {}
    for ns in (3, 8):
        sc, mlp, xyz, dirs = _case(ns, P=400)
        cases[ns] = (sc, mlp, xyz, dirs)
    return cases


@pytest.mark.parametrize("combine_type", ["average", "max"])
@pytest.mark.parametrize("ns", [3, 8])
def test_tight_bound_sees_one_mma_fault(teeth_cases, ns, combine_type):
    sc, mlp, xyz, dirs = teeth_cases[ns]
    bound = BR.tight_bound(combine_type)
    ref = BR.field_forward_bf16(sc, mlp, xyz, dirs, combine_type=combine_type)
    for name, bad in _faults(mlp).items():
        e = BR.rms_errors(BR.field_forward_bf16(sc, bad, xyz, dirs, combine_type=combine_type), ref)
        print(f"NS={ns} {combine_type} {name}: RMS moves rgb {e[0]:.2e} sigma {e[1]:.2e} (bound {bound:.1e})")
        assert max(e) > 2 * bound, (name, e)


@pytest.mark.parametrize("ns", [3, 8])
def test_report_smallest_bias_fault_seen(teeth_cases, ns):
    """A bias read from the wrong slot changes one feature by a small offset.  The response is linear in the offset (a few
    ReLU flips aside), so the smallest offset on feature 300 of blocks.4.fc_1 that moves the output's RMS by twice the bound
    is reported from the response to 0.02 and then checked."""
    sc, mlp, xyz, dirs = teeth_cases[ns]
    ref = BR.field_forward_bf16(sc, mlp, xyz, dirs)

    def moved(delta):
        bad = dict(mlp)
        b = bad["blocks.4.fc_1.bias"].clone()
        b[300] += delta
        bad["blocks.4.fc_1.bias"] = b
        return max(BR.rms_errors(BR.field_forward_bf16(sc, bad, xyz, dirs), ref))

    smallest = 2 * BR.TIGHT / (moved(0.02) / 0.02)
    print(f"NS={ns}: a bias offset of {smallest:.3f} on one feature of blocks.4.fc_1 moves the output's RMS by 2x the bound "
          f"({BR.TIGHT:.1e})")
    assert moved(1.25 * smallest) > 2 * BR.TIGHT
