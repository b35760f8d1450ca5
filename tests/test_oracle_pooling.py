"""View pooling of ResnetFC on the CPU (no GPU needed): the max-pooling restatement of the oracle (tests/pooling_oracle.py)
and the Python side of both pooling settings -- combine_type "max", and the single-view network that never pools
(combine_layer >= n_blocks, the shape of conf/default.conf)."""
import copy

import pytest
import torch

import helpers as H
import pixel_nerf_yolo_b200.synth as synth
import pooling_oracle as PO
from oracle import pixelnerf_oracle as O


def _zx(n_rows, d_latent=512, d_in=42, seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.cat((torch.randn(n_rows, d_latent, generator=g) * 0.5, torch.randn(n_rows, d_in, generator=g)), dim=-1)


def test_average_restatement_equals_oracle():
    """For combine_type "average" the restatement is the (golden-pinned) oracle, bit for bit."""
    p = synth.mlp_state(3)
    zx = _zx(2 * 3 * 7)
    ref = O.resnetfc_forward(p, zx, 512, 5, 3, (3, 7))
    assert torch.equal(PO.resnetfc_forward(p, zx, 512, 5, 3, (3, 7)), ref)
    assert torch.equal(PO.resnetfc_forward(p, zx, 512, 5, 3, (3, 7), emulate_bf16=True),
                       O.resnetfc_forward(p, zx, 512, 5, 3, (3, 7), emulate_bf16=True))


@pytest.mark.parametrize("ns", [2, 3, 5])
def test_max_pooling_and_its_gradient_match_torch_max(ns):
    """Max pooling as a direct restatement: the residual stream before block combine_layer, reduced with torch.max over the
    views; autograd sends the pooled gradient to the first maximal view only, and the per-view routing sums to it."""
    p = {k: v.clone().requires_grad_(True) for k, v in synth.mlp_state(4).items()}
    pts = 6
    zx = _zx(2 * ns * pts, seed=ns).requires_grad_(True)
    rec = {}
    out = PO.resnetfc_forward(p, zx, 512, 5, 3, (ns, pts), combine_type="max", record=rec)
    assert out.shape == (2 * pts, 4)
    # direct restatement: blocks [0, 3) per view, torch.max over the view axis, blocks [3, 5), lin_out
    lin = torch.nn.functional.linear
    z, x = zx[:, :512], lin(zx[:, 512:], p["lin_in.weight"], p["lin_in.bias"])
    for b in range(3):
        x = x + lin(z, p[f"lin_z.{b}.weight"], p[f"lin_z.{b}.bias"])
        x = x + lin(torch.relu(lin(torch.relu(x), p[f"blocks.{b}.fc_0.weight"], p[f"blocks.{b}.fc_0.bias"])),
                    p[f"blocks.{b}.fc_1.weight"], p[f"blocks.{b}.fc_1.bias"])
    xv = x.reshape(2, ns, pts, -1)
    assert torch.equal(rec["x_views"], xv.detach())
    pooled, win = torch.max(xv, dim=1)
    x = pooled.reshape(-1, pooled.shape[-1])
    for b in range(3, 5):
        x = x + lin(torch.relu(lin(torch.relu(x), p[f"blocks.{b}.fc_0.weight"], p[f"blocks.{b}.fc_0.bias"])),
                    p[f"blocks.{b}.fc_1.weight"], p[f"blocks.{b}.fc_1.bias"])
    ref = lin(torch.relu(x), p["lin_out.weight"], p["lin_out.bias"])
    assert torch.equal(out, ref)
    # gradient routing of the pooling step
    g_pooled = torch.randn_like(pooled)
    g_views, = torch.autograd.grad(PO.combine_interleaved(xv.reshape(-1, xv.shape[-1]), (ns, pts), "max"), xv, g_pooled)
    routed = torch.zeros_like(xv).scatter_(1, win.unsqueeze(1), g_pooled.unsqueeze(1))
    assert torch.equal(g_views, routed)
    assert torch.allclose(g_views.sum(1), g_pooled)
    assert ((g_views != 0).sum(1) <= 1).all()
    # ties go to the first maximal view, as torch.max(dim) documents
    t = torch.tensor([[1.0, 3.0], [3.0, 3.0], [2.0, 0.0]], requires_grad=True)
    PO.combine_interleaved(t, (3, 1), "max").sum().backward()
    assert torch.equal(t.grad, torch.tensor([[0.0, 1.0], [1.0, 0.0], [0.0, 0.0]]))
    # end to end through autograd: every parameter receives a gradient equal to the direct restatement's
    w = torch.randn_like(out)
    ga = torch.autograd.grad((out * w).sum(), [zx] + list(p.values()))
    gb = torch.autograd.grad((ref * w).sum(), [zx] + list(p.values()))
    for a, b in zip(ga, gb):
        assert torch.allclose(a, b, rtol=1e-5, atol=1e-6)


def test_combine_type_routes_the_oracle_field():
    """``with combine_type(...)`` changes the pooling of O.field_forward (and restores the oracle afterwards)."""
    scene = H.make_scene_dict(num_views=3, feat=8)
    g = torch.Generator().manual_seed(1)
    xyz = (torch.rand(1, 20, 3, generator=g) - 0.5) * 0.8
    dirs = torch.nn.functional.normalize(torch.randn(1, 20, 3, generator=g), dim=-1)
    sc, p = H.oracle_scene(scene), synth.mlp_state(1)
    avg = O.field_forward(sc, p, xyz, dirs)
    with PO.combine_type("average"):
        assert torch.equal(O.field_forward(sc, p, xyz, dirs), avg)
    with PO.combine_type("max"):
        mx = O.field_forward(sc, p, xyz, dirs)
    assert not torch.allclose(mx, avg, atol=1e-3)
    assert torch.equal(O.field_forward(sc, p, xyz, dirs), avg)


def test_single_view_network_runs_every_block():
    """combine_layer >= n_blocks (conf/default.conf): no pooling, lin_z before every block; with one view both modes agree."""
    p = synth.mlp_state(5, n_blocks=3, combine_layer=1000)
    assert sorted(k for k in p if k.startswith("lin_z")) == [f"lin_z.{b}.{t}" for b in range(3) for t in ("bias", "weight")]
    zx = _zx(9)
    ref = O.resnetfc_forward(p, zx, 512, 3, 1000, (1, 9))
    for mode in ("average", "max"):
        assert torch.equal(PO.resnetfc_forward(p, zx, 512, 3, 1000, (1, 9), combine_type=mode), ref)


def _conf(**mlp):
    conf = copy.deepcopy(H.MODEL_CONF)
    for k in ("mlp_coarse", "mlp_fine"):
        for key in ("combine_layer", "combine_type"):
            conf[k].pop(key)
        conf[k].update(mlp)
    return conf


def test_default_conf_shape_builds():
    """A network shaped like conf/default.conf (3 blocks, no combine_layer: the class default 1000) builds through make_model;
    the C view clamps combine_layer to n_blocks."""
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.model import make_model
    net = make_model(ConfigTree.from_dict(_conf(n_blocks=3)))
    for mlp in (net.mlp_coarse, net.mlp_fine):
        assert (mlp.n_blocks, mlp.combine_layer, mlp.combine_type, len(mlp.lin_z)) == (3, 1000, "average", 3)
        assert not mlp.pools_views()
        cp = mlp.c_params()
        assert (cp.n_blocks, cp.combine_layer, cp.combine_type) == (3, 3, 0)
    mlp.load_state_dict(synth.mlp_state(1, n_blocks=3, combine_layer=1000))


def test_max_conf_builds():
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.model import make_model
    net = make_model(ConfigTree.from_dict(_conf(n_blocks=5, combine_layer=3, combine_type="max")))
    for mlp in (net.mlp_coarse, net.mlp_fine):
        assert (mlp.combine_layer, mlp.combine_type) == (3, "max") and mlp.pools_views()
        assert (mlp.c_params().combine_layer, mlp.c_params().combine_type) == (3, 1)
    net.mlp_coarse.load_state_dict(synth.mlp_state(1))


def test_single_view_network_refuses_several_views_up_front():
    """A network that never pools cannot take NS > 1 source views: encode and the stand-alone ResnetFC raise
    NotImplementedError before any kernel is involved."""
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.model import make_model
    net = make_model(ConfigTree.from_dict(_conf(n_blocks=3)))
    poses = torch.eye(4).expand(1, 3, 4, 4)
    with pytest.raises(NotImplementedError, match="one view"):
        net.encode(torch.zeros(1, 3, 3, 32, 32), poses, torch.tensor(30.0))
    with pytest.raises(NotImplementedError, match="one view"):
        net.mlp_coarse(_zx(6), combine_inner_dims=(3, 2))
    from pixel_nerf_yolo_b200.model.resnetfc import ResnetFC
    with pytest.raises(NotImplementedError):
        ResnetFC(42, 4, d_latent=512, d_hidden=512, combine_type="min")


def test_pooling_mode_needs_a_pooling_step():
    """combine_type "max" selects how the views are pooled before block combine_layer; a network whose combine_layer is at or
    past its last block never pools, so the mode cannot apply and is refused rather than silently ignored."""
    from pixel_nerf_yolo_b200.model.resnetfc import ResnetFC
    with pytest.raises(NotImplementedError, match="combine_layer < n_blocks"):
        ResnetFC(42, 4, d_latent=512, d_hidden=512, combine_type="max")                 # class default combine_layer = 1000
    with pytest.raises(NotImplementedError, match="combine_layer < n_blocks"):
        ResnetFC(42, 4, n_blocks=3, d_latent=512, d_hidden=512, combine_layer=3, combine_type="max")
    assert ResnetFC(42, 4, n_blocks=3, d_latent=512, d_hidden=512, combine_layer=2, combine_type="max").pools_views()
    assert not ResnetFC(42, 4, n_blocks=3, d_latent=512, d_hidden=512).pools_views()
