"""GPU parity tests added in round 2 (all through the C-ABI, `-m gpu`):

* the headline workload against the ORACLE (not against the repo's own fp32 path): a 1 024-ray strided subset of the
  16 384-ray bf16 render of the 128x128 image;
* end-to-end n_coarse = 256 x 5 source views;
* BASELINE config 4 at its true shape (3 x 1792 x 80 x 80 maps, 640-px image, focal 656.25) on a ray subset, both
  `project_wide_latent` modes, through the single-call render;
* ray slicing over forked streams (pnr_render_args.n_splits) is bit-identical to one slice;
* a ray batch for a different number of objects than encode() saw is refused (Python assert and C-level total check);
* util.gen_rays_yolo drop-in vs the reference's golden vectors.

Tolerances: BASELINE north_star -- bf16 MLP operands max-abs <= 1e-2 on rgb / depth.
"""
import copy
import os

import numpy as np
import pytest
import torch

import helpers as H
import pixel_nerf_yolo_b200.synth as synth
from oracle import pixelnerf_oracle as O

pytestmark = pytest.mark.gpu
T = torch.from_numpy
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _renderer(**kw):
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.render import NeRFRenderer
    conf = dict(H.RENDER_CONF)
    conf.update(kw)
    return NeRFRenderer.from_conf(ConfigTree.from_dict(conf)).eval().cuda()


def _noise_obj(noise):
    return O.RenderNoise(noise["coarse"], noise["fine_u"], noise["fine_jitter"], noise["depth"])


def test_full_image_bf16_subset_matches_oracle():
    """The bench workload's size: render all 16 384 rays of the 128x128 view in ONE bf16 call, then check every 16th ray
    (1 024 rays) against the oracle fed the same rays and the same noise rows."""
    scene = H.make_scene_dict(feat=64)
    net = H.build_net(scene, precision="bf16")
    rays = synth.target_rays(128)
    B = rays.shape[1]
    noise = H.make_noise(B, seed=4)
    r = _renderer()
    r.noise_override = {k: v.cuda() for k, v in noise.items()}
    with torch.no_grad():
        res = r(net, rays.cuda())
    sub = torch.arange(0, B, 16)
    ref = O.render(H.oracle_scene(scene), synth.mlp_state(1), synth.mlp_state(2), rays[:, sub],
                   _noise_obj({k: v[sub] for k, v in noise.items()}))
    for lvl in ("coarse", "fine"):
        e_rgb = (res[lvl].rgb[:, sub].cpu() - ref[lvl]["rgb"]).abs().max().item()
        e_d = (res[lvl].depth[:, sub].cpu() - ref[lvl]["depth"]).abs().max().item()
        assert e_rgb < 1e-2 and e_d < 1e-2, (lvl, e_rgb, e_d)
    assert 0.2 < ref["fine"]["weights"].sum(-1).mean() < 0.999


def test_render_kc256_five_views_matches_oracle():
    """BASELINE config 5's heaviest corner end to end: 256 coarse + 32 fine samples, 5 source views."""
    scene = H.make_scene_dict(num_views=5)
    net = H.build_net(scene, precision="bf16")
    B = 96
    rays = H.rays_subset(1, B, seed=11)
    noise = H.make_noise(B, seed=12, kc=256)
    r = _renderer(n_coarse=256)
    r.noise_override = {k: v.cuda() for k, v in noise.items()}
    with torch.no_grad():
        res = r(net, rays.cuda(), want_weights=True)
    ref = O.render(H.oracle_scene(scene), synth.mlp_state(1), synth.mlp_state(2), rays, _noise_obj(noise), n_coarse=256)
    assert res.fine.weights.shape == (1, B, 288)
    for lvl in ("coarse", "fine"):
        assert (res[lvl].rgb.cpu() - ref[lvl]["rgb"]).abs().max() < 1e-2
        assert (res[lvl].depth.cpu() - ref[lvl]["depth"]).abs().max() < 1e-2


@pytest.mark.parametrize("project", [True, False])
def test_config4_true_shape_subset_matches_oracle(project):
    """BASELINE config 4 at its true shape: 3 x 1792 x 80 x 80 maps, 640x640 image (focal 656.25), NeRFRenderer 64+32+16, on
    a 256-ray subset; `project_wide_latent` True (lin_z pre-projections gathered, PNR_SCENE_PROJECTED, one scene per
    network) and False (the 1 792-wide lin_z streamed through the kernel), both through pnr_render_forward."""
    C = 1792
    conf = copy.deepcopy(H.MODEL_CONF)
    conf["encoder"] = {"backbone": "custom", "pretrained": False, "num_layers": 4, "index_padding": "zeros"}
    scene = H.make_scene_dict(num_objs=1, num_views=3, feat=80, size=640, C=C)
    assert abs(float(scene["focal"]) - 656.25) < 1e-3
    net = H.build_net(scene, precision="bf16", model_conf=conf)
    net.project_wide_latent = project
    allr = synth.target_rays(640)
    pick = T(np.random.default_rng(3).choice(640 * 640, 256, replace=False)).long()
    rays = allr[:, pick].contiguous()
    noise = H.make_noise(256, seed=6)
    r = _renderer()
    r.noise_override = {k: v.cuda() for k, v in noise.items()}
    assert net.fused_render_ready()
    with torch.no_grad():
        res = r(net, rays.cuda())
    assert r.last_launches == 4
    ref = O.render(H.oracle_scene(scene), synth.mlp_state(1, d_latent=C), synth.mlp_state(2, d_latent=C), rays, _noise_obj(noise))
    for lvl in ("coarse", "fine"):
        e_rgb = (res[lvl].rgb.cpu() - ref[lvl]["rgb"]).abs().max().item()
        e_d = (res[lvl].depth.cpu() - ref[lvl]["depth"]).abs().max().item()
        assert e_rgb < 1e-2 and e_d < 1e-2, (project, lvl, e_rgb, e_d)


@pytest.mark.parametrize("n_rays", [2048, 777])
def test_sliced_render_is_bit_identical(n_rays):
    """pnr_render_args.n_splits: the batch rendered as 2 / 3 slices on forked streams (tail of one field launch under the head
    of the next) equals the one-slice render bit for bit, outputs and weights; n_splits = 0 picks slicing for small batches."""
    scene = H.make_scene_dict(feat=32)
    net = H.build_net(scene, precision="bf16")
    rays = synth.target_rays(128)[:, :n_rays].contiguous().cuda()
    noise = {k: v.cuda() for k, v in H.make_noise(n_rays, seed=5).items()}
    outs = {}
    for splits in (1, 2, 3, 0):
        r = _renderer()
        r.n_splits = splits
        r.noise_override = noise
        with torch.no_grad():
            outs[splits] = r(net, rays, want_weights=True)
        expect = {1: 4, 2: 8, 3: 12, 0: 8 if n_rays >= 512 else 4}[splits]
        assert r.last_launches == expect, (splits, r.last_launches)
    torch.cuda.synchronize()
    for splits in (2, 3, 0):
        for lvl in ("coarse", "fine"):
            for k in ("rgb", "depth", "weights"):
                assert torch.equal(outs[splits][lvl][k], outs[1][lvl][k]), (splits, lvl, k)


def test_object_count_mismatch_is_refused():
    """A scene encoded for 2 objects must not be rendered with a 1-object ray batch (the kernels take SB from the scene and
    would run past the ray / output buffers): Python asserts, and the C entry points check the buffer totals themselves."""
    from pixel_nerf_yolo_b200 import _lib
    scene = H.make_scene_dict(num_objs=2)
    net = H.build_net(scene, precision="bf16")
    r = _renderer()
    rays1 = H.rays_subset(1, 40).cuda()
    with pytest.raises(AssertionError):
        with torch.no_grad():
            r(net, rays1)
    # C level: a pnr_points whose buffers hold 1 object's points against a 2-object scene
    lib = _lib.load()
    sc, keep = net._scene(fp32_maps=False)
    xyz = torch.zeros(1, 64, 3, device="cuda")
    pts = _lib.points_xyz(xyz, xyz)
    out = torch.empty(2, 64, 4, device="cuda")
    ws = torch.empty(lib.pnr_field_workspace_bytes(sc, pts, _lib.PREC_BF16), dtype=torch.uint8, device="cuda")
    rc = lib.pnr_field_forward(sc, pts, net.mlp_coarse.c_params(), net.mlp_coarse.packed().data_ptr(), out.data_ptr(),
                               ws.data_ptr(), ws.numel(), _lib.PREC_BF16, 6, 1.5, _lib.stream_ptr(xyz.device))
    assert rc == -1 and b"disagree" in lib.pnr_last_error()


def test_gen_rays_yolo_matches_reference_golden():
    """util.gen_rays_yolo (src/util/util.py:808-876) vs the unmodified reference's output.  Tolerance 2e-6: the reference's
    two small matmuls go through torch's sgemm, whose accumulation order is not specified; the kernel uses one fma chain."""
    from pixel_nerf_yolo_b200.util import gen_rays_yolo
    g = np.load(os.path.join(GOLD, "reference_rays_yolo.npz"))
    w2c = T(g["w2c"]).cuda()
    r = gen_rays_yolo(w2c, 20, 15, T(g["focal"]), T(g["c"]), 0.5, 6.0)
    assert r.shape == (3, 15, 20, 8)
    np.testing.assert_allclose(r.cpu().numpy(), g["rays_20x15"], atol=2e-6, rtol=2e-6)
    r1 = gen_rays_yolo(w2c[:1], 1, 1, T(g["focal"]), T(g["c"]), 0.1, 2.0)
    np.testing.assert_allclose(r1.cpu().numpy(), g["rays_1x1"], atol=2e-6, rtol=2e-6)
    # a YoloTrainer-sized grid (640 / 32 = 20 cells) against the oracle restatement
    ref = O.gen_rays_yolo(T(g["w2c"]), 20, 20, [20.5, 20.5], [10.0, 10.0], 0.5, 6.0)
    big = gen_rays_yolo(w2c, 20, 20, torch.tensor([20.5, 20.5]), torch.tensor([10.0, 10.0]), 0.5, 6.0)
    np.testing.assert_allclose(big.cpu().numpy(), ref.numpy(), atol=2e-6, rtol=2e-6)


def test_render_plan_follows_state_changes():
    """The single-call render keeps a prepared argument block per renderer; a new encode, new weights (load_state_dict or an
    in-place optimizer-style update) or changed sampling settings must all be picked up on the next call."""
    scene = H.make_scene_dict(feat=16)
    net = H.build_net(scene, precision="bf16")
    rays = H.rays_subset(1, 64).cuda()
    noise = {k: v.cuda() for k, v in H.make_noise(64).items()}
    r = _renderer()
    r.noise_override = noise

    def go():
        with torch.no_grad():
            return r(net, rays).fine.rgb.clone()
    a = go()
    assert torch.equal(a, go())
    net.encoder.set_latent(net.encoder.latent * 0.5)                      # new scene
    b = go()
    assert not torch.equal(a, b)
    fresh = H.build_net(scene, precision="bf16")
    fresh.encoder.set_latent(net.encoder.latent.clone())
    with torch.no_grad():
        assert torch.equal(b, r(fresh, rays).fine.rgb)
        assert torch.equal(b, go())                                        # and back to the first network
    saved = net.mlp_fine.lin_out.bias.detach().clone()
    with torch.no_grad():
        net.mlp_fine.lin_out.bias.add_(0.25)                               # in-place update bumps the version
    c = go()
    assert not torch.equal(b, c)
    net.mlp_fine.lin_out.bias.data.copy_(saved)                            # behind autograd's back: needs invalidate()
    net.mlp_fine.invalidate()
    assert torch.equal(b, go())
