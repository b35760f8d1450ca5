"""View pooling of ResnetFC on the GPU (`-m gpu`), every path through the C-ABI library:

* the single-view network that never pools (combine_layer >= n_blocks, the shape of conf/default.conf: 3 blocks, lin_z before
  every block) with one source view;
* combine_type "max" (the reference's other pooling mode, util.py:489-499) with NS = 2, 3, 5 source views.

Against the CPU oracle, whose max pooling is tests/pooling_oracle.py.  Tolerances as elsewhere: fp32 SIMT arithmetic 1e-4 on the
field (summation order only), bf16 tensor-core operands 1e-2, the training step fp32 1e-3 / TF32 2e-2 of each gradient's
scale.  Single field calls with a random output gradient over ~100-300 points are held in NORM (fp32 1e-3, TF32 5e-2, tcgen05
3e-2 against the bf16-operand emulation) with a loose bound on the worst element: gradients of a piecewise-linear network are
discontinuous, and a pre-activation -- or, with max pooling, the gap between two views -- within the forward error of zero takes
the other branch and changes one gradient term by O(1); with a few hundred rows nothing averages that out
(tests/test_gpu_train.py).  Max pooling passes the rounding of one view through where the mean averages NS of them, so its bf16
forward bounds are 1.5x those of the mean (measured 1.1e-2 on sigma at NS = 5, relative to 1 + |sigma|).
"""
import copy

import numpy as np
import pytest
import torch

import helpers as H
import pixel_nerf_yolo_b200.synth as synth
import pooling_oracle as PO
from oracle import pixelnerf_oracle as O

pytestmark = pytest.mark.gpu

# kind -> (mlp conf, synth.mlp_state shape, oracle field keywords)
KINDS = {
    "single": (dict(n_blocks=3), dict(n_blocks=3, combine_layer=1000), dict(n_blocks=3, combine_layer=1000)),
    "max": (dict(n_blocks=5, combine_layer=3, combine_type="max"), dict(n_blocks=5, combine_layer=3), dict(n_blocks=5, combine_layer=3)),
}
CUSTOM_ENCODER = {"backbone": "custom", "pretrained": False, "num_layers": 4, "index_padding": "zeros"}


@pytest.fixture(scope="module")
def lib():
    from pixel_nerf_yolo_b200 import _lib
    assert torch.cuda.is_available()
    _lib.require_device(torch.device("cuda", 0))
    return _lib.load()


def _model_conf(kind, C=512):
    conf = copy.deepcopy(H.MODEL_CONF)
    for k in ("mlp_coarse", "mlp_fine"):
        conf[k].pop("combine_layer")
        conf[k].pop("combine_type")
        conf[k].update(KINDS[kind][0])
    if C != 512:
        conf["encoder"] = dict(CUSTOM_ENCODER)
    return conf


def _state(kind, seed, C=512):
    return synth.mlp_state(seed, d_latent=C, **KINDS[kind][1])


def _net(kind, scene, precision="bf16", train=False):
    """helpers.build_net for the two pooling settings (same synthetic weights recipe, seeds 1 / 2)."""
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.model import make_model
    C = scene["latent"].shape[1]
    net = make_model(ConfigTree.from_dict(_model_conf(kind, C))).eval()
    net.mlp_coarse.load_state_dict(_state(kind, 1, C))
    net.mlp_fine.load_state_dict(_state(kind, 2, C))
    net = net.cuda()
    poses = scene["poses"]
    net.num_objs, net.num_views_per_obj = poses.shape[0], poses.shape[1]
    net.encoder.set_latent(scene["latent"].cuda())
    net.set_cameras(poses.reshape(-1, 4, 4).cuda(), scene["focal"].cuda(), scene["image_wh"])
    net.precision = precision
    if train:
        net.train()
    else:
        net.requires_grad_(False)
    return net


def _oracle(kind, record=None):
    return PO.combine_type("max" if kind == "max" else "average", record)


def _points(P, seed, num_objs=1):
    g = torch.Generator().manual_seed(seed)
    xyz = (torch.rand(num_objs, P, 3, generator=g) - 0.5) * 0.9
    dirs = torch.nn.functional.normalize(torch.randn(num_objs, P, 3, generator=g), dim=-1)
    return xyz, dirs


def _renderer(**kw):
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.render import NeRFRenderer
    conf = dict(H.RENDER_CONF)
    conf.update(kw)
    return NeRFRenderer.from_conf(ConfigTree.from_dict(conf)).eval().cuda()


def _noise_obj(noise):
    return O.RenderNoise(noise["coarse"], noise["fine_u"], noise["fine_jitter"], noise["depth"])


CASES = [("single", 1), ("max", 2), ("max", 3), ("max", 5)]


# ------------------------------------------------------------------------------------------------ field
@pytest.mark.parametrize("kind,num_views", CASES)
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("bf16", 1e-2)])
def test_field_matches_oracle(lib, kind, num_views, precision, tol):
    tol_sig = 1.5 * tol if (kind == "max" and precision == "bf16") else tol
    scene = H.make_scene_dict(num_views=num_views)
    net = _net(kind, scene, precision)
    xyz, dirs = _points(257, num_views)
    with torch.no_grad():
        out = net(xyz.cuda(), coarse=True, viewdirs=dirs.cuda()).cpu()
    with _oracle(kind):
        ref = O.field_forward(H.oracle_scene(scene), _state(kind, 1), xyz, dirs, **KINDS[kind][2])
    err_rgb = (out[..., :3] - ref[..., :3]).abs().max().item()
    err_sig = ((out[..., 3] - ref[..., 3]).abs() / (1 + ref[..., 3].abs())).max().item()
    assert err_rgb < tol and err_sig < tol_sig, (err_rgb, err_sig)
    assert ref[..., 3].max() > 0.5 and ref[..., :3].std() > 0.01          # the comparison is not vacuous
    if kind == "max":                                                       # and max pooling is not the mean in disguise
        with _oracle("average"):
            avg = O.field_forward(H.oracle_scene(scene), _state(kind, 1), xyz, dirs, **KINDS[kind][2])
        assert (avg - ref).abs().max() > 20 * tol


@pytest.mark.parametrize("kind,ns", [("single", 1), ("max", 3)])
def test_resnetfc_operator(lib, kind, ns):
    """ResnetFC.forward stand-alone (fp32 SIMT kernels) vs the oracle's ResnetFC."""
    net = _net(kind, H.make_scene_dict(num_views=ns))
    rows = 2 * ns * 5
    g = torch.Generator().manual_seed(ns)
    zx = torch.cat((torch.randn(rows, 512, generator=g) * 0.5, torch.randn(rows, 42, generator=g)), dim=-1)
    out = net.mlp_coarse(zx.cuda(), combine_inner_dims=(ns, 5)).cpu()
    ref = PO.resnetfc_forward(_state(kind, 1), zx, 512, KINDS[kind][2]["n_blocks"], KINDS[kind][2]["combine_layer"], (ns, 5),
                              combine_type=net.mlp_coarse.combine_type)
    np.testing.assert_allclose(out.numpy(), ref.numpy(), atol=5e-5, rtol=1e-4)


# ------------------------------------------------------------------------------------------------ render
@pytest.mark.parametrize("kind,num_views", [("single", 1), ("max", 3)])
def test_render_matches_oracle_and_staged_path(lib, kind, num_views):
    """The single-call render (pnr_render_forward, four launches) equals the stage-by-stage path bit for bit, and both are within
    the bf16 tolerance of the oracle."""
    scene = H.make_scene_dict(num_views=num_views)
    net = _net(kind, scene)
    B = 300
    rays = H.rays_subset(1, B, seed=2)
    noise = H.make_noise(B, seed=6)
    r = _renderer()
    r.noise_override = {k: v.cuda() for k, v in noise.items()}
    assert net.fused_render_ready()
    with torch.no_grad():
        a = r(net, rays.cuda(), want_weights=True)
        assert r.last_launches == 4
        net.fused_render_ready = lambda: False
        b = r(net, rays.cuda(), want_weights=True)
        assert r.last_launches == 6
    for lvl in ("coarse", "fine"):
        for k in ("rgb", "depth", "weights"):
            assert torch.equal(a[lvl][k], b[lvl][k]), (lvl, k)
    with _oracle(kind):
        ref = O.render(H.oracle_scene(scene), _state(kind, 1), _state(kind, 2), rays, _noise_obj(noise), **KINDS[kind][2])
    for lvl in ("coarse", "fine"):
        e_rgb = (a[lvl].rgb.cpu() - ref[lvl]["rgb"]).abs().max().item()
        e_d = (a[lvl].depth.cpu() - ref[lvl]["depth"]).abs().max().item()
        assert e_rgb < 1e-2 and e_d < 1e-2, (lvl, e_rgb, e_d)
    assert 0.2 < ref["fine"]["weights"].sum(-1).mean() < 0.999


@pytest.mark.parametrize("project", [True, False])
def test_render_max_projected_wide_latent(lib, project):
    """Max pooling with 1792-channel (YOLO backbone) maps: the lin_z pre-projections gathered (PNR_SCENE_PROJECTED) and the wide
    lin_z streamed through the kernel, through pnr_render_forward."""
    C = 1792
    scene = H.make_scene_dict(num_views=3, feat=16, C=C)
    net = _net("max", scene)
    net.project_wide_latent = project
    B = 128
    rays = H.rays_subset(1, B, seed=3)
    noise = H.make_noise(B, seed=7)
    r = _renderer()
    r.noise_override = {k: v.cuda() for k, v in noise.items()}
    with torch.no_grad():
        res = r(net, rays.cuda())
    assert r.last_launches == 4
    with _oracle("max"):
        ref = O.render(H.oracle_scene(scene), _state("max", 1, C), _state("max", 2, C), rays, _noise_obj(noise))
    for lvl in ("coarse", "fine"):
        e_rgb = (res[lvl].rgb.cpu() - ref[lvl]["rgb"]).abs().max().item()
        e_d = (res[lvl].depth.cpu() - ref[lvl]["depth"]).abs().max().item()
        assert e_rgb < 1e-2 and e_d < 1e-2, (project, lvl, e_rgb, e_d)


# ------------------------------------------------------------------------------------------------ training
def _close(got, ref, what, rtol):
    got, ref = got.detach().cpu().double(), ref.detach().cpu().double()
    assert got.shape == ref.shape, what
    err, scale = (got - ref).abs().max().item(), ref.abs().max().item()
    assert err <= rtol * scale + 1e-12, f"{what}: max err {err:.3e}, scale {scale:.3e}"


def _norm_close(got, ref, what, rtol, rmax):
    got, ref = got.detach().cpu().double(), ref.detach().cpu().double()
    rel = ((got - ref).norm() / ref.norm().clamp_min(1e-30)).item()
    worst = ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()
    assert rel <= rtol and worst <= rmax, f"{what}: rel-norm err {rel:.3e} (<= {rtol}), worst element {worst:.3e} (<= {rmax})"


def _oracle_field_grads(kind, scene, xyz, dirs, gout, emulate_bf16=False, record=None):
    sc = H.oracle_scene(scene)
    sc.latent = sc.latent.clone().requires_grad_(True)
    C = scene["latent"].shape[1]
    mc = {k: v.clone().requires_grad_(True) for k, v in _state(kind, 1, C).items()}
    xo = xyz.clone().requires_grad_(True)
    with _oracle(kind, record):
        ref = O.field_forward(sc, mc, xo, dirs, emulate_bf16=emulate_bf16, **KINDS[kind][2])
    (ref * gout).sum().backward()
    return ref.detach(), {k: v.grad for k, v in mc.items()}, sc.latent.grad, xo.grad


def _untied_points(kind, scene, P, seed, gap=1e-4):
    """Query points whose views are nowhere closer than `gap` at the pooling step (for every feature): the fp32 paths agree with
    the oracle to ~1e-6 there, so both pick the same maximal view and the gradients are comparable element by element."""
    xyz, dirs = _points(P, seed)
    if kind != "max":
        return xyz, dirs
    rec = {}
    with torch.no_grad(), _oracle(kind, rec):
        O.field_forward(H.oracle_scene(scene), _state(kind, 1), xyz, dirs, **KINDS[kind][2])
    top2 = rec["x_views"].topk(2, dim=1).values                       # (1, 2, P, H)
    keep = ((top2[:, 0] - top2[:, 1]).amin(-1) > gap)[0]
    assert keep.float().mean() > 0.5, keep.float().mean()
    return xyz[:, keep].contiguous(), dirs[:, keep].contiguous()


@pytest.mark.parametrize("kind,num_views", CASES)
@pytest.mark.parametrize("train_precision,rtol", [("fp32", 1e-3), ("tf32", 5e-2)])
def test_field_backward_matches_autograd(lib, kind, num_views, train_precision, rtol):
    """PixelNeRFNet.forward(xyz, viewdirs) in training mode: outputs and the gradients of every MLP parameter, of the encoder output
    and of the query points vs autograd over the oracle (max pooling: the gradient goes to the first maximal view)."""
    scene = H.make_scene_dict(num_views=num_views, feat=16)
    xyz, dirs = _untied_points(kind, scene, 120, 10 + num_views)
    gout = torch.randn(*xyz.shape[:2], 4, generator=torch.Generator().manual_seed(num_views))
    ref, g_ref, lat_ref, x_ref = _oracle_field_grads(kind, scene, xyz, dirs, gout)
    net = _net(kind, scene, train=True)
    net.train_precision = train_precision
    lat = scene["latent"].cuda().clone().requires_grad_(True)
    net.encoder.set_latent(lat)
    xc = xyz.cuda().requires_grad_(True)
    out = net(xc, coarse=True, viewdirs=dirs.cuda())
    np.testing.assert_allclose(out.detach().cpu().numpy(), ref.numpy(), atol=1e-4 if train_precision == "fp32" else 3e-3, rtol=0)
    (out * gout.cuda()).sum().backward()
    rmax = 3e-2 if train_precision == "fp32" else 2e-1
    for name, p in net.mlp_coarse.named_parameters():
        _norm_close(p.grad, g_ref[name], f"{train_precision} d {name}", rtol, rmax)
    _norm_close(lat.grad, lat_ref, f"{train_precision} d latent", rtol, rmax)
    # d xyz is one 3-vector per point (~100 rows in all), so a single flip weighs more in its norm: 3x, as test_gpu_train.py's
    # bf16 field test loosens it
    _norm_close(xc.grad, x_ref, f"{train_precision} d xyz", 3 * rtol, rmax)


@pytest.mark.parametrize("kind,num_views", CASES)
def test_field_backward_bf16_matches_autograd(lib, kind, num_views):
    """The tcgen05 training path (bf16 tape + the winning view of every (point, feature) for max pooling): outputs against the fp32
    reference and the bf16-operand emulation, gradients in norm against the emulation's autograd."""
    scene = H.make_scene_dict(num_views=num_views, feat=16)
    xyz, dirs = _points(300, 20 + num_views)
    gout = torch.randn(1, 300, 4, generator=torch.Generator().manual_seed(num_views))
    ref32, _, _, _ = _oracle_field_grads(kind, scene, xyz, dirs, gout)
    ref16, g16, lat16, x16 = _oracle_field_grads(kind, scene, xyz, dirs, gout, emulate_bf16=True)
    net = _net(kind, scene, train=True)
    net.train_precision = "bf16"
    lat = scene["latent"].cuda().clone().requires_grad_(True)
    net.encoder.set_latent(lat)
    xc = xyz.cuda().requires_grad_(True)
    out = net(xc, coarse=True, viewdirs=dirs.cuda())
    o = out.detach().cpu()
    np.testing.assert_allclose(o.numpy()[..., :3], ref32.numpy()[..., :3], atol=1e-2, rtol=0)
    np.testing.assert_allclose(o.numpy()[..., 3], ref32.numpy()[..., 3], atol=1e-2, rtol=1e-2)
    same = 3e-3 if kind == "max" else 2e-3          # same arithmetic: summation order only
    np.testing.assert_allclose(o.numpy(), ref16.numpy(), atol=same, rtol=same)
    (out * gout.cuda()).sum().backward()
    for name, p in net.mlp_coarse.named_parameters():
        _norm_close(p.grad, g16[name], f"bf16 d {name}", 3e-2, 1.5e-1)
    _norm_close(lat.grad, lat16, "bf16 d latent", 3e-2, 1.5e-1)
    _norm_close(xc.grad, x16, "bf16 d xyz", 5e-2, 2e-1)


@pytest.mark.parametrize("train_precision,rtol", [("fp32", 1e-3), ("tf32", 2e-2), ("bf16", 2e-2)])
def test_train_step_single_view_matches_oracle(lib, train_precision, rtol):
    """The full training step (NeRFRenderer.forward + MSE on coarse and fine + backward) of the single-view network against
    autograd over the oracle, on all three arithmetics of the training path."""
    num_objs, nrays = 2, 48
    scene = H.make_scene_dict(num_objs=num_objs, num_views=1, feat=16)
    rays = H.rays_subset(num_objs, nrays, seed=3)
    noise = H.make_noise(num_objs * nrays, seed=4)
    gt = torch.rand(num_objs, nrays, 3, generator=torch.Generator().manual_seed(5))
    # oracle under autograd
    sc = H.oracle_scene(scene)
    sc.latent = sc.latent.clone().requires_grad_(True)
    mc = {k: v.clone().requires_grad_(True) for k, v in _state("single", 1).items()}
    mf = {k: v.clone().requires_grad_(True) for k, v in _state("single", 2).items()}
    res_o = O.render(sc, mc, mf, rays, _noise_obj(noise), grad=True, **KINDS["single"][2])
    mse = torch.nn.functional.mse_loss
    loss_o = mse(res_o["coarse"]["rgb"], gt) + mse(res_o["fine"]["rgb"], gt)
    loss_o.backward()
    # CUDA
    net = _net("single", scene, train=True)
    net.train_precision = train_precision
    lat = scene["latent"].cuda().clone().requires_grad_(True)
    net.encoder.set_latent(lat)
    r = _renderer().train()
    r.noise_override = {k: v.cuda() for k, v in noise.items()}
    res = r(net, rays.cuda())
    loss = mse(res.coarse.rgb, gt.cuda()) + mse(res.fine.rgb, gt.cuda())
    loss.backward()
    assert abs(loss.item() - loss_o.item()) <= (1e-4 if train_precision == "fp32" else 1e-2) * abs(loss_o.item())
    for lvl, mlp, ref in (("coarse", net.mlp_coarse, mc), ("fine", net.mlp_fine, mf)):
        for name, p in mlp.named_parameters():
            what = f"{train_precision} {lvl} d {name}"
            if train_precision == "bf16":   # as against the reference's goldens (test_oracle_grads.check_against_golden)
                got, want = p.grad.detach().cpu().double(), ref[name].grad.double()
                rms = want.norm().item() / want.numel() ** 0.5
                assert (got - want).abs().max().item() <= rtol * 30 * rms + 1e-12, what
                assert abs(got.norm().item() - want.norm().item()) <= rtol * want.norm().item() + 1e-12, what + " norm"
            elif train_precision == "fp32":   # the fine network's gradients are small and carried by few samples: one ReLU flip
                _norm_close(p.grad, ref[name].grad, what, rtol, 1e-2)   # showed as 2.7e-3 of the max of one tensor
            else:
                _close(p.grad, ref[name].grad, what, rtol)
    if train_precision == "bf16":   # a sparse scatter: bf16 ReLU flips do not average out element by element (test_gpu_train.py)
        a, b = lat.grad.detach().cpu().double(), sc.latent.grad.double()
        assert (a - b).norm() <= 5e-2 * b.norm(), ((a - b).norm() / b.norm()).item()
    else:
        _close(lat.grad, sc.latent.grad, f"{train_precision} d latent", rtol)


# ------------------------------------------------------------------------------------------------ refusals
def test_single_view_network_with_several_views_raises(lib):
    """No pooling is only defined for one source view: the Python API raises NotImplementedError before any launch, and every
    C entry point returns PNR_ERR_UNSUPPORTED on its own."""
    from pixel_nerf_yolo_b200 import _lib
    scene = H.make_scene_dict(num_views=3, feat=16)
    net = _net("single", scene)
    xyz, dirs = _points(64, 1)
    with torch.no_grad(), pytest.raises(NotImplementedError, match="one view"):
        net(xyz.cuda(), coarse=True, viewdirs=dirs.cuda())
    with torch.no_grad(), pytest.raises(NotImplementedError, match="one view"):
        _renderer()(net, H.rays_subset(1, 16).cuda())
    # C level, with the Python check bypassed
    net._check_views = lambda: None
    mlp = net.mlp_coarse
    pts = _lib.points_xyz(xyz.cuda(), dirs.cuda())
    keep = (xyz, dirs)
    out = torch.empty(1, 64, 4, device="cuda")
    st = _lib.stream_ptr(torch.device("cuda", 0))
    sc16, _k16 = net._scene(fp32_maps=False)
    ws = torch.empty(lib.pnr_field_workspace_bytes(sc16, pts, _lib.PREC_BF16), dtype=torch.uint8, device="cuda")
    assert lib.pnr_field_forward(sc16, pts, mlp.c_params(), mlp.packed().data_ptr(), out.data_ptr(), ws.data_ptr(), ws.numel(),
                                 _lib.PREC_BF16, 6, 1.5, st) == -3
    assert b"one source view" in lib.pnr_last_error()
    sc32, _k32 = net._scene(fp32_maps=True)
    ws = torch.empty(lib.pnr_field_workspace_bytes(sc32, pts, _lib.PREC_FP32), dtype=torch.uint8, device="cuda")
    assert lib.pnr_field_forward(sc32, pts, mlp.c_params(), None, out.data_ptr(), ws.data_ptr(), ws.numel(), _lib.PREC_FP32, 6, 1.5,
                                 st) == -3
    tape = torch.empty(lib.pnr_field_tape_bytes(sc32, pts, mlp.c_params()), dtype=torch.uint8, device="cuda")
    assert lib.pnr_field_forward_train(sc32, pts, mlp.c_params(), out.data_ptr(), tape.data_ptr(), tape.numel(), 6, 1.5, st) == -3
    del keep
