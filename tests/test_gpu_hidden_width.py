"""ResnetFC hidden widths other than 512 on every path (`-m gpu`), through the public API.

The tcgen05 field kernel runs a network zero-padded to Hp = 256 features (one 256-feature tile, ``MT = 1``) for d_hidden <= 256
and to Hp = 512 (``MT = 2``) above; the fp32 check path, the stand-alone ResnetFC and the training path run the width as it is.
Each field case is held to the bounds of tests/test_gpu_field_coverage.py: the fp32 path at 1e-4 and the tcgen05 path at 1e-2
against the fp32 oracle, and the tcgen05 path at the tight RMS bound against ``bf16_field_reference`` (whose teeth at these
widths tests/test_oracle_hidden_width.py pins).  A network narrower than its latent gathers lin_z pre-projections by default
(``PixelNeRFNet.projects_latent``: d_latent > d_hidden), so at d_hidden <= 448 the 512-channel maps run the projected path
unless ``project_wide_latent = False``.

Measured on one B200 (1000 W power limit): worst RMS error against the bf16 reference over all cases of a width, rgb / sigma,
average pooling 5.9e-5 / 9.3e-5 (64), 7.1e-5 / 1.0e-4 (128), 8.5e-5 / 1.5e-4 (192), 1.2e-4 / 2.3e-4 (256, the (8, 8) network),
9.9e-5 / 1.5e-4 (320), 1.2e-4 / 2.1e-4 (448); max pooling (NS 8) 1.4e-4 / 1.8e-4 (64) up to 3.2e-4 / 4.9e-4 (448).  TIGHT is
6e-4 (1.2e-3 with max pooling).  Whole file: about 35 s.
"""
import copy
import math

import numpy as np
import pytest
import torch

import bf16_field_reference as BR
import helpers as H
import pixel_nerf_yolo_b200.synth as synth
import pooling_oracle as PO
from oracle import pixelnerf_oracle as O

pytestmark = pytest.mark.gpu

LOOSE = 1e-2
FP32 = 1e-4
WIDTHS = (64, 128, 192, 256, 320, 448)
BUILT_NS = (1, 2, 3, 4, 5, 6, 8)
POOLING = [(ns, "average") for ns in BUILT_NS] + [(ns, "max") for ns in BUILT_NS if ns > 1]


@pytest.fixture(scope="module")
def lib():
    from pixel_nerf_yolo_b200 import _lib
    assert torch.cuda.is_available()
    _lib.require_device(torch.device("cuda", 0))
    return _lib.load()


def _points(P, seed, num_objs=1, extent=0.9):
    g = torch.Generator().manual_seed(seed)
    xyz = (torch.rand(num_objs, P, 3, generator=g) - 0.5) * extent
    dirs = torch.nn.functional.normalize(torch.randn(num_objs, P, 3, generator=g), dim=-1)
    return xyz, dirs


def _model_conf(d_hidden, n_blocks=5, combine_layer=3, combine_type="average"):
    conf = copy.deepcopy(H.MODEL_CONF)
    for k in ("mlp_coarse", "mlp_fine"):
        conf[k].update(d_hidden=d_hidden, n_blocks=n_blocks, combine_layer=combine_layer, combine_type=combine_type)
    return conf


class Net:
    """One PixelNeRFNet of hidden width d_hidden (the coarse network is queried) and the matching oracle inputs."""

    def __init__(self, scene, d_hidden, n_blocks=5, combine_layer=3, combine_type="average", anchors=None, precision="bf16",
                 train=False, project=None):
        from pixel_nerf_yolo_b200.conf import ConfigTree
        from pixel_nerf_yolo_b200.model import make_model
        from pixel_nerf_yolo_b200.model.model_util import make_mlp
        C = scene["latent"].shape[1]
        self.yolo = anchors is not None
        d_out = 7 * anchors if self.yolo else 4
        conf = _model_conf(d_hidden, n_blocks, combine_layer, combine_type)
        if self.yolo:
            conf["mlp_coarse"].update({"d_out": 7, "num_scales": 1, "num_anchors_per_scale": anchors, "yolo": True})
            conf["mlp_fine"] = {"type": "empty"}
        conf = ConfigTree.from_dict(conf)
        net = make_model(conf).eval()
        if C != net.d_latent:                # the maps come from set_latent: size the networks for them
            net.mlp_coarse = make_mlp(conf["mlp_coarse"], net.d_in, C)
            net.mlp_fine = None if self.yolo else make_mlp(conf["mlp_fine"], net.d_in, C)
            net.d_latent = net.latent_size = C
        assert net.mlp_coarse.d_hidden == d_hidden
        shape = dict(d_latent=C, d_hidden=d_hidden, n_blocks=n_blocks, combine_layer=combine_layer)
        self.state = synth.mlp_state(1, d_out=d_out, **shape)
        net.mlp_coarse.load_state_dict(self.state)
        if net.mlp_fine is not None:
            net.mlp_fine.load_state_dict(synth.mlp_state(2, **shape))
        net = net.cuda()
        poses = scene["poses"]
        sb, ns = poses.shape[:2]
        cams = poses.reshape(-1, 4, 4)
        if self.yolo:                        # YOLO mode takes world -> camera poses as given
            cams = torch.linalg.inv(cams)
        net.num_objs, net.num_views_per_obj = sb, ns
        net.encoder.set_latent(scene["latent"].cuda())
        net.set_cameras(cams.cuda(), scene["focal"].cuda(), scene["image_wh"])
        net.precision = precision
        net.project_wide_latent = project
        if train:
            net.train()
        else:
            net.requires_grad_(False)
        self.net, self.scene, self.d_hidden = net, scene, d_hidden
        self.sc = O.encode_cameras(scene["latent"], cams.reshape(sb, ns, 4, 4), scene["focal"], scene["image_wh"], yolo=self.yolo)
        self.kw = dict(n_blocks=n_blocks, combine_layer=combine_layer)
        self.combine_type = combine_type
        self.projected = net.projects_latent()

    def __call__(self, xyz, dirs):
        with torch.no_grad():
            return self.net(xyz.cuda(), coarse=True, viewdirs=dirs.cuda()).cpu()

    def oracle(self, xyz, dirs, combine_type=None):
        with PO.combine_type(combine_type or self.combine_type):
            return O.field_forward(self.sc, self.state, xyz, dirs, yolo=self.yolo, **self.kw)

    def bf16_ref(self, xyz, dirs):
        return BR.field_forward_bf16(self.sc, self.state, xyz, dirs, combine_type=self.combine_type, yolo=self.yolo,
                                     projected=self.projected, **self.kw)


def _errors(out, ref, yolo=False, rms=False):
    if yolo:                                 # raw head values are unbounded: relative to their scale (tests/test_gpu_yolo.py)
        d = (out - ref).double() / ref.abs().max().clamp_min(1.0).item()
        return (d.pow(2).mean().sqrt() if rms else d.abs().max()).item(), 0.0
    return BR.rms_errors(out, ref) if rms else BR.errors(out, ref)


def _check(case, m, out, xyz, dirs, ref32=None, ref16=None):
    """Worst element against the fp32 oracle (1e-2), RMS against the bf16 reference (tight bound).  Returns the oracle."""
    ref32 = m.oracle(xyz, dirs) if ref32 is None else ref32
    ref16 = m.bf16_ref(xyz, dirs) if ref16 is None else ref16
    loose = _errors(out, ref32, m.yolo)
    tight = _errors(out, ref16, m.yolo, rms=True)
    print(f"\nHIDDEN d_hidden={m.d_hidden} {case}: bf16 reference RMS rgb {tight[0]:.2e} sigma {tight[1]:.2e} | fp32 oracle "
          f"worst rgb {loose[0]:.2e} sigma {loose[1]:.2e}")
    sig_loose = 1.5 * LOOSE if m.combine_type == "max" else LOOSE
    assert loose[0] < LOOSE and loose[1] < sig_loose, (case, "fp32 oracle", loose)
    bound = BR.tight_bound(m.combine_type)
    assert tight[0] < bound and tight[1] < bound, (case, "bf16 reference RMS", tight)
    return ref32


# ------------------------------------------------------------------------------------------------ field: widths x views x pooling
@pytest.mark.parametrize("sb", [1, 3])
@pytest.mark.parametrize("ns,combine_type", [(1, "average"), (3, "average"), (8, "average"), (3, "max"), (8, "max")])
@pytest.mark.parametrize("d_hidden", WIDTHS)
def test_widths(lib, d_hidden, ns, combine_type, sb):
    """tcgen05 against the oracle and the bf16 reference, then the fp32 check path of the same network at 1e-4.  SB = 1 gathers
    the lin_z pre-projections (the default below 512), SB = 3 streams the 512-channel latent."""
    m = Net(H.make_scene_dict(num_objs=sb, num_views=ns), d_hidden, combine_type=combine_type, project=None if sb == 1 else False)
    xyz, dirs = _points(300 // sb, 100 + ns + d_hidden, sb)
    ref = _check(f"NS={ns} {combine_type} SB={sb} projected={m.projected}", m, m(xyz, dirs), xyz, dirs)
    assert ref[..., 3].max() > 0.5 and ref[..., :3].std() > 0.01          # the comparison is not vacuous
    m.net.precision = "fp32"
    np.testing.assert_allclose(m(xyz, dirs).numpy(), ref.numpy(), atol=FP32, rtol=FP32)


# ------------------------------------------------------------------------------------------------ MT = 1: tiles and super groups
def _tile(ns):
    pp = 64 // ns
    return pp, 64 // pp


@pytest.mark.parametrize("ns", BUILT_NS)
def test_one_tile_kernel_tile_and_super_group_edges(lib, ns):
    """Partial tiles, a partial super group, an odd number of tiles, one point: d_hidden = 128 (MT = 1), streamed latent."""
    pp, g = _tile(ns)
    sizes = sorted({1, pp - 1, pp, pp + 1, 2 * g * pp - 1, 2 * g * pp, 2 * g * pp + 1} - {0})
    m = Net(H.make_scene_dict(num_objs=3, num_views=ns), 128, project=False)
    xyz, dirs = _points(sizes[-1], 200 + ns, 3)
    ref32, ref16 = m.oracle(xyz, dirs), m.bf16_ref(xyz, dirs)
    outs = []
    for P in sizes:
        out = m(xyz[:, :P].contiguous(), dirs[:, :P].contiguous())
        assert out.shape == (3, P, 4)
        loose = _errors(out, ref32[:, :P])
        assert loose[0] < LOOSE and loose[1] < LOOSE, (P, loose)
        outs.append((out, ref32[:, :P], ref16[:, :P]))
    cat = lambda i: torch.cat([o[i].reshape(-1, 4) for o in outs])
    _check(f"edges NS={ns} P={sizes}", m, cat(0), None, None, cat(1), cat(2))


@pytest.mark.parametrize("ns,combine_type", POOLING)
def test_one_tile_kernel_several_super_groups_per_pair(lib, ns, combine_type):
    """At least three super groups per CTA pair at d_hidden = 128 (MT = 1, projected maps): the big launch equals launches of
    under one wave bit for bit."""
    pp, g = _tile(ns)
    n_pairs = torch.cuda.get_device_properties(0).multi_processor_count // 2
    per_sg = 2 * g * pp
    sb = 3
    P = math.ceil(3 * n_pairs * per_sg / sb) + 5
    m = Net(H.make_scene_dict(num_objs=sb, num_views=ns), 128, combine_type=combine_type)
    xyz, dirs = _points(P, 300 + ns, sb)
    big = m(xyz, dirs)
    step = n_pairs * per_sg // (2 * sb)
    assert math.ceil(math.ceil(sb * math.ceil(step / pp) / 2) / g) < n_pairs
    for a in range(0, P, step):
        part = m(xyz[:, a:a + step].contiguous(), dirs[:, a:a + step].contiguous())
        assert torch.equal(big[:, a:a + step], part), (a, (big[:, a:a + step] - part).abs().max().item())
    stride = math.ceil(sb * P / 512)
    xs, ds = xyz[:, ::stride].contiguous(), dirs[:, ::stride].contiguous()
    _check(f"super groups NS={ns} {combine_type} P={P}x{sb}", m, big[:, ::stride], xs, ds)


# ------------------------------------------------------------------------------------------------ network shapes, latents, heads
@pytest.mark.parametrize("d_hidden,n_blocks,combine_layer,ns", [(128, 3, 1000, 1), (256, 1, 1, 1), (256, 5, 3, 3), (256, 8, 8, 1)])
def test_network_shapes(lib, d_hidden, n_blocks, combine_layer, ns):
    """(3, 1000): the unpooled single-view network of conf/default.conf."""
    m = Net(H.make_scene_dict(num_views=ns), d_hidden, n_blocks=n_blocks, combine_layer=combine_layer)
    xyz, dirs = _points(200, 400 + n_blocks, 1)
    ref = _check(f"n_blocks={n_blocks} combine_layer={combine_layer} NS={ns}", m, m(xyz, dirs), xyz, dirs)
    assert ref[..., 3].max() > 0.5 and ref[..., :3].std() > 0.01


@pytest.mark.parametrize("C,project", [(64, False), (576, False), (1792, True), (1792, False)])
@pytest.mark.parametrize("combine_type", ["average", "max"])
@pytest.mark.parametrize("d_hidden", [128, 256])
def test_latent_widths(lib, d_hidden, combine_type, C, project):
    """Streamed latents narrower than one 512-channel pass or one pass and a partial one; 1792-channel maps gathered as lin_z
    pre-projections (n_linz x d_hidden channels) or streamed."""
    m = Net(H.make_scene_dict(num_views=3, C=C), d_hidden, combine_type=combine_type, project=project)
    assert m.projected == project
    xyz, dirs = _points(200, 500 + C, 1)
    _check(f"d_latent={C} projected={project} {combine_type}", m, m(xyz, dirs), xyz, dirs)


def test_yolo_head(lib):
    m = Net(H.make_scene_dict(num_views=3), 256, anchors=3)
    xyz, dirs = _points(200, 603, 1, extent=3.2)
    out = m(xyz, dirs)
    assert out.shape == (1, 200, 21)
    _check("YOLO d_out=21", m, out, xyz, dirs)


def test_resnetfc_operator(lib):
    """ResnetFC.forward stand-alone (fp32 SIMT kernels) at widths that are not multiples of the SGEMM's 128-wide tile."""
    for d_hidden in (64, 192, 320, 448):
        m = Net(H.make_scene_dict(num_views=3), d_hidden, combine_type="max")
        rows = 2 * 3 * 5
        g = torch.Generator().manual_seed(d_hidden)
        zx = torch.cat((torch.randn(rows, 512, generator=g) * 0.5, torch.randn(rows, 42, generator=g)), dim=-1)
        out = m.net.mlp_coarse(zx.cuda(), combine_inner_dims=(3, 5)).cpu()
        ref = PO.resnetfc_forward(m.state, zx, 512, 5, 3, (3, 5), combine_type="max")
        np.testing.assert_allclose(out.numpy(), ref.numpy(), atol=5e-5, rtol=1e-4)


# ------------------------------------------------------------------------------------------------ render
def _renderer(**kw):
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.render import NeRFRenderer
    conf = dict(H.RENDER_CONF)
    conf.update(kw)
    return NeRFRenderer.from_conf(ConfigTree.from_dict(conf)).eval().cuda()


def _noise_obj(noise):
    return O.RenderNoise(noise["coarse"], noise["fine_u"], noise["fine_jitter"], noise["depth"])


@pytest.mark.parametrize("d_hidden", [128, 256])
def test_render_single_call_equals_staged_path(lib, d_hidden):
    scene = H.make_scene_dict(num_views=3)
    m = Net(scene, d_hidden)
    net = m.net
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
    for lvl in ("coarse", "fine"):
        for k in ("rgb", "depth", "weights"):
            assert torch.equal(a[lvl][k], b[lvl][k]), (lvl, k)
    fine_state = synth.mlp_state(2, d_hidden=d_hidden)
    ref = O.render(H.oracle_scene(scene), m.state, fine_state, rays, _noise_obj(noise))
    for lvl in ("coarse", "fine"):
        e_rgb = (a[lvl].rgb.cpu() - ref[lvl]["rgb"]).abs().max().item()
        e_d = (a[lvl].depth.cpu() - ref[lvl]["depth"]).abs().max().item()
        assert e_rgb < 1e-2 and e_d < 1e-2, (lvl, e_rgb, e_d)


# ------------------------------------------------------------------------------------------------ training
def _norm_close(got, ref, what, rtol, rmax):
    got, ref = got.detach().cpu().double(), ref.detach().cpu().double()
    rel = ((got - ref).norm() / ref.norm().clamp_min(1e-30)).item()
    worst = ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()
    assert rel <= rtol and worst <= rmax, f"{what}: rel-norm err {rel:.3e} (<= {rtol}), worst element {worst:.3e} (<= {rmax})"


def _oracle_grads(m, xyz, dirs, gout, emulate_bf16=False):
    sc = copy.copy(m.sc)
    sc.latent = sc.latent.clone().requires_grad_(True)
    mc = {k: v.clone().requires_grad_(True) for k, v in m.state.items()}
    xo = xyz.clone().requires_grad_(True)
    with PO.combine_type(m.combine_type):
        ref = O.field_forward(sc, mc, xo, dirs, emulate_bf16=emulate_bf16, **m.kw)
    (ref * gout).sum().backward()
    return ref.detach(), {k: v.grad for k, v in mc.items()}, sc.latent.grad, xo.grad


def _untied(m, xyz, dirs, gap=1e-4):
    """Points whose views are nowhere closer than `gap` at the max-pooling step, so that the fp32 paths pick the oracle's view."""
    if m.combine_type != "max":
        return xyz, dirs
    rec = {}
    with torch.no_grad(), PO.combine_type("max", rec):
        O.field_forward(m.sc, m.state, xyz, dirs, **m.kw)
    top2 = rec["x_views"].topk(2, dim=1).values
    keep = ((top2[:, 0] - top2[:, 1]).amin(-1) > gap)[0]
    assert keep.float().mean() > 0.3, keep.float().mean()
    return xyz[:, keep].contiguous(), dirs[:, keep].contiguous()


@pytest.mark.parametrize("train_precision", ["fp32", "tf32", "bf16"])
@pytest.mark.parametrize("combine_type", ["average", "max"])
@pytest.mark.parametrize("d_hidden", [128, 256])
def test_field_backward(lib, d_hidden, combine_type, train_precision):
    """One field call in training mode and its backward vs autograd over the oracle, with the bounds of
    tests/test_gpu_pooling.py (fp32, TF32) and tests/test_gpu_field_coverage.py (tcgen05)."""
    scene = H.make_scene_dict(num_views=3, feat=16)
    m = Net(scene, d_hidden, combine_type=combine_type, train=True)
    m.net.train_precision = train_precision
    xyz, dirs = _points(300 if train_precision == "bf16" else 160, 1000 + d_hidden, 1)
    if train_precision != "bf16":
        xyz, dirs = _untied(m, xyz, dirs)
    gout = torch.randn(*xyz.shape[:2], 4, generator=torch.Generator().manual_seed(d_hidden))
    ref32, g32, lat32, x32 = _oracle_grads(m, xyz, dirs, gout)
    lat = scene["latent"].cuda().clone().requires_grad_(True)
    m.net.encoder.set_latent(lat)
    xc = xyz.cuda().requires_grad_(True)
    out = m.net(xc, coarse=True, viewdirs=dirs.cuda())
    o = out.detach().cpu()
    (out * gout.cuda()).sum().backward()
    if train_precision == "fp32":
        np.testing.assert_allclose(o.numpy(), ref32.numpy(), atol=1e-4, rtol=0)
        ref_g, ref_lat, ref_x, rtol, rmax, xtol = g32, lat32, x32, 1e-3, 3e-2, 3e-3
    elif train_precision == "tf32":
        np.testing.assert_allclose(o.numpy(), ref32.numpy(), atol=3e-3, rtol=0)
        ref_g, ref_lat, ref_x, rtol, rmax, xtol = g32, lat32, x32, 5e-2, 2e-1, 1.5e-1
    else:
        np.testing.assert_allclose(o.numpy()[..., :3], ref32.numpy()[..., :3], atol=LOOSE, rtol=0)
        np.testing.assert_allclose(o.numpy()[..., 3], ref32.numpy()[..., 3], atol=LOOSE, rtol=LOOSE)
        ref16, ref_g, ref_lat, ref_x = _oracle_grads(m, xyz, dirs, gout, emulate_bf16=True)
        same = 3e-3 if combine_type == "max" else 2e-3
        np.testing.assert_allclose(o.numpy(), ref16.numpy(), atol=same, rtol=same)
        rtol, rmax, xtol = 5e-2, 3e-1, 5e-2
    for name, p in m.net.mlp_coarse.named_parameters():
        _norm_close(p.grad, ref_g[name], f"{train_precision} d {name}", rtol, rmax)
    _norm_close(lat.grad, ref_lat, f"{train_precision} d latent", rtol, rmax)
    _norm_close(xc.grad, ref_x, f"{train_precision} d xyz", xtol, rmax)


def test_train_step_from_conf_without_d_hidden(lib):
    """make_model with mlp confs that leave out d_hidden builds 128-wide networks (the reference's default); one full training
    step on the tcgen05 arithmetic (NeRFRenderer.forward + MSE on coarse and fine + backward) against autograd over the oracle,
    with the bounds of tests/test_gpu_pooling.py."""
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.model import make_model
    conf = copy.deepcopy(H.MODEL_CONF)
    for k in ("mlp_coarse", "mlp_fine"):
        conf[k].pop("d_hidden")
    num_objs, ns, nrays = 2, 3, 48
    scene = H.make_scene_dict(num_objs=num_objs, num_views=ns, feat=16)
    net = make_model(ConfigTree.from_dict(conf))
    assert net.mlp_coarse.d_hidden == 128 and net.mlp_fine.d_hidden == 128
    mc0, mf0 = synth.mlp_state(1, d_hidden=128), synth.mlp_state(2, d_hidden=128)
    net.mlp_coarse.load_state_dict(mc0)
    net.mlp_fine.load_state_dict(mf0)
    net = net.cuda().train()
    net.num_objs, net.num_views_per_obj = num_objs, ns
    net.set_cameras(scene["poses"].reshape(-1, 4, 4).cuda(), scene["focal"].cuda(), scene["image_wh"])
    net.train_precision = "bf16"
    lat = scene["latent"].cuda().clone().requires_grad_(True)
    net.encoder.set_latent(lat)
    rays = H.rays_subset(num_objs, nrays, seed=3)
    noise = H.make_noise(num_objs * nrays, seed=4)
    gt = torch.rand(num_objs, nrays, 3, generator=torch.Generator().manual_seed(5))
    sc = H.oracle_scene(scene)
    sc.latent = sc.latent.clone().requires_grad_(True)
    mc = {k: v.clone().requires_grad_(True) for k, v in mc0.items()}
    mf = {k: v.clone().requires_grad_(True) for k, v in mf0.items()}
    res_o = O.render(sc, mc, mf, rays, _noise_obj(noise), grad=True)
    mse = torch.nn.functional.mse_loss
    loss_o = mse(res_o["coarse"]["rgb"], gt) + mse(res_o["fine"]["rgb"], gt)
    loss_o.backward()
    r = _renderer().train()
    r.noise_override = {k: v.cuda() for k, v in noise.items()}
    res = r(net, rays.cuda())
    loss = mse(res.coarse.rgb, gt.cuda()) + mse(res.fine.rgb, gt.cuda())
    loss.backward()
    assert abs(loss.item() - loss_o.item()) <= 1e-2 * abs(loss_o.item())
    rtol = 2e-2
    for lvl, mlp, ref in (("coarse", net.mlp_coarse, mc), ("fine", net.mlp_fine, mf)):
        for name, p in mlp.named_parameters():
            got, want = p.grad.detach().cpu().double(), ref[name].grad.double()
            rms = want.norm().item() / want.numel() ** 0.5
            assert (got - want).abs().max().item() <= rtol * 30 * rms + 1e-12, (lvl, name)
            assert abs(got.norm().item() - want.norm().item()) <= rtol * want.norm().item() + 1e-12, (lvl, name, "norm")
    a, b = lat.grad.detach().cpu().double(), sc.latent.grad.double()
    assert (a - b).norm() <= 5e-2 * b.norm(), ((a - b).norm() / b.norm()).item()


# ------------------------------------------------------------------------------------------------ refusals
@pytest.mark.parametrize("d_hidden", [100, 576])
def test_unsupported_widths_are_refused(lib, d_hidden):
    """Widths that are not a multiple of 64 in [64, 512]: NotImplementedError naming the width and the supported ones, before any
    launch, on both field paths; the C entry points leave the output unwritten."""
    from pixel_nerf_yolo_b200 import _lib
    m = Net(H.make_scene_dict(num_views=3), d_hidden)
    xyz, dirs = _points(64, 800, 1)
    for precision in ("bf16", "fp32"):
        m.net.precision = precision
        with pytest.raises(NotImplementedError, match=f"d_hidden={d_hidden} .*multiples of 64"):
            m(xyz, dirs)
    mlp = m.net.mlp_coarse
    cp = mlp.c_params()
    assert lib.pnr_mlp_pack_bytes(cp) == 0 and lib.pnr_mlp_pack_projected_bytes(cp) == 0
    with pytest.raises(NotImplementedError, match=f"d_hidden={d_hidden}"):
        mlp.packed()
    assert lib.pnr_last_launch_count() == 0
    pts = _lib.points_xyz(xyz.cuda(), dirs.cuda())
    sc, _keep = m.net._scene(fp32_maps=False)
    out = torch.full((1, 64, 4), float("nan"), device="cuda")
    ws = torch.empty(lib.pnr_field_workspace_bytes(sc, pts, _lib.PREC_BF16), dtype=torch.uint8, device="cuda")
    dummy = torch.empty(1024, dtype=torch.uint8, device="cuda")
    rc = lib.pnr_field_forward(sc, pts, cp, dummy.data_ptr(), out.data_ptr(), ws.data_ptr(), ws.numel(), _lib.PREC_BF16, 6, 1.5,
                               _lib.stream_ptr(torch.device("cuda", 0)))
    assert rc == -3 and f"d_hidden={d_hidden}".encode() in lib.pnr_last_error()
    assert lib.pnr_last_launch_count() == 0
    torch.cuda.synchronize()
    assert out.isnan().all()
