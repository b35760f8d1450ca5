"""PixelNeRFNet's z-feature switches on every path (`-m gpu`): use_viewdirs, use_code_viewdirs, normalize_z, use_xyz, use_code
and code.include_input, through the public API.

"The oracle" below is tests/zfeature_oracle.py: the golden-pinned oracle's PixelNeRFNet.forward with the switched z-feature
(``switched`` runs O.render and bf16_field_reference with it).

Every switch combination whose z-feature fits one K = 64 slab of lin_in (d_in <= 64), at 6 frequencies and at 4 and 9:
* ``pnr_gather_encode``'s z-feature against the oracle's, at 3e-6 plus what a 2-ulp difference of the fp32 coordinate becomes
  through the encoding's frequency f (|d sin(f u) / du| <= f: at 9 frequencies f reaches 384);
* the fp32 field at 1e-4 and the tcgen05 field at 1e-2 against the oracle, and the tcgen05 field at the tight RMS bound of
  tests/test_gpu_field_coverage.py against the switched bf16 reference;
and at 6 frequencies (plus a few layouts at 4 and 9):
* the staged render bit for bit equal to the single-call render, and the render against the oracle at 1e-2;
* one training field call on fp32, TF32 and tcgen05 arithmetic: parameter, feature-map and sample-depth gradients against
  autograd over the oracle, with the bounds of tests/test_gpu_hidden_width.py::test_field_backward (fp32 at 9 frequencies
  3e-3, TF32 7.5e-2 / 3e-1, see test_training_step); the fp32 case drops rays with a ReLU input within 1e-5 of zero.
One YOLO-mode and one max-pooling case show that the bits do not interact with those modes.
"""
import copy

import numpy as np
import pytest
import torch

import bf16_field_reference as BR
import helpers as H
import pixel_nerf_yolo_b200.synth as synth
import pooling_oracle as PO
import zfeature_oracle as ZO
from oracle import pixelnerf_oracle as O
from test_oracle_zfeature import COMBOS, DEFAULT, combo_id, oracle_zfeature, reference_d_in

pytestmark = pytest.mark.gpu

LOOSE = 1e-2
FP32 = 1e-4
FF = 1.5
SHAPE = dict(d_hidden=128, n_blocks=3, combine_layer=2)
CASES = [(sw, nf) for nf in (6, 4, 9) for sw in COMBOS if reference_d_in(sw, nf)[0] <= 64]
CASE_IDS = [f"{combo_id(sw)}-nf{nf}" for sw, nf in CASES]
# a few layouts at 4 and 9 frequencies for the render and the training step: default, PE without its input over -z, and the
# encoded view directions
FEW = [DEFAULT, dict(DEFAULT, use_xyz=False, include_input=False, normalize_z=False),
       dict(DEFAULT, use_xyz=False, use_code_viewdirs=True)]
SLOW = [(sw, 6) for sw in COMBOS if reference_d_in(sw, 6)[0] <= 64] + [(sw, nf) for nf in (4, 9) for sw in FEW
                                                                          if reference_d_in(sw, nf)[0] <= 64]
SLOW_IDS = [f"{combo_id(sw)}-nf{nf}" for sw, nf in SLOW]


@pytest.fixture(scope="module")
def lib():
    from pixel_nerf_yolo_b200 import _lib
    assert torch.cuda.is_available()
    _lib.require_device(torch.device("cuda", 0))
    return _lib.load()


def _points(P, seed, extent=0.9):
    g = torch.Generator().manual_seed(seed)
    xyz = (torch.rand(1, P, 3, generator=g) - 0.5) * extent
    dirs = torch.nn.functional.normalize(torch.randn(1, P, 3, generator=g), dim=-1)
    return xyz, dirs


class Net:
    """A PixelNeRFNet built from a conf with the switches ``sw`` at ``num_freqs`` frequencies on a 64-channel latent, with the
    matching oracle arguments (the coarse network is queried)."""

    def __init__(self, sw, num_freqs, ns=2, combine_type="average", anchors=None, train=False):
        from pixel_nerf_yolo_b200.conf import ConfigTree
        from pixel_nerf_yolo_b200.model import make_model
        from pixel_nerf_yolo_b200.model.model_util import make_mlp
        scene = H.make_scene_dict(num_views=ns, C=64)
        self.yolo = anchors is not None
        d_out = 7 * anchors if self.yolo else 4
        conf = copy.deepcopy(H.MODEL_CONF)
        conf.update({k: v for k, v in sw.items() if k != "include_input"})
        conf["code"] = {"num_freqs": num_freqs, "freq_factor": FF, "include_input": sw["include_input"]}
        for k in ("mlp_coarse", "mlp_fine"):
            conf[k].update(combine_type=combine_type, **SHAPE)
        if self.yolo:
            conf["mlp_coarse"].update({"d_out": 7, "num_scales": 1, "num_anchors_per_scale": anchors, "yolo": True})
            conf["mlp_fine"] = {"type": "empty"}
        conf = ConfigTree.from_dict(conf)
        net = make_model(conf).eval()
        d_in = reference_d_in(sw, num_freqs)[0]
        assert net.d_in == d_in
        net.mlp_coarse = make_mlp(conf["mlp_coarse"], d_in, 64)
        net.mlp_fine = None if self.yolo else make_mlp(conf["mlp_fine"], d_in, 64)
        net.d_latent = net.latent_size = 64
        self.state = synth.mlp_state(1, d_in=d_in, d_latent=64, d_out=d_out, **SHAPE)
        self.fine_state = synth.mlp_state(2, d_in=d_in, d_latent=64, **SHAPE)
        net.mlp_coarse.load_state_dict(self.state)
        if net.mlp_fine is not None:
            net.mlp_fine.load_state_dict(self.fine_state)
        net = net.cuda()
        cams = scene["poses"].reshape(-1, 4, 4)
        if self.yolo:
            cams = torch.linalg.inv(cams)
        net.num_objs, net.num_views_per_obj = 1, ns
        net.encoder.set_latent(scene["latent"].cuda())
        net.set_cameras(cams.cuda(), scene["focal"].cuda(), scene["image_wh"])
        if train:
            net.train()
        else:
            net.requires_grad_(False)
        assert not net.projects_latent()
        self.net, self.scene, self.sw, self.num_freqs, self.combine_type = net, scene, sw, num_freqs, combine_type
        self.sc = O.encode_cameras(scene["latent"], cams.reshape(1, ns, 4, 4), scene["focal"], scene["image_wh"], yolo=self.yolo)
        self.kw = dict(n_blocks=SHAPE["n_blocks"], combine_layer=SHAPE["combine_layer"])
        self.zkw = dict(num_freqs=num_freqs, freq_factor=FF, **sw)           # the z-feature of tests/zfeature_oracle.py

    def dirs(self, dirs):
        """What the caller passes: the reference asserts view directions only when the network uses them."""
        return dirs if self.sw["use_viewdirs"] else None

    def __call__(self, xyz, dirs, precision="bf16"):
        self.net.precision = precision
        d = self.dirs(dirs)
        with torch.no_grad():
            return self.net(xyz.cuda(), coarse=True, viewdirs=None if d is None else d.cuda()).cpu()

    def oracle(self, xyz, dirs):
        with PO.combine_type(self.combine_type):
            return ZO.field_forward(self.sc, self.state, xyz, self.dirs(dirs), yolo=self.yolo, **self.kw, **self.zkw)

    def bf16_ref(self, xyz, dirs):
        with ZO.switched(**self.zkw):
            return BR.field_forward_bf16(self.sc, self.state, xyz, self.dirs(dirs), combine_type=self.combine_type, yolo=self.yolo,
                                         projected=False, **self.kw)


def _errors(out, ref, yolo=False, rms=False):
    if yolo:                                 # raw head values are unbounded: relative to their scale (tests/test_gpu_yolo.py)
        d = (out - ref).double() / ref.abs().max().clamp_min(1.0).item()
        return (d.pow(2).mean().sqrt() if rms else d.abs().max()).item(), 0.0
    return BR.rms_errors(out, ref) if rms else BR.errors(out, ref)


def _check_field(case, m, xyz, dirs):
    """tcgen05: worst element against the oracle (1e-2), RMS against the bf16 reference (tight); fp32 path at 1e-4."""
    out = m(xyz, dirs)
    ref32, ref16 = m.oracle(xyz, dirs), m.bf16_ref(xyz, dirs)
    loose = _errors(out, ref32, m.yolo)
    tight = _errors(out, ref16, m.yolo, rms=True)
    print(f"\nZFEAT {case}: bf16 reference RMS rgb {tight[0]:.2e} sigma {tight[1]:.2e} | oracle worst rgb {loose[0]:.2e} "
          f"sigma {loose[1]:.2e}")
    sig_loose = 1.5 * LOOSE if m.combine_type == "max" else LOOSE
    assert loose[0] < LOOSE and loose[1] < sig_loose, (case, "fp32 oracle", loose)
    bound = BR.tight_bound(m.combine_type)
    assert tight[0] < bound and tight[1] < bound, (case, "bf16 reference RMS", tight)
    if not m.yolo:
        assert ref32[..., :3].std() > 0.01          # the comparison is not vacuous (some z-features leave sigma at 0 here)
    fp32 = m(xyz, dirs, precision="fp32")
    np.testing.assert_allclose(fp32.numpy(), ref32.numpy(), atol=FP32, rtol=FP32)


# ------------------------------------------------------------------------------------------------ gather + encode, field
def _encoder_input_scale(m, xyz, dirs):
    """Per z-feature column: the slope bound f (1 for the raw columns) times 2 ulp of the fp32 input it is computed from."""
    sw, nf = m.sw, m.num_freqs
    NS = m.sc.num_views
    R = m.sc.poses[:, None, :3, :3]
    x_rot = torch.matmul(R, xyz.expand(NS, -1, 3).unsqueeze(-1))[..., 0]
    mag = (x_rot.abs() + (x_rot + m.sc.poses[:, None, :3, 3]).abs()).amax(-1).reshape(-1, 1)    # |coordinates| of the row
    ulp2 = torch.maximum(mag, torch.ones_like(mag)) * 2.0 ** -22
    d_in, code_in = reference_d_in(sw, nf)
    if code_in is None:
        return ulp2.expand(-1, d_in)
    slopes = ([1.0] * code_in if sw["include_input"] else []) + [FF * 2.0 ** k for k in range(nf) for _ in range(2 * code_in)]
    slopes += [1.0] * (d_in - len(slopes))
    return ulp2 * torch.tensor(slopes)


@pytest.mark.parametrize("sw,num_freqs", CASES, ids=CASE_IDS)
def test_gather_encode_zfeature(lib, sw, num_freqs):
    from pixel_nerf_yolo_b200 import _lib
    m = Net(sw, num_freqs)
    xyz, dirs = _points(301, 3)
    d_in = m.net.d_in
    want = oracle_zfeature(m.sc, m.state, xyz, m.dirs(dirs), 64, **m.kw, **m.zkw)
    tol = 3e-6 + _encoder_input_scale(m, xyz, dirs)
    for fp32 in (True, False):
        sc, _keep = m.net._scene(fp32_maps=fp32)
        xd, dd = xyz.cuda(), dirs.cuda()                 # alive until the kernel has run: pts holds raw pointers
        pts = _lib.points_xyz(xd, dd)
        zf = torch.full((2 * 301, d_in), float("nan"), device="cuda")
        _lib.check(lib.pnr_gather_encode(sc, pts, None, zf.data_ptr(), 1, *m.net.code_args(), _lib.stream_ptr(zf.device)),
                   "pnr_gather_encode")
        err = (zf.cpu() - want).abs()
        assert (err <= tol).all(), (err.max().item(), (err / tol).max().item())


@pytest.mark.parametrize("sw,num_freqs", CASES, ids=CASE_IDS)
def test_field(lib, sw, num_freqs):
    m = Net(sw, num_freqs)
    xyz, dirs = _points(240, 100 + num_freqs)
    _check_field(f"{combo_id(sw)} nf={num_freqs}", m, xyz, dirs)


def test_field_yolo_mode(lib):
    sw = dict(DEFAULT, use_viewdirs=False, normalize_z=False, use_xyz=False)
    m = Net(sw, 6, ns=3, anchors=3)
    xyz, dirs = _points(200, 603, extent=3.2)
    out = m(xyz, dirs)
    assert out.shape == (1, 200, 21)
    _check_field("YOLO", m, xyz, dirs)


@pytest.mark.parametrize("ns", [3, 8])
def test_field_max_pooling(lib, ns):
    sw = dict(DEFAULT, use_code_viewdirs=True, use_xyz=False, include_input=False)
    m = Net(sw, 6, ns=ns, combine_type="max")
    xyz, dirs = _points(200, 700 + ns)
    _check_field(f"max NS={ns}", m, xyz, dirs)


# ------------------------------------------------------------------------------------------------ render
def _renderer():
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.render import NeRFRenderer
    return NeRFRenderer.from_conf(ConfigTree.from_dict(dict(H.RENDER_CONF))).eval().cuda()


@pytest.mark.parametrize("sw,num_freqs", SLOW, ids=SLOW_IDS)
def test_render(lib, sw, num_freqs):
    """Single-call render (pnr_render_forward) bit for bit equal to the staged path, and the render against the oracle."""
    m = Net(sw, num_freqs)
    net = m.net
    B = 96
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
    n = O.RenderNoise(noise["coarse"], noise["fine_u"], noise["fine_jitter"], noise["depth"])
    with ZO.switched(**m.zkw):
        ref = O.render(m.sc, m.state, m.fine_state, rays, n, **m.kw)
    for lvl in ("coarse", "fine"):
        e_rgb = (a[lvl].rgb.cpu() - ref[lvl]["rgb"]).abs().max().item()
        e_d = (a[lvl].depth.cpu() - ref[lvl]["depth"]).abs().max().item()
        assert e_rgb < LOOSE and e_d < LOOSE, (lvl, e_rgb, e_d)


# ------------------------------------------------------------------------------------------------ training
def _norm_close(got, ref, what, rtol, rmax):
    got, ref = got.detach().cpu().double(), ref.detach().cpu().double()
    rel = ((got - ref).norm() / ref.norm().clamp_min(1e-30)).item()
    worst = ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()
    assert rel <= rtol and worst <= rmax, f"{what}: rel-norm err {rel:.3e} (<= {rtol}), worst element {worst:.3e} (<= {rmax})"


def _oracle_grads(m, rays, z, gout, emulate_bf16=False):
    """Autograd over the oracle for the field at o + z d: output and gradients of the parameters, the maps and the depths."""
    sc = copy.copy(m.sc)
    sc.latent = sc.latent.clone().requires_grad_(True)
    mc = {k: v.clone().requires_grad_(True) for k, v in m.state.items()}
    zo = z.clone().requires_grad_(True)
    pts, dirs = O.ray_points(rays, zo)
    out = ZO.field_forward(sc, mc, pts.reshape(1, -1, 3), m.dirs(dirs.reshape(1, -1, 3)), emulate_bf16=emulate_bf16, **m.kw,
                           **m.zkw)
    (out * gout).sum().backward()
    return out.detach(), {k: v.grad for k, v in mc.items()}, sc.latent.grad, zo.grad


def _relu_margin(m, rays, z):
    """Per ray: the smallest |ReLU input| of the oracle's forward over the ray's samples and views.  Where that is within the
    fp32 arithmetic's distance of zero, the CUDA path may take the other side of the ReLU and move a parameter gradient by far
    more than its rounding (the counterpart of tests/test_gpu_hidden_width.py::_untied for max pooling)."""
    seen, relu = [], torch.relu

    def spy(x):
        seen.append(x.detach())
        return relu(x)
    pts, dirs = O.ray_points(rays, z)
    n = pts.shape[0] * pts.shape[1]
    torch.relu = spy
    try:
        with torch.no_grad():
            ZO.field_forward(m.sc, m.state, pts.reshape(1, -1, 3), m.dirs(dirs.reshape(1, -1, 3)), **m.kw, **m.zkw)
    finally:
        torch.relu = relu
    margin = torch.full((n,), float("inf"))
    for x in seen:
        margin = torch.minimum(margin, x.abs().reshape(-1, n, x.shape[-1]).amin(dim=(0, 2)))
    return margin.reshape(z.shape).amin(dim=1)


@pytest.mark.parametrize("train_precision", ["fp32", "tf32", "bf16"])
@pytest.mark.parametrize("sw,num_freqs", SLOW, ids=SLOW_IDS)
def test_training_step(lib, sw, num_freqs, train_precision):
    m = Net(sw, num_freqs, train=True)
    m.net.train_precision = train_precision
    B, K = 48, 8
    rays = H.rays_subset(1, B, seed=3)[0]
    g = torch.Generator().manual_seed(num_freqs)
    z, _ = torch.sort(rays[:, 6:7] + (rays[:, 7:8] - rays[:, 6:7]) * torch.rand(B, K, generator=g), dim=-1)
    if train_precision == "fp32":
        keep = _relu_margin(m, rays, z) > 1e-5
        assert keep.sum() >= 8, keep.sum()
        rays, z = rays[keep].contiguous(), z[keep].contiguous()
        B = rays.shape[0]
    gout = torch.randn(1, B * K, 4, generator=g)
    ref32, g32, lat32, z32 = _oracle_grads(m, rays, z, gout)
    lat = m.scene["latent"].cuda().clone().requires_grad_(True)
    m.net.encoder.set_latent(lat)
    zc = z.cuda().requires_grad_(True)
    out = m.net.field_from_rays(rays.cuda(), zc, coarse=True, sb=1).reshape(1, B * K, 4)
    o = out.detach().cpu()
    (out * gout.cuda()).sum().backward()
    if train_precision == "fp32":
        np.testing.assert_allclose(o.numpy(), ref32.numpy(), atol=1e-4, rtol=0)
        # at 9 frequencies the encoding turns a last-bit difference of an fp32 coordinate into f = 384 times as much
        ref_g, ref_lat, ref_z, rtol, rmax, xtol = g32, lat32, z32, (3e-3 if num_freqs == 9 else 1e-3), 3e-2, 3e-3
    elif train_precision == "tf32":
        np.testing.assert_allclose(o.numpy(), ref32.numpy(), atol=3e-3, rtol=0)
        # 7.5e-2 / 3e-1 rather than test_field_backward's 5e-2 / 2e-1: TF32 moves pre-activations by ~1e-3, and in a call of a
        # few hundred rows the ReLU flips that causes average out less (measured on a B200 over these layouts: up to 6.6e-2
        # rel-norm, 2.1e-1 worst element)
        ref_g, ref_lat, ref_z, rtol, rmax, xtol = g32, lat32, z32, 7.5e-2, 3e-1, 1.5e-1
    else:
        np.testing.assert_allclose(o.numpy()[..., :3], ref32.numpy()[..., :3], atol=LOOSE, rtol=0)
        np.testing.assert_allclose(o.numpy()[..., 3], ref32.numpy()[..., 3], atol=LOOSE, rtol=LOOSE)
        ref16, ref_g, ref_lat, ref_z = _oracle_grads(m, rays, z, gout, emulate_bf16=True)
        same = BR.rms_errors(o, ref16)                  # single bf16 rounding flips move single values (bf16_field_reference)
        assert same[0] < BR.TIGHT and same[1] < BR.TIGHT, same
        rtol, rmax, xtol = 5e-2, 3e-1, 5e-2
    for name, p in m.net.mlp_coarse.named_parameters():
        _norm_close(p.grad, ref_g[name], f"{train_precision} d {name}", rtol, rmax)
    _norm_close(lat.grad, ref_lat, f"{train_precision} d latent", rtol, rmax)
    _norm_close(zc.grad, ref_z, f"{train_precision} d z", xtol, rmax)


# ------------------------------------------------------------------------------------------------ the C entry points
def test_width_mismatch_is_refused(lib):
    """A network whose d_in is not the width of the scene's z-feature layout: PNR_ERR_ARG naming both, before any launch."""
    from pixel_nerf_yolo_b200 import _lib
    m = Net(dict(DEFAULT, use_viewdirs=False), 6)            # d_in = 39
    xyz, dirs = _points(64, 800)
    pts = _lib.points_xyz(xyz.cuda(), dirs.cuda())
    cp = m.net.mlp_coarse.c_params()
    out = torch.full((1, 64, 4), float("nan"), device="cuda")
    for precision, fp32_maps in ((_lib.PREC_BF16, False), (_lib.PREC_FP32, True)):
        sc, _keep = m.net._scene(fp32_maps=fp32_maps)
        sc.flags &= ~_lib.SCENE_ZF_NO_VIEWDIRS                 # the default layout: 42 wide
        ws = torch.empty(lib.pnr_field_workspace_bytes(sc, pts, precision), dtype=torch.uint8, device="cuda")
        packed = m.net.mlp_coarse.packed().data_ptr() if precision == _lib.PREC_BF16 else None
        rc = lib.pnr_field_forward(sc, pts, cp, packed, out.data_ptr(), ws.data_ptr(), ws.numel(), precision, 6, 1.5,
                                   _lib.stream_ptr(torch.device("cuda", 0)))
        assert rc == -1 and b"d_in=39" in lib.pnr_last_error() and b"width 42" in lib.pnr_last_error()
        assert lib.pnr_last_launch_count() == 0
    torch.cuda.synchronize()
    assert out.isnan().all()
