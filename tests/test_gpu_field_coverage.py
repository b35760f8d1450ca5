"""The tcgen05 field kernel (``pair::field_pair_kernel``) over everything its dispatcher accepts (`-m gpu`), through the public API.

Every case is held to two references:

* the fp32 oracle at the bf16 tolerance used elsewhere (1e-2; sigma relative to 1 + |sigma|, 1.5x for max pooling, see
  tests/test_gpu_pooling.py): the reference BEHAVIOUR;
* ``bf16_field_reference.field_forward_bf16``, a restatement of the kernel's own bf16 arithmetic, with the RMS of the error
  over the points at ``TIGHT`` (2x for max pooling): what is left is fp32 summation order and the bf16 roundings it flips,
  while a skipped MMA or a wrong bias slot moves every point (tests/test_oracle_bf16_reference.py shows such faults move the
  reference's RMS by more than 2x the bound).  The worst element is not a usable bound: flips move single points by up to
  1.5e-3 (average) / 5.6e-3 (max pooling), as much as one skipped MMA does.

The fp32 check path (``precision="fp32"``) runs the view-count matrix at 1e-4 against the oracle.

Matrix:

1. every built view count with both pooling modes (NS 1-6 and 8 average, NS 2-6 and 8 max), SB = 1 and 3;
2. tile and super-group edges for every NS: P in {1, PP - 1, PP, PP + 1, 2 G PP - 1, 2 G PP, 2 G PP + 1}, SB = 3
   (PP = 64 / NS points per tile, G = NS tiles per super group);
3. at least three super groups per CTA pair, sized from the SM count: the big launch equals, bit for bit, the same points
   evaluated in launches of less than one wave each, and a strided subset is held to the tight bound;
4. network shapes: (n_blocks, combine_layer) from (1, 1) to (8, 8), streamed latents of 64 / 192 / 576 channels (one pass of
   the latent tile is 8 k-blocks = 512 channels), pre-projected 1792-channel latents, the longest stage program the kernel
   takes, and the YOLO head with d_out = 7 and 28;
5. refusals: NS = 7 and 9 on the tcgen05 path (the fp32 path is generic in NS), a stage program that does not fit;

and the training path (fp32 and tcgen05 arithmetics) at NS 4 and 8 with both pooling modes and at (n_blocks, combine_layer)
(4, 2) and (8, 6), with the bounds and reasons of tests/test_gpu_pooling.py.

Measured on one B200 (148 SMs, 1000 W power limit), RMS error against the bf16 reference, rgb / sigma (relative to
1 + |sigma|), worst case of each group; TIGHT = 6e-4, 1.2e-3 with max pooling:

* view counts, average, NS 1-8: 1.22e-4 / 2.33e-4 (NS 1); NS 8: 8.7e-5 / 1.3e-4;
* view counts, max, NS 2-8: 3.04e-4 / 5.57e-4 (NS 8); NS 2: 1.8e-4 / 3.1e-4;
* tile edges, all NS: 1.30e-4 / 2.18e-4 (NS 1);
* several super groups per pair: average 1.20e-4 / 2.32e-4 (NS 1), max 2.96e-4 / 5.64e-4 (NS 8);
* (n_blocks, combine_layer): 1.48e-4 / 2.40e-4 at (8, 7) NS 3; 1.94e-4 / 4.44e-4 at (8, 8) NS 1, the one case within 1.4x of
  the bound: eight blocks and lin_z before each, and no view mean to average the flips out;
* streamed latents 64 / 192 / 576: 1.17e-4 / 1.87e-4 (average), 2.33e-4 / 4.27e-4 (max); projected 1792: 9.7e-5 / 1.5e-4
  (average), 1.9e-4 / 3.8e-4 (max);
* YOLO d_out 7 / 28 (relative to the raw values' scale): 9.1e-5 / 9.5e-5;
* the 1018-stage program (n_blocks 8, 3008 streamed channels, NS 1): 2.36e-4 / 3.86e-4.

Whole file: about 45 s on the B200.
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
BUILT_NS = (1, 2, 3, 4, 5, 6, 8)


@pytest.fixture(scope="module")
def lib():
    from pixel_nerf_yolo_b200 import _lib
    assert torch.cuda.is_available()
    _lib.require_device(torch.device("cuda", 0))
    return _lib.load()


def _tile(ns):
    """(PP, G): points per pre-combine tile and tile pairs per super group (field_pair_kernel)."""
    pp = 64 // ns
    return pp, 64 // pp


def _scene(ns, sb=1, C=512):
    """synth.scene_config1 (up to 8 views around the object); a 9th view for the refusal test."""
    s = H.make_scene_dict(num_objs=sb, num_views=min(ns, 8), C=C)
    if ns > 8:
        extra = torch.stack([synth.pose_spherical(200.0 + 10.0 * o, -20.0, 1.3) for o in range(sb)])[:, None]
        s["poses"] = torch.cat((s["poses"], extra), dim=1)
        s["latent"] = synth.feature_maps(1005, sb * ns, C, 16, 16)
    return s


def _points(P, seed, num_objs=1, extent=0.9):
    g = torch.Generator().manual_seed(seed)
    xyz = (torch.rand(num_objs, P, 3, generator=g) - 0.5) * extent
    dirs = torch.nn.functional.normalize(torch.randn(num_objs, P, 3, generator=g), dim=-1)
    return xyz, dirs


class Net:
    """One PixelNeRFNet (coarse network only is queried) and the matching oracle inputs."""

    def __init__(self, scene, n_blocks=5, combine_layer=3, combine_type="average", anchors=None, precision="bf16",
                 train=False, project=None):
        from pixel_nerf_yolo_b200.conf import ConfigTree
        from pixel_nerf_yolo_b200.model import make_model
        from pixel_nerf_yolo_b200.model.model_util import make_mlp
        C = scene["latent"].shape[1]
        self.yolo = anchors is not None
        d_out = 7 * anchors if self.yolo else 4
        conf = copy.deepcopy(H.MODEL_CONF)
        for k in ("mlp_coarse", "mlp_fine"):
            conf[k].update(n_blocks=n_blocks, combine_layer=combine_layer, combine_type=combine_type)
        if self.yolo:
            conf["mlp_coarse"].update({"d_out": 7, "num_scales": 1, "num_anchors_per_scale": anchors, "yolo": True})
            conf["mlp_fine"] = {"type": "empty"}
        conf = ConfigTree.from_dict(conf)
        net = make_model(conf).eval()
        if C != net.d_latent:                # the maps come from set_latent: size the networks for them
            net.mlp_coarse = make_mlp(conf["mlp_coarse"], net.d_in, C)
            net.mlp_fine = None if self.yolo else make_mlp(conf["mlp_fine"], net.d_in, C)
            net.d_latent = net.latent_size = C
        self.state = synth.mlp_state(1, d_latent=C, n_blocks=n_blocks, combine_layer=combine_layer, d_out=d_out)
        net.mlp_coarse.load_state_dict(self.state)
        if net.mlp_fine is not None:
            net.mlp_fine.load_state_dict(synth.mlp_state(2, d_latent=C, n_blocks=n_blocks, combine_layer=combine_layer))
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
        self.net, self.scene = net, scene
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
    """The two bounds of a bf16 result: worst element against the fp32 oracle, RMS against the bf16 reference.  Returns the
    fp32 oracle's output."""
    ref32 = m.oracle(xyz, dirs) if ref32 is None else ref32
    ref16 = m.bf16_ref(xyz, dirs) if ref16 is None else ref16
    loose = _errors(out, ref32, m.yolo)
    worst = _errors(out, ref16, m.yolo)
    tight = _errors(out, ref16, m.yolo, rms=True)
    print(f"\nCOVERAGE {case}: bf16 reference RMS rgb {tight[0]:.2e} sigma {tight[1]:.2e} worst rgb {worst[0]:.2e} sigma "
          f"{worst[1]:.2e} | fp32 oracle worst rgb {loose[0]:.2e} sigma {loose[1]:.2e}")
    sig_loose = 1.5 * LOOSE if m.combine_type == "max" else LOOSE
    assert loose[0] < LOOSE and loose[1] < sig_loose, (case, "fp32 oracle", loose)
    bound = BR.tight_bound(m.combine_type)
    assert tight[0] < bound and tight[1] < bound, (case, "bf16 reference RMS", tight)
    return ref32


# ------------------------------------------------------------------------------------------------ 1. view counts x pooling
POOLING = [(ns, "average") for ns in BUILT_NS] + [(ns, "max") for ns in BUILT_NS if ns > 1]


@pytest.mark.parametrize("sb", [1, 3])
@pytest.mark.parametrize("ns,combine_type", POOLING)
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_view_counts(lib, precision, ns, combine_type, sb):
    m = Net(_scene(ns, sb), combine_type=combine_type, precision=precision)
    xyz, dirs = _points(300 // sb, 100 + ns, sb)
    out = m(xyz, dirs)
    if precision == "bf16":
        ref = _check(f"NS={ns} {combine_type} SB={sb}", m, out, xyz, dirs)
    else:
        ref = m.oracle(xyz, dirs)
        np.testing.assert_allclose(out.numpy(), ref.numpy(), atol=FP32, rtol=FP32)
    assert ref[..., 3].max() > 0.5 and ref[..., :3].std() > 0.01          # the comparison is not vacuous
    if combine_type == "max":                                               # and max pooling is not the mean in disguise
        assert (m.oracle(xyz, dirs, "average") - ref).abs().max() > 20 * LOOSE


# ------------------------------------------------------------------------------------------------ 2. tile edges
@pytest.mark.parametrize("ns", BUILT_NS)
def test_tile_and_super_group_edges(lib, ns):
    """Partial tiles, a partial super group, an odd number of tiles (the last pair's second CTA idles), one point."""
    pp, g = _tile(ns)
    sizes = sorted({1, pp - 1, pp, pp + 1, 2 * g * pp - 1, 2 * g * pp, 2 * g * pp + 1} - {0})
    m = Net(_scene(ns, 3))
    xyz, dirs = _points(sizes[-1], 200 + ns, 3)
    ref32, ref16 = m.oracle(xyz, dirs), m.bf16_ref(xyz, dirs)
    outs = []
    for P in sizes:
        out = m(xyz[:, :P].contiguous(), dirs[:, :P].contiguous())
        assert out.shape == (3, P, 4)
        loose = _errors(out, ref32[:, :P])
        assert loose[0] < LOOSE and loose[1] < LOOSE, (P, loose)
        outs.append((out, ref32[:, :P], ref16[:, :P]))
    # a few points are too few for an RMS: the tight bound holds over all launches of this NS together
    cat = lambda i: torch.cat([o[i].reshape(-1, 4) for o in outs])
    _check(f"edges NS={ns} P={sizes}", m, cat(0), None, None, cat(1), cat(2))


# ------------------------------------------------------------------------------------------------ 3. several super groups
@pytest.mark.parametrize("ns,combine_type", POOLING)
def test_several_super_groups_per_pair(lib, ns, combine_type):
    """Every CTA pair runs at least three super groups: the weight ring, the barrier parities and the relay continue across
    them.  A column's arithmetic does not depend on where it sits, so the big launch must equal launches of under one wave."""
    pp, g = _tile(ns)
    n_pairs = torch.cuda.get_device_properties(0).multi_processor_count // 2
    per_sg = 2 * g * pp                                  # points of one super group
    sb = 3
    P = math.ceil(3 * n_pairs * per_sg / sb) + 5         # >= 3 super groups per pair, and a partial last tile
    m = Net(_scene(ns, sb), combine_type=combine_type)
    xyz, dirs = _points(P, 300 + ns, sb)
    big = m(xyz, dirs)
    step = n_pairs * per_sg // (2 * sb)                  # a slice: about half a wave of super groups
    assert math.ceil(math.ceil(sb * math.ceil(step / pp) / 2) / g) < n_pairs
    for a in range(0, P, step):
        part = m(xyz[:, a:a + step].contiguous(), dirs[:, a:a + step].contiguous())
        assert torch.equal(big[:, a:a + step], part), (a, (big[:, a:a + step] - part).abs().max().item())
    stride = math.ceil(sb * P / 512)
    xs, ds = xyz[:, ::stride].contiguous(), dirs[:, ::stride].contiguous()
    _check(f"super groups NS={ns} {combine_type} P={P}x{sb}", m, big[:, ::stride], xs, ds)


# ------------------------------------------------------------------------------------------------ 4. network shapes
SHAPES = [(5, 1, 3), (5, 2, 3), (5, 4, 3), (4, 2, 3), (2, 1, 3), (1, 1, 1), (8, 4, 3), (8, 7, 3), (8, 8, 1)]


@pytest.mark.parametrize("n_blocks,combine_layer,ns", SHAPES)
def test_network_shapes(lib, n_blocks, combine_layer, ns):
    m = Net(_scene(ns), n_blocks=n_blocks, combine_layer=combine_layer)
    xyz, dirs = _points(200, 400 + n_blocks, 1)
    ref = _check(f"n_blocks={n_blocks} combine_layer={combine_layer} NS={ns}", m, m(xyz, dirs), xyz, dirs)
    assert ref[..., 3].max() > 0.5 and ref[..., :3].std() > 0.01


@pytest.mark.parametrize("C,project", [(64, False), (192, False), (576, False), (1792, True)])
@pytest.mark.parametrize("combine_type", ["average", "max"])
def test_latent_widths(lib, C, project, combine_type):
    """Streamed latents narrower than one 512-channel pass of the latent tile, or one pass and a partial one; and the
    pre-projected wide maps."""
    m = Net(_scene(3, C=C), combine_type=combine_type, project=project)
    assert m.projected == project
    xyz, dirs = _points(200, 500 + C, 1)
    _check(f"d_latent={C} projected={project} {combine_type}", m, m(xyz, dirs), xyz, dirs)


@pytest.mark.parametrize("anchors", [1, 4])
def test_yolo_head(lib, anchors):
    """d_out = 7 x anchors raw outputs, and the latent masked where a point is not in front of a view (z >= 0)."""
    m = Net(_scene(3), anchors=anchors)
    xyz, dirs = _points(200, 600 + anchors, 1, extent=3.2)
    w2c = m.sc.poses
    zc = torch.einsum("pj,vj->vp", xyz[0], w2c[:, 2, :3]) + w2c[:, 2, 3:4]     # camera z of every (view, point)
    assert 0.05 < (zc >= 0).float().mean() < 0.95          # the mask is exercised both ways
    out = m(xyz, dirs)
    assert out.shape == (1, 200, 7 * anchors)
    _check(f"YOLO d_out={7 * anchors}", m, out, xyz, dirs)


def test_longest_stage_program(lib):
    """The weight stream of n_blocks = 8 with lin_z before every block and a 3008-channel streamed latent is 1018 stages, the
    most the kernel's stage program holds (1024 entries, one of them padding) for this network; 3072 channels do not fit."""
    m = Net(_scene(1, C=3008), n_blocks=8, combine_layer=8, project=False)
    xyz, dirs = _points(100, 700, 1)
    _check("stage program 1018 stages", m, m(xyz, dirs), xyz, dirs)


# ------------------------------------------------------------------------------------------------ 5. refusals
@pytest.mark.parametrize("ns", [7, 9])
def test_unbuilt_view_counts_are_refused(lib, ns):
    """NS = 7 and 9 have no tcgen05 instantiation: an error that names NS, and the output is not written."""
    from pixel_nerf_yolo_b200 import _lib
    m = Net(_scene(ns))
    net = m.net
    xyz, dirs = _points(64, 800 + ns, 1)
    with torch.no_grad(), pytest.raises(NotImplementedError, match=f"NS={ns}"):
        net(xyz.cuda(), coarse=True, viewdirs=dirs.cuda())
    keep = (xyz.cuda(), dirs.cuda())
    pts = _lib.points_xyz(*keep)
    out = torch.full((1, 64, 4), float("nan"), device="cuda")
    sc, _keep = net._scene(fp32_maps=False)
    mlp = net.mlp_coarse
    ws = torch.empty(max(lib.pnr_field_workspace_bytes(sc, pts, _lib.PREC_BF16), 16), dtype=torch.uint8, device="cuda")
    rc = lib.pnr_field_forward(sc, pts, mlp.c_params(), mlp.packed().data_ptr(), out.data_ptr(), ws.data_ptr(), ws.numel(),
                               _lib.PREC_BF16, 6, 1.5, _lib.stream_ptr(torch.device("cuda", 0)))
    assert rc == -3 and f"NS={ns}".encode() in lib.pnr_last_error()
    torch.cuda.synchronize()
    assert out.isnan().all()
    if ns == 7:                                          # the fp32 check path is generic in NS
        net.precision = "fp32"
        np.testing.assert_allclose(m(xyz, dirs).numpy(), m.oracle(xyz, dirs).numpy(), atol=FP32, rtol=FP32)


def test_stage_program_overflow_is_refused_at_pack_time(lib):
    m = Net(_scene(1, C=3072), n_blocks=8, combine_layer=8, project=False)
    with pytest.raises(NotImplementedError, match="stage program"):
        m.net.mlp_coarse.packed()
    assert lib.pnr_last_launch_count() == 0
    xyz, dirs = _points(16, 900, 1)
    with pytest.raises(NotImplementedError, match="stage program"):
        m(xyz, dirs)


# ------------------------------------------------------------------------------------------------ training path
def _norm_close(got, ref, what, rtol, rmax):
    got, ref = got.detach().cpu().double(), ref.detach().cpu().double()
    rel = ((got - ref).norm() / ref.norm().clamp_min(1e-30)).item()
    worst = ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()
    assert rel <= rtol and worst <= rmax, f"{what}: rel-norm err {rel:.3e} (<= {rtol}), worst element {worst:.3e} (<= {rmax})"


def _oracle_grads(m, xyz, dirs, gout, emulate_bf16=False, record=None):
    sc = copy.copy(m.sc)
    sc.latent = sc.latent.clone().requires_grad_(True)
    mc = {k: v.clone().requires_grad_(True) for k, v in m.state.items()}
    xo = xyz.clone().requires_grad_(True)
    with PO.combine_type(m.combine_type, record):
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


TRAIN = [(4, "average", 5, 3), (4, "max", 5, 3), (8, "average", 5, 3), (8, "max", 5, 3), (3, "average", 4, 2),
         (3, "average", 8, 6)]


@pytest.mark.parametrize("ns,combine_type,n_blocks,combine_layer", TRAIN)
@pytest.mark.parametrize("train_precision", ["fp32", "bf16"])
def test_field_backward(lib, train_precision, ns, combine_type, n_blocks, combine_layer):
    """PixelNeRFNet.forward(xyz, viewdirs) in training mode and its backward vs autograd over the oracle: fp32 against the fp32
    oracle (1e-3 in norm), tcgen05 against the bf16-operand emulation (5e-2 in norm; see tests/test_gpu_pooling.py)."""
    scene = _scene(ns)
    m = Net(scene, n_blocks=n_blocks, combine_layer=combine_layer, combine_type=combine_type, train=True)
    m.net.train_precision = train_precision
    xyz, dirs = _points(300 if train_precision == "bf16" else 160, 1000 + ns + n_blocks, 1)
    if train_precision == "fp32":
        xyz, dirs = _untied(m, xyz, dirs)
    gout = torch.randn(*xyz.shape[:2], 4, generator=torch.Generator().manual_seed(ns))
    ref32, g32, lat32, x32 = _oracle_grads(m, xyz, dirs, gout)
    lat = scene["latent"].cuda().clone().requires_grad_(True)
    m.net.encoder.set_latent(lat)
    xc = xyz.cuda().requires_grad_(True)
    out = m.net(xc, coarse=True, viewdirs=dirs.cuda())
    o = out.detach().cpu()
    (out * gout.cuda()).sum().backward()
    if train_precision == "fp32":
        np.testing.assert_allclose(o.numpy(), ref32.numpy(), atol=1e-4, rtol=0)
        ref_g, ref_lat, ref_x, rtol, rmax, xtol, xmax = g32, lat32, x32, 1e-3, 3e-2, 3e-3, 3e-2
    else:
        np.testing.assert_allclose(o.numpy()[..., :3], ref32.numpy()[..., :3], atol=LOOSE, rtol=0)
        np.testing.assert_allclose(o.numpy()[..., 3], ref32.numpy()[..., 3], atol=LOOSE, rtol=LOOSE)
        ref16, ref_g, ref_lat, ref_x = _oracle_grads(m, xyz, dirs, gout, emulate_bf16=True)
        # same arithmetic: summation order and the bf16 rounding flips it causes.  Max pooling passes the flips of the winning
        # view through, and with more views more of them: measured 4.0e-3 on one element of 1200 at NS = 8 (the inference
        # kernel's worst element is 5.3e-3 at NS = 6), hence 6e-3 above NS = 5
        same = (6e-3 if ns > 5 else 3e-3) if combine_type == "max" else 2e-3
        np.testing.assert_allclose(o.numpy(), ref16.numpy(), atol=same, rtol=same)
        # one ReLU (or, with max pooling, argmax) flip changes one gradient term by O(1), and 300 rows do not average it out
        # (DESIGN.md section 2).  Measured: worst element 2.4e-1 on d blocks.2.fc_0.weight at (n_blocks, combine_layer) =
        # (4, 2); norm 3.4e-2 on d blocks.2.fc_0.bias there and 3.3e-2 on d lin_in.weight at NS = 8 max (3e-2 holds at the
        # default shape, test_gpu_pooling.py).  The fp32 arithmetic above runs the same pooling and stage loops at 1e-3.
        rtol, rmax, xtol, xmax = 5e-2, 3e-1, 5e-2, 3e-1
    for name, p in m.net.mlp_coarse.named_parameters():
        _norm_close(p.grad, ref_g[name], f"{train_precision} d {name}", rtol, rmax)
    _norm_close(lat.grad, ref_lat, f"{train_precision} d latent", rtol, rmax)
    _norm_close(xc.grad, ref_x, f"{train_precision} d xyz", xtol, xmax)
