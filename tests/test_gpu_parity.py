"""GPU parity tests (run on the B200 box with -m gpu): every call goes through the C-ABI library
(ctypes), results are compared with the CPU oracle on the same seeded inputs and with the golden vectors
produced by the unmodified reference.

Tolerances
  * sampler stages (sample_coarse, depth samples, sort, searchsorted bins): BIT-EXACT vs the oracle;
    the only admitted deviation is an inverse-CDF bin flip where u lies within 4 ulp of a CDF knot
    (the oracle's torch.sum order is host-CPU dependent);
  * compositing given identical field values: 1e-6;
  * field / render with fp32 arithmetic (SIMT check path): 1e-4  (summation order only);
  * field / render with bf16 tensor-core operands (production path): 1e-2 max-abs on rgb/depth,
    as stated by BASELINE.json north_star.  That bound cannot see one skipped MMA: tests/test_gpu_field_coverage.py
    holds the field kernel to a restatement of its own bf16 arithmetic (tests/bf16_field_reference.py, DESIGN.md
    section 2) at a bound that can.
"""
import numpy as np
import pytest
import torch

import helpers as H
import pixel_nerf_yolo_b200.synth as synth
from oracle import pixelnerf_oracle as O

pytestmark = pytest.mark.gpu
T = torch.from_numpy


@pytest.fixture(scope="module")
def lib():
    from pixel_nerf_yolo_b200 import _lib
    assert torch.cuda.is_available()
    _lib.require_device(torch.device("cuda", 0))
    return _lib.load()


def _renderer(**kw):
    from pixel_nerf_yolo_b200.render import NeRFRenderer
    from pixel_nerf_yolo_b200.conf import ConfigTree
    conf = dict(H.RENDER_CONF)
    conf.update(kw)
    return NeRFRenderer.from_conf(ConfigTree.from_dict(conf)).eval().cuda()


# ------------------------------------------------------------------------------------------------ ray tile
@pytest.mark.parametrize("Kc,lindisp", [(64, False), (128, False), (256, False), (96, False), (64, True)])
def test_sample_coarse_bit_exact(lib, Kc, lindisp):
    B = 777
    rays = H.rays_subset(1, B)[0]
    rays[:, 6] = 0.8 + 0.1 * torch.rand(B)
    noise = torch.rand(B, Kc, generator=torch.Generator().manual_seed(1))
    r = _renderer(n_coarse=Kc)
    r.lindisp = lindisp
    z = r.sample_coarse(rays.cuda(), noise.cuda()).cpu()
    assert torch.equal(z, O.sample_coarse(rays, noise, Kc, lindisp))


def test_sample_coarse_golden(lib, golden):
    rays = synth.target_rays(128)[:, T(golden["sb1_ray_idx"]).long()][0]
    z = _renderer().sample_coarse(rays.cuda(), T(golden["sb1_noise_coarse"]).cuda()).cpu()
    assert torch.equal(z, T(golden["sb1_z_coarse"]))


@pytest.mark.parametrize("K,white", [(64, True), (96, True), (96, False), (288, True), (1, True)])
def test_composite_matches_oracle(lib, K, white):
    B = 1111
    g = torch.Generator().manual_seed(K)
    rays = H.rays_subset(1, B)[0]
    z, _ = torch.sort(0.8 + torch.rand(B, K, generator=g), dim=-1)
    out = torch.cat((torch.rand(B, K, 3, generator=g), 30 * torch.rand(B, K, 1, generator=g) ** 3 - 1.0), dim=-1)
    r = _renderer(white_bkgd=white)
    w, rgb, depth = r.composite_values(out.cuda(), z.cuda(), rays.cuda())
    wo, rgbo, do = O.alpha_composite(out, z, rays, white)
    np.testing.assert_allclose(w.cpu().numpy(), wo.numpy(), atol=1e-6, rtol=0)
    np.testing.assert_allclose(rgb.cpu().numpy(), rgbo.numpy(), atol=2e-6, rtol=0)
    np.testing.assert_allclose(depth.cpu().numpy(), do.numpy(), atol=2e-6, rtol=0)


@pytest.mark.parametrize("Kc,kf,kfd", [(64, 16, 16), (128, 16, 16), (256, 16, 16), (64, 32, 0), (64, 0, 16)])
def test_resample_matches_oracle(lib, Kc, kf, kfd):
    B = 2000
    g = torch.Generator().manual_seed(Kc + kf)
    rays = H.rays_subset(1, B)[0]
    zc = O.sample_coarse(rays, torch.rand(B, Kc, generator=g), Kc)
    w = torch.rand(B, Kc, generator=g) ** 6          # peaky weights, many near-zero bins
    w[::7] = 0.0                                     # all-zero rows: uniform pdf from the 1e-5 floor
    depth = 0.7 + 1.2 * torch.rand(B, generator=g)   # some outside [near, far]: exercises the clamp
    u, j = torch.rand(B, kf, generator=g), torch.rand(B, kf, generator=g)
    u[:, :1] = 0.0                                   # edge: u == cdf[0]
    gz = torch.randn(B, kfd, generator=g)
    r = _renderer(n_coarse=Kc, n_fine=kf + kfd, n_fine_depth=kfd)
    cu = lambda t: t.cuda() if t.numel() else None
    z_all, dbg = r.resample(rays.cuda(), zc.cuda(), cu(w), cu(depth), cu(u), cu(j), cu(gz), debug=True)
    parts = [zc]
    if kf:
        zf, inds = O.sample_fine(rays, w, u, j, Kc, return_inds=True)
        mism = dbg[0].cpu().long() != inds
        if mism.any():   # admitted only at CDF knots (|u - knot| within a few ulp)
            pdf = (w + 1e-5) / (w + 1e-5).sum(-1, keepdim=True)
            cdf = torch.cat((torch.zeros(B, 1), torch.cumsum(pdf, -1)), -1)
            near_knot = (cdf[:, None, :] - u[:, :, None]).abs().min(-1).values < 4e-7
            assert (near_knot | ~mism).all() and mism.float().mean() < 1e-3
        ok = ~mism
        assert torch.equal(dbg[1].cpu()[ok], zf[ok])
        parts.append(torch.where(ok, zf, dbg[1].cpu()))
    if kfd:
        zd = O.sample_fine_depth(rays, depth, gz, 0.01)
        assert torch.equal(dbg[2].cpu(), zd)
        parts.append(zd)
    assert torch.equal(z_all.cpu(), torch.sort(torch.cat(parts, -1), -1).values)


def test_resample_golden(lib, golden):
    for tag, nobj in (("sb1", 1), ("sb2", 2)):
        allr = torch.cat([synth.target_rays(128, 15.0 + 20 * s, -10.0) for s in range(nobj)])
        rays = allr[:, T(golden[f"{tag}_ray_idx"]).long()].reshape(-1, 8)
        g = lambda k: T(golden[f"{tag}_{k}"]).cuda()
        r = _renderer()
        z_all, dbg = r.resample(rays.cuda(), g("z_coarse"), g("coarse_weights").reshape(-1, 64), g("coarse_depth").reshape(-1),
                                g("noise_fine_u"), g("noise_fine_jitter"), g("noise_depth"), debug=True)
        assert torch.equal(dbg[1].cpu(), T(golden[f"{tag}_z_fine"]))
        assert torch.equal(dbg[2].cpu(), T(golden[f"{tag}_z_depth"]))


# ------------------------------------------------------------------------------------------------ operators
def test_positional_encoding_operator(lib, golden):
    from pixel_nerf_yolo_b200.model.code import PositionalEncoding
    out = PositionalEncoding(6, 3, 1.5, True).cuda()(T(golden["pe_x"]).cuda()).cpu()
    np.testing.assert_allclose(out.numpy(), golden["pe_out"], atol=2e-6, rtol=0)
    x = torch.randn(1000, 3) * 2
    np.testing.assert_allclose(PositionalEncoding(6, 3, 1.5, True).cuda()(x.cuda()).cpu().numpy(),
                               O.positional_encoding(x).numpy(), atol=3e-6, rtol=0)


def test_index_operator_matches_grid_sample(lib, golden):
    scene = H.make_scene_dict()
    net = H.build_net(scene)
    out = net.encoder.index(T(golden["index_uv"]).cuda(), None, net.image_shape).cpu()
    np.testing.assert_allclose(out.numpy(), golden["index_out"], atol=3e-6, rtol=0)


def test_resnetfc_operator(lib, golden):
    net = H.build_net(H.make_scene_dict(), coarse_seed=21)
    out = net.mlp_coarse(T(golden["mlp_zx"]).cuda(), combine_inner_dims=(3, 5)).cpu()
    np.testing.assert_allclose(out.reshape(2, 5, 4).numpy(), golden["mlp_out"], atol=5e-5, rtol=1e-4)


def test_gather_encode_matches_oracle(lib):
    from pixel_nerf_yolo_b200 import _lib
    scene = H.make_scene_dict(num_objs=2)
    net = H.build_net(scene)
    sc_o = H.oracle_scene(scene)
    g = torch.Generator().manual_seed(3)
    P = 301
    xyz = (torch.rand(2, P, 3, generator=g) - 0.5) * 1.2       # some project outside the maps
    dirs = torch.nn.functional.normalize(torch.randn(2, P, 3, generator=g), dim=-1)
    for fp32 in (True, False):
        sc, keep = net._scene(fp32_maps=fp32)
        xd, dd = xyz.cuda(), dirs.cuda()
        pts = _lib.points_xyz(xd, dd)
        lat = torch.empty(2 * 3 * P, 512, device="cuda", dtype=torch.float32)
        zf = torch.empty(2 * 3 * P, 42, device="cuda")
        _lib.check(lib.pnr_gather_encode(sc, pts, lat.data_ptr(), zf.data_ptr(), 1, 6, 1.5, _lib.stream_ptr(lat.device)), "gather")
        # oracle pieces
        NS = 3
        rep = lambda t: t.unsqueeze(1).expand(-1, NS, *t.shape[1:]).reshape(-1, *t.shape[1:])
        R = sc_o.poses[:, None, :3, :3]
        x_rot = torch.matmul(R, rep(xyz).unsqueeze(-1))[..., 0]
        x_cam = x_rot + sc_o.poses[:, None, :3, 3]
        uv = -x_cam[:, :, :2] / x_cam[:, :, 2:] * sc_o.focal.unsqueeze(1) + sc_o.c.unsqueeze(1)
        lat_o = O.bilinear_index(sc_o.latent, uv, sc_o.latent_scaling, sc_o.image_shape).transpose(1, 2).reshape(-1, 512)
        zf_o = torch.cat((O.positional_encoding(x_rot.reshape(-1, 3)), torch.matmul(R, rep(dirs.unsqueeze(-1))).reshape(-1, 3)), 1)
        np.testing.assert_allclose(zf.cpu().numpy(), zf_o.numpy(), atol=2e-5, rtol=0)
        np.testing.assert_allclose(lat.cpu().numpy(), lat_o.numpy(), atol=(2e-5 if fp32 else 1.5e-2), rtol=0)
        assert (lat_o.abs().sum(-1) == 0).any() and (lat_o.abs().sum(-1) > 0).any()   # zero-padding branch is hit


# ------------------------------------------------------------------------------------------------ field
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("bf16", 1e-2)])
def test_field_matches_reference_golden(lib, golden, precision, tol):
    """PixelNeRFNet.forward vs outputs of the unmodified reference (19 points, both MLPs)."""
    net = H.build_net(H.make_scene_dict(), precision=precision)
    with torch.no_grad():
        c = net(T(golden["field_xyz"]).cuda(), coarse=True, viewdirs=T(golden["field_dirs"]).cuda()).cpu()
        f = net(T(golden["field_xyz"]).cuda(), coarse=False, viewdirs=T(golden["field_dirs"]).cuda()).cpu()
    for out, ref in ((c, golden["field_coarse"]), (f, golden["field_fine"])):
        assert np.abs(out.numpy()[..., :3] - ref[..., :3]).max() < tol
        assert np.abs(out.numpy()[..., 3] - ref[..., 3]).max() < tol * max(1.0, np.abs(ref[..., 3]).max())


@pytest.mark.parametrize("num_objs,num_views,P", [(1, 3, 1000), (2, 3, 333), (1, 1, 500), (1, 5, 257), (1, 2, 64), (3, 4, 100)])
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("bf16", 1e-2)])
def test_field_matches_oracle(lib, precision, tol, num_objs, num_views, P):
    scene = H.make_scene_dict(num_objs=num_objs, num_views=num_views)
    net = H.build_net(scene, precision=precision)
    g = torch.Generator().manual_seed(P)
    xyz = (torch.rand(num_objs, P, 3, generator=g) - 0.5) * 0.9
    dirs = torch.nn.functional.normalize(torch.randn(num_objs, P, 3, generator=g), dim=-1)
    with torch.no_grad():
        out = net(xyz.cuda(), coarse=True, viewdirs=dirs.cuda()).cpu()
    ref = O.field_forward(H.oracle_scene(scene), synth.mlp_state(1), xyz, dirs)
    err_rgb = (out[..., :3] - ref[..., :3]).abs().max().item()
    err_sig = ((out[..., 3] - ref[..., 3]).abs() / (1 + ref[..., 3].abs())).max().item()
    assert err_rgb < tol and err_sig < tol, (err_rgb, err_sig)
    assert ref[..., 3].max() > 0.5 and ref[..., :3].std() > 0.01          # the comparison is not vacuous


@pytest.mark.parametrize("C,enc", [(1792, {"backbone": "custom", "pretrained": False, "index_padding": "zeros"}),
                                   (256, {"backbone": "resnet34", "pretrained": False, "num_layers": 3, "index_padding": "zeros"}),
                                   (1024, {"backbone": "resnet34", "pretrained": False, "num_layers": 5, "index_padding": "zeros"})])
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("bf16", 1e-2)])
def test_field_other_latent_widths(lib, precision, tol, C, enc):
    """BASELINE config 4 shape: YOLO-sized 1792-channel maps (and 256 / 1024-channel resnet pyramids): lin_z is streamed
    through the 512-channel latent tile in passes."""
    conf = dict(H.MODEL_CONF)
    conf["encoder"] = enc
    scene = H.make_scene_dict(num_objs=1, num_views=3, feat=12, C=C)
    net = H.build_net(scene, precision=precision, model_conf=conf)
    g = torch.Generator().manual_seed(C)
    P = 150
    xyz = (torch.rand(1, P, 3, generator=g) - 0.5) * 0.9
    dirs = torch.nn.functional.normalize(torch.randn(1, P, 3, generator=g), dim=-1)
    ref = O.field_forward(H.oracle_scene(scene), synth.mlp_state(1, d_latent=C), xyz, dirs)
    # bf16: both ways of feeding a latent to lin_z -- streamed through the kernel in 512-channel passes, and (default for
    # C > 512) the pre-projected maps with identity lin_z stages (PNR_SCENE_PROJECTED)
    for project in ((False, True) if precision == "bf16" else (None,)):
        net.project_wide_latent = project
        with torch.no_grad():
            out = net(xyz.cuda(), coarse=True, viewdirs=dirs.cuda()).cpu()
        err_rgb = (out[..., :3] - ref[..., :3]).abs().max().item()
        err_sig = ((out[..., 3] - ref[..., 3]).abs() / (1 + ref[..., 3].abs())).max().item()
        assert err_rgb < tol and err_sig < tol, (project, err_rgb, err_sig)


# ------------------------------------------------------------------------------------------------ render
def _render_cuda(net, rays, noise, **kw):
    r = _renderer(**kw)
    r.noise_override = {k: v.cuda() for k, v in noise.items()}
    with torch.no_grad():
        return r(net, rays.cuda(), want_weights=True)


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("bf16", 1e-2)])
def test_render_matches_reference_golden(lib, golden, precision, tol):
    """End-to-end NeRFRenderer.forward vs the unmodified reference, SB=1 (configs 1/2) and SB=2 (config 3)."""
    for tag, nobj in (("sb1", 1), ("sb2", 2)):
        scene = H.make_scene_dict(num_objs=nobj)
        net = H.build_net(scene, precision=precision)
        allr = torch.cat([synth.target_rays(128, 15.0 + 20 * s, -10.0) for s in range(nobj)])
        rays = allr[:, T(golden[f"{tag}_ray_idx"]).long()]
        noise = {k: T(golden[f"{tag}_noise_{k}"]) for k in ("coarse", "fine_u", "fine_jitter", "depth")}
        res = _render_cuda(net, rays, noise)
        for lvl in ("coarse", "fine"):
            for k in ("rgb", "depth"):
                err = np.abs(res[lvl][k].cpu().numpy() - golden[f"{tag}_{lvl}_{k}"]).max()
                assert err < tol, (tag, lvl, k, err)
        if precision == "fp32":
            np.testing.assert_allclose(res.fine.weights.cpu().numpy(), golden[f"{tag}_fine_weights"], atol=1e-4)


@pytest.mark.parametrize("num_views,Kc", [(3, 64), (1, 64), (5, 64), (3, 128)])
def test_render_bf16_matches_oracle(lib, num_views, Kc):
    scene = H.make_scene_dict(num_views=num_views)
    net = H.build_net(scene, precision="bf16")
    B = 300
    rays = H.rays_subset(1, B)
    noise = H.make_noise(B, kc=Kc)
    res = _render_cuda(net, rays, noise, n_coarse=Kc)
    ref = O.render(H.oracle_scene(scene), synth.mlp_state(1), synth.mlp_state(2), rays,
                   O.RenderNoise(noise["coarse"], noise["fine_u"], noise["fine_jitter"], noise["depth"]), n_coarse=Kc)
    for lvl in ("coarse", "fine"):
        assert (res[lvl].rgb.cpu() - ref[lvl]["rgb"]).abs().max() < 1e-2
        assert (res[lvl].depth.cpu() - ref[lvl]["depth"]).abs().max() < 1e-2
    assert 0.2 < ref["fine"]["weights"].sum(-1).mean() < 0.999


def test_render_edge_cases(lib):
    """Empty ray batch, a batch that is not a multiple of any tile size, coarse-only rendering."""
    scene = H.make_scene_dict()
    net = H.build_net(scene, precision="bf16")
    r = _renderer()
    wrapped = r.bind_parallel(net, None, simple_output=True).eval()
    rgb, depth = wrapped(torch.zeros(0, 5, 8).cuda())
    assert rgb.shape == (0, 3) and depth.shape == (0,)
    rays = H.rays_subset(1, 37)
    rgb, depth = wrapped(rays.cuda())
    assert rgb.shape == (1, 37, 3) and depth.shape == (1, 37) and torch.isfinite(rgb).all()
    r2 = _renderer(n_fine=0, n_fine_depth=0)
    out = r2(net, rays.cuda())
    assert len(out.fine) == 0 and out.coarse.rgb.shape == (1, 37, 3)


def test_full_image_properties(lib):
    """BASELINE config 2 size (128x128, 16384 rays, 3 views) through size-independent properties:
    (a) rendering the image in two halves gives bit-identical pixels to one call (tiles are independent),
    (b) weights are a sub-probability, depth lies in [near, far] scaled by opacity, rgb in [0, 1+eps],
    (c) bf16 and fp32 paths agree within the stated tolerance on a 1024-ray subset of the same image."""
    scene = H.make_scene_dict(feat=64)
    net = H.build_net(scene, precision="bf16")
    rays = synth.target_rays(128)
    B = rays.shape[1]
    noise = H.make_noise(B, seed=4)
    res = _render_cuda(net, rays, noise)
    half = B // 2 + 13
    r = _renderer()
    parts = []
    for s, e in ((0, half), (half, B)):
        r.noise_override = {k: v[s:e].cuda() for k, v in noise.items()}
        with torch.no_grad():
            parts.append(r(net, rays[:, s:e].cuda(), want_weights=True))
    for k in ("rgb", "depth", "weights"):
        assert torch.equal(torch.cat([p.fine[k] for p in parts], 1), res.fine[k]), k
    w = res.fine.weights
    assert (w >= 0).all() and (w.sum(-1) <= 1 + 1e-4).all()
    assert (res.fine.depth <= 1.8 * (1 + 1e-4)).all() and (res.fine.depth >= 0).all()
    assert (res.fine.rgb >= -1e-4).all() and (res.fine.rgb <= 1 + 1e-3).all()
    sub = torch.arange(0, B, 16)
    net.precision = "fp32"
    sub_noise = {k: v[sub] for k, v in noise.items()}
    res32 = _render_cuda(net, rays[:, sub], sub_noise)
    assert (res32.fine.rgb - res.fine.rgb[:, sub]).abs().max() < 1e-2
    assert (res32.fine.depth - res.fine.depth[:, sub]).abs().max() < 1e-2


@pytest.mark.parametrize("num_objs,want_weights", [(1, True), (2, False)])
def test_single_call_render_equals_staged_path(lib, num_objs, want_weights):
    """pnr_render_forward (the whole NeRFRenderer.forward as one C call, FOUR launches: sample_coarse folded into the coarse
    field's point fetch, composite + resampling fused) computes the same values as the stage-by-stage path (six launches):
    bit-identical outputs."""
    scene = H.make_scene_dict(num_objs=num_objs, num_views=3)
    net = H.build_net(scene, precision="bf16")
    rays = H.rays_subset(num_objs, 333, seed=2)
    noise = H.make_noise(num_objs * 333, seed=6)
    r = _renderer()
    r.noise_override = {k: v.cuda() for k, v in noise.items()}
    assert net.fused_render_ready()
    with torch.no_grad():
        a = r(net, rays.cuda(), want_weights=want_weights)
        n_single = r.last_launches
        net.fused_render_ready = lambda: False
        b = r(net, rays.cuda(), want_weights=want_weights)
        n_staged = r.last_launches
    assert n_single == 4 and n_staged == 6
    for lvl in ("coarse", "fine"):
        assert torch.equal(a[lvl].rgb, b[lvl].rgb) and torch.equal(a[lvl].depth, b[lvl].depth)
        if want_weights:
            assert torch.equal(a[lvl].weights, b[lvl].weights)
    # coarse-only renderer and the RNG contract: same seed -> same image on both paths
    r2 = _renderer(n_fine=0, n_fine_depth=0)
    with torch.no_grad():
        torch.manual_seed(3)
        c = r2(net, rays.cuda())
        del net.fused_render_ready
        torch.manual_seed(3)
        d = r2(net, rays.cuda())
    assert len(c.fine) == 0 and torch.equal(c.coarse.rgb, d.coarse.rgb)
    r3 = _renderer()
    with torch.no_grad():
        torch.manual_seed(4)
        e = r3(net, rays.cuda())
        net.fused_render_ready = lambda: False
        torch.manual_seed(4)
        f = r3(net, rays.cuda())
    assert torch.equal(e.fine.rgb, f.fine.rgb) and torch.equal(e.fine.depth, f.fine.depth)


# ------------------------------------------------------------------------------------------------ lindisp (nerf.py:121,153)
def _lindisp_renderer():
    r = _renderer(white_bkgd=False)
    r.lindisp = True                      # the reference passes it as a from_conf/constructor argument (dataset property)
    assert not r.white_bkgd
    return r


def test_lindisp_samplers_bit_exact_vs_reference_golden(lib):
    """Linear-in-disparity depths (the DTU setting) with per-ray near/far: coarse samples, importance samples, depth samples
    and the merged sorted depths equal the unmodified reference's bit for bit."""
    from test_oracle_golden import lindisp_case
    g, rays, nz = lindisp_case()
    r = _lindisp_renderer()
    rc = rays.reshape(-1, 8).cuda()
    zc = r.sample_coarse(rc, nz["coarse"].cuda())
    assert torch.equal(zc.cpu(), T(g["z_coarse"]))
    z_all, dbg = r.resample(rc, zc, T(g["coarse_weights"]).reshape(-1, 64).cuda(), T(g["coarse_depth"]).reshape(-1).cuda(),
                            nz["fine_u"].cuda(), nz["fine_jitter"].cuda(), nz["depth"].cuda(), debug=True)
    assert torch.equal(dbg[1].cpu(), T(g["z_fine"]))
    assert torch.equal(dbg[2].cpu(), T(g["z_depth"]))
    merged = torch.sort(torch.cat((T(g["z_coarse"]), T(g["z_fine"]), T(g["z_depth"])), -1), -1).values
    assert torch.equal(z_all.cpu(), merged)


def test_lindisp_resample_matches_oracle(lib):
    """Same as test_resample_matches_oracle at B = 2000 with lindisp: only bin flips at CDF knots are admitted."""
    B, Kc, kf, kfd = 2000, 64, 16, 16
    g = torch.Generator().manual_seed(77)
    rays = H.rays_subset(1, B)[0].clone()
    rays[:, 6] = 0.5 + 0.5 * torch.rand(B, generator=g)
    rays[:, 7] = 1.5 + torch.rand(B, generator=g)
    zc = O.sample_coarse(rays, torch.rand(B, Kc, generator=g), Kc, lindisp=True)
    w = torch.rand(B, Kc, generator=g) ** 6
    depth = 0.4 + 2.4 * torch.rand(B, generator=g)
    u, j = torch.rand(B, kf, generator=g), torch.rand(B, kf, generator=g)
    gz = torch.randn(B, kfd, generator=g)
    r = _lindisp_renderer()
    z_all, dbg = r.resample(rays.cuda(), zc.cuda(), w.cuda(), depth.cuda(), u.cuda(), j.cuda(), gz.cuda(), debug=True)
    zf, inds = O.sample_fine(rays, w, u, j, Kc, lindisp=True, return_inds=True)
    ok = dbg[0].cpu().long() == inds
    assert ok.float().mean() > 1 - 1e-3
    assert torch.equal(dbg[1].cpu()[ok], zf[ok])
    zd = O.sample_fine_depth(rays, depth, gz, 0.01)
    assert torch.equal(dbg[2].cpu(), zd)
    assert torch.equal(z_all.cpu(), torch.sort(torch.cat((zc, torch.where(ok, zf, dbg[1].cpu()), zd), -1), -1).values)


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("bf16", 1e-2)])
def test_lindisp_render_matches_reference_golden(lib, precision, tol):
    """Full NeRFRenderer.forward with lindisp=True, black background, per-ray bounds vs the unmodified reference; the
    single-call path (pnr_render_forward) and the staged path both carry the flag."""
    from test_oracle_golden import lindisp_case
    g, rays, nz = lindisp_case()
    scene = H.make_scene_dict()
    net = H.build_net(scene, precision=precision)
    r = _lindisp_renderer()
    r.noise_override = {k: v.cuda() for k, v in nz.items()}
    with torch.no_grad():
        res = r(net, rays.cuda(), want_weights=True)
        for lvl in ("coarse", "fine"):
            for k in ("rgb", "depth"):
                err = np.abs(res[lvl][k].cpu().numpy() - g[f"{lvl}_{k}"]).max()
                assert err < tol, (lvl, k, err)
        if precision == "fp32":
            np.testing.assert_allclose(res.fine.weights.cpu().numpy(), g["fine_weights"], atol=1e-4)
        else:
            assert net.fused_render_ready()
            net.fused_render_ready = lambda: False
            staged = r(net, rays.cuda(), want_weights=True)
            assert torch.equal(staged.fine.rgb, res.fine.rgb) and torch.equal(staged.fine.depth, res.fine.depth)


def test_scheduled_resolution_is_applied_at_forward(lib):
    """nerf.py:271-273: a renderer restored from a checkpoint renders at the resolution its last_sched buffer names."""
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.render import NeRFRenderer
    conf = {"n_coarse": 64, "n_fine": 32, "n_fine_depth": 16, "white_bkgd": True, "sched": [[2, 5], [96, 128], [48, 64]]}
    src = NeRFRenderer.from_conf(ConfigTree.from_dict(conf))
    src.sched_step(5)
    r = NeRFRenderer.from_conf(ConfigTree.from_dict(conf)).eval().cuda()
    r.load_state_dict(src.state_dict())
    net = H.build_net(H.make_scene_dict(), precision="bf16")
    rays = H.rays_subset(1, 50)
    with torch.no_grad():
        out = r(net, rays.cuda(), want_weights=True)
    assert (r.n_coarse, r.n_fine) == (128, 64)
    assert out.coarse.weights.shape == (1, 50, 128) and out.fine.weights.shape == (1, 50, 192)
    noise = H.make_noise(50, kc=128, kf=48, kfd=16)
    r.noise_override = {k: v.cuda() for k, v in noise.items()}
    with torch.no_grad():
        res = r(net, rays.cuda())
    ref = O.render(H.oracle_scene(H.make_scene_dict()), synth.mlp_state(1), synth.mlp_state(2), rays,
                   O.RenderNoise(noise["coarse"], noise["fine_u"], noise["fine_jitter"], noise["depth"]), n_coarse=128, n_fine=64)
    assert (res.fine.rgb.cpu() - ref["fine"]["rgb"]).abs().max() < 1e-2
    assert (res.fine.depth.cpu() - ref["fine"]["depth"]).abs().max() < 1e-2


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("bf16", 1e-2)])
def test_camera_formats_match_reference_golden(lib, precision, tol):
    """focal as a scalar / (SB,) / (SB, 2) / one (1, 2) row, principal point absent / scalar / (SB,) / (SB, 2): the drop-in's
    set_cameras broadcasts per-object rows over the source views exactly as models.py:225-230 does (SB = 2 x 3 views)."""
    from test_oracle_golden import CAMERA_CASES, camera_goldens
    g = camera_goldens()
    scene = H.make_scene_dict(num_objs=2)
    net = H.build_net(scene, precision=precision)
    xyz, dirs = T(g["xyz"]).cuda(), T(g["dirs"]).cuda()
    for name in CAMERA_CASES:
        c = T(g[name + "_c"]).cuda() if name + "_c" in g else None
        net.set_cameras(scene["poses"].reshape(-1, 4, 4).cuda(), T(g[name + "_focal"]).cuda(), scene["image_wh"], c)
        with torch.no_grad():
            out = net(xyz, coarse=True, viewdirs=dirs)
        ref = g[name]
        err_rgb = np.abs(out[..., :3].cpu().numpy() - ref[..., :3]).max()
        # sigma is unbounded (values up to ~10 here): bf16 operand rounding scales with it
        err_sig = (np.abs(out[..., 3].cpu().numpy() - ref[..., 3]) / np.maximum(1.0, np.abs(ref[..., 3]))).max()
        assert err_rgb < tol and err_sig < tol, (name, err_rgb, err_sig)


def test_render_without_fine_network_uses_coarse_network(lib):
    """eval/eval.py:140 sets ``net.mlp_fine = None`` for coarse-only checkpoints; the fine pass then runs the coarse network
    (models.py:291) -- on the single-call path (null mlp_fine in pnr_render_args) and on the staged path alike."""
    scene = H.make_scene_dict()
    net = H.build_net(scene, precision="bf16")
    net.mlp_fine = None
    rays, noise = H.rays_subset(1, 100), H.make_noise(100)
    res = _render_cuda(net, rays, noise)
    ref = O.render(H.oracle_scene(scene), synth.mlp_state(1), None, rays,
                   O.RenderNoise(noise["coarse"], noise["fine_u"], noise["fine_jitter"], noise["depth"]))
    for lvl in ("coarse", "fine"):
        assert (res[lvl].rgb.cpu() - ref[lvl]["rgb"]).abs().max() < 1e-2
        assert (res[lvl].depth.cpu() - ref[lvl]["depth"]).abs().max() < 1e-2
    two = O.render(H.oracle_scene(scene), synth.mlp_state(1), synth.mlp_state(2), rays,
                   O.RenderNoise(noise["coarse"], noise["fine_u"], noise["fine_jitter"], noise["depth"]))
    assert (two["fine"]["rgb"] - ref["fine"]["rgb"]).abs().max() > 5e-2      # the fine network would have given another image
    net.fused_render_ready = lambda: False
    staged = _render_cuda(net, rays, noise)
    assert torch.equal(staged.fine.rgb, res.fine.rgb) and torch.equal(staged.fine.depth, res.fine.depth)


def test_render_wrapper_dict_output(lib):
    """nerf.py:28-48: without simple_output the bound module returns plain dicts (what DataParallel can gather)."""
    net = H.build_net(H.make_scene_dict(), precision="bf16")
    r = _renderer()
    wrapped = r.bind_parallel(net, None, simple_output=False).eval()
    rays = H.rays_subset(1, 40).cuda()
    with torch.no_grad():
        out = wrapped(rays, want_weights=True)
        plain = wrapped(rays)
    assert type(out) is dict and set(out) == {"coarse", "fine"} and type(out["fine"]) is dict
    assert set(out["fine"]) == {"rgb", "depth", "weights"} and set(plain["fine"]) == {"rgb", "depth"}
    assert out["coarse"]["weights"].shape == (1, 40, 64) and out["fine"]["weights"].shape == (1, 40, 96)
    w = out["fine"]["weights"]
    assert (w >= 0).all() and (w.sum(-1) <= 1 + 1e-5).all()
