"""Camera gradients, the CPU half: the bookkeeping and the formulas the CUDA backward relies on.

* ``PixelNeRFNet.set_cameras`` + ``_camera_tensors`` (the per-view poses / focal / center the kernels read) keep torch's graph,
  so a gradient of the kernel's projection with respect to them reaches the caller's camera-to-world poses, focal and c exactly
  as it does through a literal transcription of the reference's ``encode`` bookkeeping (models.py:116-148) and projection
  (models.py:216-230): every focal / c format ``encode`` accepts, NeRF and YOLO mode.
* The near / far gradients of ``pnr_sample_bounds_backward`` (coarse, importance and clamped depth samples, routed through the
  merged sort by value) and the far gradient of ``pnr_composite_backward_rays`` (the last interval far - z_K), restated here as
  the kernels compute them, equal autograd over the oracle's samplers and compositing.
No reference goldens exist for camera gradients; the ground truth is autograd over the reference's formulas.
"""
import copy

import pytest
import torch

import helpers as H
from oracle import pixelnerf_oracle as O


# ------------------------------------------------------------------------------------------------ encode bookkeeping
def reference_uv(poses, focal, c, image_wh, NS, xyz, yolo):
    """models.py:116-148 (encode, minus the encoder) and models.py:168-230 (forward's projection), transcribed."""
    if not yolo:
        rot = poses[:, :3, :3].transpose(1, 2)                              # models.py:116
        trans = -torch.bmm(rot, poses[:, :3, 3:])                           # models.py:117
        w2c = torch.cat((rot, trans), dim=-1)                               # models.py:118
    else:
        w2c = poses[:, :3, :4]                                              # models.py:120
    image_shape = torch.tensor([float(image_wh[0]), float(image_wh[1])])
    if len(focal.shape) == 0:                                               # models.py:126-134
        focal = focal[None, None].repeat((1, 2))
    elif len(focal.shape) == 1:
        focal = focal.unsqueeze(-1).repeat((1, 2))
    else:
        focal = focal.clone()
    focal = focal.float()
    if not yolo:
        focal[..., 1] *= -1.0                                               # models.py:137
    if c is None:                                                           # models.py:139-148
        c = (image_shape * 0.5).unsqueeze(0)
    elif len(c.shape) == 0:
        c = c[None, None].repeat((1, 2))
    elif len(c.shape) == 1:
        c = c.unsqueeze(-1).repeat((1, 2))
    SB, P, _ = xyz.shape
    x = torch.repeat_interleave(xyz, NS, dim=0)                             # models.py:168 (util.repeat_interleave)
    x = torch.matmul(w2c[:, None, :3, :3], x.unsqueeze(-1))[..., 0] + w2c[:, None, :3, 3]
    uv = (x[:, :, :2] if yolo else -x[:, :, :2]) / x[:, :, 2:]              # models.py:220-222
    rep = lambda t: torch.repeat_interleave(t.unsqueeze(1), NS if t.shape[0] > 1 else 1, dim=0)
    return uv * rep(focal) + rep(c)                                         # models.py:225-230


def kernel_uv(poses, focal, center, NS, xyz):
    """The kernels' projection (pnr_common.cuh project_point) over the per-view tensors: uv = -x_cam.xy / x_cam.z f + c."""
    x = torch.repeat_interleave(xyz, NS, dim=0)
    x = torch.matmul(poses[:, None, :3, :3], x.unsqueeze(-1))[..., 0] + poses[:, None, :3, 3]
    return -x[:, :, :2] / x[:, :, 2:] * focal[:, None] + center[:, None]


def _net(yolo):
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.model import make_model
    conf = copy.deepcopy(H.MODEL_CONF)
    if yolo:
        conf["mlp_coarse"].update({"d_out": 7, "num_scales": 1, "num_anchors_per_scale": 3, "yolo": True})
        conf["mlp_fine"] = {"type": "empty"}
    return make_model(ConfigTree.from_dict(conf))


FORMATS = ["scalar", "per_object", "per_object_xy", "one_xy"]


def _intrinsic(fmt, SB, base, g):
    if fmt == "scalar":
        return torch.tensor(base)
    if fmt == "per_object":
        return base + torch.rand(SB, generator=g)
    if fmt == "per_object_xy":
        return base + torch.rand(SB, 2, generator=g)
    return base + torch.rand(1, 2, generator=g)


@pytest.mark.parametrize("yolo", [False, True], ids=["nerf", "yolo"])
@pytest.mark.parametrize("c_fmt", [None] + FORMATS)
@pytest.mark.parametrize("focal_fmt", FORMATS)
def test_camera_tensors_chain_like_reference_encode(focal_fmt, c_fmt, yolo):
    SB, NS, P = 2, 3, 17
    g = torch.Generator().manual_seed(FORMATS.index(focal_fmt) * 10 + (FORMATS + [None]).index(c_fmt) + 100 * yolo)
    scene = H.make_scene_dict(num_objs=SB, num_views=NS, C=64, feat=8)
    poses = scene["poses"].reshape(-1, 4, 4)
    if yolo:
        poses = torch.linalg.inv(poses)                 # YOLO mode takes world -> camera extrinsics as they are
    focal = _intrinsic(focal_fmt, SB, 131.25, g)
    c = None if c_fmt is None else _intrinsic(c_fmt, SB, 64.0, g)
    xyz = (torch.rand(SB, P, 3, generator=g) - 0.5) * 0.9
    w = torch.randn(SB * NS, P, 2, generator=g)

    def leaves():
        return [None if t is None else t.clone().requires_grad_(True) for t in (poses, focal, c)]

    ref_in = leaves()
    (reference_uv(*ref_in, scene["image_wh"], NS, xyz, yolo) * w).sum().backward()
    net = _net(yolo)
    net.num_objs, net.num_views_per_obj = SB, NS
    got_in = leaves()
    net.set_cameras(*got_in[:2], scene["image_wh"], got_in[2])
    cam_poses, cam_focal, cam_center = net._camera_tensors()[:3]
    (kernel_uv(cam_poses, cam_focal, cam_center, NS, xyz) * w).sum().backward()
    for name, a, b in zip(("poses", "focal", "c"), got_in, ref_in):
        if a is None:
            continue
        assert a.grad is not None, name
        # c's gradient is a sum of the weights: summation order alone moves it by ~1e-6 absolute
        torch.testing.assert_close(a.grad, b.grad, rtol=1e-5, atol=1e-5 * max(b.grad.abs().max().item(), 1.0), msg=name)


def test_camera_cache_rebuilt_with_graph():
    """A per-view cache built under no_grad (an inference render) is rebuilt once a camera input requires grad."""
    net = _net(False)
    scene = H.make_scene_dict(num_objs=1, num_views=2, C=64, feat=8)
    net.num_objs, net.num_views_per_obj = 1, 2
    focal = scene["focal"].clone().requires_grad_(True)
    net.set_cameras(scene["poses"].reshape(-1, 4, 4), focal, scene["image_wh"])
    with torch.no_grad():
        assert not net._camera_tensors()[1].requires_grad
    assert net._camera_tensors()[1].requires_grad


# ------------------------------------------------------------------------------------------------ ray bounds
def lerp_grads(near, far, s, lindisp):
    """d z / d near, d z / d far of z = near (1 - s) + far s, or of 1 / ((1 - s) / near + s / far) (sample_bounds_bwd_kernel)."""
    if not lindisp:
        return 1 - s, s
    z = 1 / (1 / near * (1 - s) + 1 / far * s)
    return z * z * (1 - s) / (near * near), z * z * s / (far * far)


def bounds_reference(rays, noise, Kc, lindisp, d_zc, z_sorted=None, d_sorted=None, z_coarse=None, inds=None, jitter=None,
                     depth=None, gauss=None, depth_std=0.0):
    """sample_bounds_bwd_kernel restated: -> (d near, d far) per ray and, for the fine pass, d z_coarse."""
    near, far = rays[:, 6:7], rays[:, 7:8]
    if z_sorted is None:
        s = torch.linspace(0, 1 - 1.0 / Kc, Kc)[None] + noise * (1.0 / Kc)
        a, b = lerp_grads(near, far, s, lindisp)
        return (d_zc * a).sum(1), (d_zc * b).sum(1), None
    B = rays.shape[0]
    dn, df = torch.zeros(B), torch.zeros(B)
    dzc = torch.zeros_like(z_coarse)
    for b in range(B):
        vals = list(z_coarse[b])
        srcs = [("c", k) for k in range(Kc)]
        if inds is not None:
            s_f = (inds[b].float() + jitter[b]) / Kc
            zf = near[b] * (1 - s_f) + far[b] * s_f if not lindisp else 1 / (1 / near[b] * (1 - s_f) + 1 / far[b] * s_f)
            vals += list(zf)
            srcs += [("f", s) for s in s_f]
        if depth is not None:
            raw = depth[b] + gauss[b] * depth_std
            vals += list(torch.clamp(raw, near[b].item(), far[b].item()))
            srcs += [("d", r) for r in raw]
        zs = z_sorted[b]
        for ci, (v, (kind, arg)) in enumerate(zip(vals, srcs)):
            pos = int(torch.searchsorted(zs, v.reshape(1)).item()) + sum(1 for cc in range(ci) if vals[cc] == v)
            gz = d_sorted[b, pos]
            if kind == "c":
                dzc[b, arg] = gz
            elif kind == "f":
                a_, b_ = lerp_grads(near[b], far[b], arg, lindisp)
                dn[b] += gz * a_.reshape(-1)[0]
                df[b] += gz * b_.reshape(-1)[0]
            elif arg <= near[b]:
                dn[b] += gz
            elif arg >= far[b]:
                df[b] += gz
    return dn, df, dzc


@pytest.mark.parametrize("lindisp", [False, True])
def test_coarse_bounds_match_autograd(lindisp):
    B, Kc = 37, 24
    g = torch.Generator().manual_seed(3)
    rays = H.rays_subset(1, B)[0].clone().requires_grad_(True)
    noise = torch.rand(B, Kc, generator=g)
    d_z = torch.randn(B, Kc, generator=g)
    (O.sample_coarse(rays, noise, Kc, lindisp) * d_z).sum().backward()
    dn, df, _ = bounds_reference(rays.detach(), noise, Kc, lindisp, d_z)
    torch.testing.assert_close(dn, rays.grad[:, 6], rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(df, rays.grad[:, 7], rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("lindisp", [False, True])
def test_fine_bounds_match_autograd(lindisp):
    """Importance samples (piecewise-constant bins over detached weights), depth samples clamped at both bounds (a wide
    depth_std), all merged and sorted with the coarse depths: near / far and the coarse depths' share of the gradient."""
    B, Kc, Kf, Kfd, std = 29, 16, 8, 8, 0.6
    g = torch.Generator().manual_seed(4)
    r0 = H.rays_subset(1, B)[0]
    zc0 = O.sample_coarse(r0, torch.rand(B, Kc, generator=g), Kc, lindisp)
    w = torch.rand(B, Kc, generator=g)
    u, jit = torch.rand(B, Kf, generator=g), torch.rand(B, Kf, generator=g)
    gauss = torch.randn(B, Kfd, generator=g)
    depth0 = 1.3 + 0.2 * torch.randn(B, generator=g)
    d_sorted = torch.randn(B, Kc + Kf + Kfd, generator=g)
    rays, zc, depth = r0.clone().requires_grad_(True), zc0.clone().requires_grad_(True), depth0.clone().requires_grad_(True)
    zf, inds = O.sample_fine(rays, w, u, jit, Kc, lindisp, return_inds=True)
    zd = O.sample_fine_depth(rays, depth, gauss, std)
    z_sorted, _ = torch.sort(torch.cat((zc, zf, zd), dim=-1), dim=-1)
    (z_sorted * d_sorted).sum().backward()
    raw = depth0[:, None] + gauss * std
    assert (raw < r0[:, 6:7]).any() and (raw > r0[:, 7:8]).any()          # both clamps occur
    dn, df, dzc = bounds_reference(r0, None, Kc, lindisp, None, z_sorted.detach(), d_sorted, zc0, inds, jit, depth0, gauss, std)
    torch.testing.assert_close(dn, rays.grad[:, 6], rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(df, rays.grad[:, 7], rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(dzc, zc.grad, rtol=0, atol=0)


@pytest.mark.parametrize("white", [False, True])
def test_composite_far_matches_autograd(white):
    """d far of the compositing = d(last interval) = d alpha_K relu(sigma_K) (1 - alpha_K), d alpha_K = d w_K T_K (the
    composite_bwd_kernel terms of the last sample)."""
    B, K = 31, 20
    g = torch.Generator().manual_seed(5)
    rays = H.rays_subset(1, B)[0].clone().requires_grad_(True)
    z, _ = torch.sort(0.8 + torch.rand(B, K, generator=g), dim=-1)
    out = torch.cat((torch.rand(B, K, 3, generator=g), 30 * torch.rand(B, K, 1, generator=g) ** 3 - 1.0), dim=-1)
    gw, grgb, gd = torch.randn(B, K, generator=g), torch.randn(B, 3, generator=g), torch.randn(B, generator=g)
    w, rgb, depth = O.alpha_composite(out, z, rays, white)
    ((w * gw).sum() + (rgb * grgb).sum() + (depth * gd).sum()).backward()
    with torch.no_grad():
        deltas = torch.cat((z[:, 1:] - z[:, :-1], rays[:, 7:8] - z[:, -1:]), dim=-1)
        alphas = 1 - torch.exp(-deltas * torch.relu(out[..., 3]))
        T = torch.cumprod(1 - alphas[:, :-1] + 1e-10, dim=-1)[:, -1]
        sig, alpha = torch.relu(out[:, -1, 3]), alphas[:, -1]
        dw = (grgb * out[:, -1, :3]).sum(1) + gd * z[:, -1] + gw[:, -1] - (grgb.sum(1) if white else 0)
        d_far = dw * T * sig * (1 - alpha)
    torch.testing.assert_close(d_far, rays.grad[:, 7], rtol=1e-4, atol=1e-6)
