"""Camera gradients on the training path (`-m gpu`): source poses, focal lengths, principal points, view directions and rays.

Ground truth is autograd over the oracle with the camera tensors requiring grad: ``tests/zfeature_oracle.py``'s field (the
golden-pinned oracle with the switched z-feature) for one field call, ``O.render`` / ``O.yolo_render`` for the renders.  The
network's parameters and the maps are frozen, so each call records its backward pass because a camera input requires grad.
Bounds are relative errors in norm per tensor:
* fp32 arithmetic, 3e-3 against the fp32 oracle (the position derivative of a bilinear tap is piecewise constant, so a last-bit
  difference of a tap position may move a row's term, as in the depth-loss case of tests/test_gpu_train.py);
* tcgen05 bf16 arithmetic, 3e-2 against the oracle's bf16-operand emulation (``emulate_bf16``);
* TF32 arithmetic, 3e-2 against the fp32 oracle.  (Against the bf16 emulation TF32 differs by what bf16 rounding moves: up to
  1.4e-1 measured on a B200, where TF32 against the fp32 oracle is the comparison of like with like.)  With 1 792-channel
  latents, 1.5e-1: d focal = sum over rows of d u (-x / z), where d u is a 1 792-long product of TF32-rounded gradients with tap
  differences and the row terms have both signs; measured 9.8e-2 on a B200 for focal (poses 1.8e-2, c 1.4e-2), while the same
  case is at 2.8e-6 on fp32 arithmetic.
"""
import copy

import pytest
import torch

import helpers as H
import pixel_nerf_yolo_b200.synth as synth
import pooling_oracle as PO
import zfeature_oracle as ZO
from oracle import pixelnerf_oracle as O
from test_oracle_zfeature import DEFAULT

pytestmark = pytest.mark.gpu

FF = 1.5
SHAPE = dict(d_hidden=128, n_blocks=3, combine_layer=2)
BOUND = {"fp32": 3e-3, "tf32": 3e-2, "bf16": 3e-2}
LAYOUTS = {
    "default": DEFAULT,
    "cam_coords": dict(DEFAULT, normalize_z=False),
    "z_only": dict(DEFAULT, use_xyz=False),
    "code_viewdirs": dict(DEFAULT, use_xyz=False, use_code_viewdirs=True),
    "no_viewdirs": dict(DEFAULT, use_viewdirs=False),
    "yolo": dict(DEFAULT, use_viewdirs=False, normalize_z=False, use_xyz=False),
}


@pytest.fixture(scope="module")
def lib():
    from pixel_nerf_yolo_b200 import _lib
    assert torch.cuda.is_available()
    _lib.require_device(torch.device("cuda", 0))
    return _lib.load()


def rel_err(got, ref):
    got, ref = got.detach().cpu().double(), ref.detach().cpu().double()
    return ((got - ref).norm() / ref.norm().clamp_min(1e-30)).item()


class Case:
    """A frozen PixelNeRFNet (layout ``sw`` at 6 frequencies, C-channel latent, SB objects x NS views) whose cameras are given
    as leaves that require grad: camera-to-world poses (world-to-camera in YOLO mode), focal and c in the format ``fmt``."""

    def __init__(self, sw, sb, ns, C=64, combine_type="average", yolo=False, fmt="scalar"):
        from pixel_nerf_yolo_b200.conf import ConfigTree
        from pixel_nerf_yolo_b200.model import make_model
        from pixel_nerf_yolo_b200.model.model_util import make_mlp
        self.scene = H.make_scene_dict(num_objs=sb, num_views=ns, C=C, feat=16)
        conf = copy.deepcopy(H.MODEL_CONF)
        conf.update({k: v for k, v in sw.items() if k != "include_input"})
        conf["code"] = {"num_freqs": 6, "freq_factor": FF, "include_input": sw["include_input"]}
        conf["mlp_coarse"].update(combine_type=combine_type, **SHAPE)
        conf["mlp_fine"] = {"type": "empty"}
        if yolo:
            conf["mlp_coarse"].update({"d_out": 7, "num_scales": 1, "num_anchors_per_scale": 3, "yolo": True})
        conf = ConfigTree.from_dict(conf)
        net = make_model(conf).eval()
        net.mlp_coarse = make_mlp(conf["mlp_coarse"], net.d_in, C)
        net.d_latent = net.latent_size = C
        self.state = synth.mlp_state(1, d_in=net.d_in, d_latent=C, d_out=21 if yolo else 4, **SHAPE)
        net.mlp_coarse.load_state_dict(self.state)
        net = net.cuda().requires_grad_(False)
        net.num_objs, net.num_views_per_obj = sb, ns
        net.encoder.set_latent(self.scene["latent"].cuda())
        cams = self.scene["poses"].reshape(-1, 4, 4)
        if yolo:
            cams = torch.linalg.inv(cams)
        g = torch.Generator().manual_seed(sb * 10 + ns)
        size = self.scene["image_wh"][0]
        if fmt == "scalar":
            focal, c = torch.tensor(131.25), torch.tensor(0.5 * size + 1.5)
        else:                                   # per object, (SB, 2)
            focal = 131.25 + torch.rand(sb, 2, generator=g)
            c = 0.5 * size + torch.rand(sb, 2, generator=g) - 0.5
        self.cams = (cams, focal, c)
        self.net, self.sw, self.sb, self.ns, self.yolo, self.combine_type = net, sw, sb, ns, yolo, combine_type

    def leaves(self, device=None):
        return [t.clone().to(device).requires_grad_(True) for t in self.cams]

    def field(self, precision, xyz, dirs, gout):
        """One PixelNeRFNet.forward on the training path: (out, grads of poses, focal, c, viewdirs)."""
        poses, focal, c = self.leaves("cuda")
        self.net.set_cameras(poses, focal, self.scene["image_wh"], c)
        self.net.train_precision = precision
        d = dirs.cuda().requires_grad_(True) if self.sw["use_viewdirs"] else None
        out = self.net(xyz.cuda(), coarse=True, viewdirs=d)
        (out * gout.cuda()).sum().backward()
        return out.detach().cpu(), (poses.grad, focal.grad, c.grad, None if d is None else d.grad)

    def oracle(self, xyz, dirs, gout, emulate_bf16):
        poses, focal, c = self.leaves()
        sc = O.encode_cameras(self.scene["latent"], poses.reshape(self.sb, self.ns, 4, 4), focal, self.scene["image_wh"], c,
                              yolo=self.yolo)
        d = dirs.clone().requires_grad_(True) if self.sw["use_viewdirs"] else None
        with PO.combine_type(self.combine_type):
            out = ZO.field_forward(sc, self.state, xyz, d, yolo=self.yolo, emulate_bf16=emulate_bf16, num_freqs=6,
                                   freq_factor=FF, n_blocks=SHAPE["n_blocks"], combine_layer=SHAPE["combine_layer"], **self.sw)
        (out * gout).sum().backward()
        return out.detach(), (poses.grad, focal.grad, c.grad, None if d is None else d.grad)


FIELD_CASES = {
    "default-sb1-ns1": dict(sw="default", sb=1, ns=1),
    "default-sb1-ns3": dict(sw="default", sb=1, ns=3),
    "default-sb2-ns3-max-per_object": dict(sw="default", sb=2, ns=3, combine_type="max", fmt="per_object"),
    "cam_coords-sb2-ns8": dict(sw="cam_coords", sb=2, ns=8),
    "z_only-sb1-ns3-max": dict(sw="z_only", sb=1, ns=3, combine_type="max"),
    "code_viewdirs-sb2-ns3-per_object": dict(sw="code_viewdirs", sb=2, ns=3, fmt="per_object"),
    "no_viewdirs-sb1-ns8": dict(sw="no_viewdirs", sb=1, ns=8),
    "default-C1792-sb1-ns3": dict(sw="default", sb=1, ns=3, C=1792),
    "yolo-sb1-ns3": dict(sw="yolo", sb=1, ns=3, yolo=True),
}


@pytest.mark.parametrize("precision", ["fp32", "tf32", "bf16"])
@pytest.mark.parametrize("case", list(FIELD_CASES))
def test_field_camera_grads(lib, case, precision):
    kw = dict(FIELD_CASES[case])
    kw["sw"] = LAYOUTS[kw["sw"]]
    m = Case(**kw)
    P = 160
    g = torch.Generator().manual_seed(P + m.ns)
    xyz = (torch.rand(m.sb, P, 3, generator=g) - 0.5) * (3.2 if m.yolo else 0.9)
    dirs = torch.nn.functional.normalize(torch.randn(m.sb, P, 3, generator=g), dim=-1)
    gout = torch.randn(m.sb, P, 21 if m.yolo else 4, generator=g)
    out, got = m.field(precision, xyz, dirs, gout)
    ref_out, ref = m.oracle(xyz, dirs, gout, emulate_bf16=precision == "bf16")
    errs = {name: rel_err(a, b) for name, a, b in zip(("poses", "focal", "c", "viewdirs"), got, ref) if b is not None}
    print(f"\nCAMGRAD {case} {precision}: " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    if m.yolo:
        nonneg = torch.stack([(p[:3, :3] @ xyz[i // m.ns].T + p[:3, 3:]).T[:, 2] >= 0 for i, p in enumerate(m.cams[0])])
        assert nonneg.any() and not nonneg.all()             # masked and unmasked rows both occur
    assert m.net.last_bwd_launches > 0
    bound = 1.5e-1 if (precision == "tf32" and kw.get("C", 64) == 1792) else BOUND[precision]
    for name, e in errs.items():
        assert e <= bound, (case, precision, name, e)


# ------------------------------------------------------------------------------------------------ renders
def _renderer(**kw):
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.render import NeRFRenderer
    conf = dict(H.RENDER_CONF)
    conf.update(kw)
    lindisp = conf.pop("lindisp", False)
    return NeRFRenderer.from_conf(ConfigTree.from_dict(conf), lindisp=lindisp).cuda()


RENDER_CASES = {
    "coarse": dict(n_fine=0, n_fine_depth=0),
    "coarse-lindisp-black": dict(n_fine=0, n_fine_depth=0, lindisp=True, white_bkgd=False),
    "fine-depth": dict(),
    "fine-depth-lindisp-black": dict(lindisp=True, white_bkgd=False),
}


@pytest.mark.parametrize("case", list(RENDER_CASES))
def test_render_ray_grads(lib, case):
    """NeRFRenderer on the training path with the rays requiring grad (network frozen): origin, direction, near and far
    against autograd over ``O.render``.  depth_std = 0.5 puts depth samples beyond both bounds, where they clamp."""
    kw = dict(RENDER_CASES[case], depth_std=0.5)
    B = 64
    scene = H.make_scene_dict(num_objs=2, num_views=3, feat=16)
    net = H.build_net(scene, precision="bf16")
    net.train_precision = "fp32"
    r = _renderer(**kw)
    kc, kf, kfd = r.n_coarse, r.n_fine - r.n_fine_depth, r.n_fine_depth
    rays = H.rays_subset(2, B, seed=11)
    noise = H.make_noise(2 * B, seed=12, kc=kc, kf=max(kf, 1), kfd=max(kfd, 1))
    r.noise_override = {k: v.cuda() for k, v in noise.items()}
    g = torch.Generator().manual_seed(13)
    grgb, gdep = torch.randn(2, B, 3, generator=g), torch.randn(2, B, generator=g)
    rc = rays.cuda().requires_grad_(True)
    res = r(net, rc)
    lvls = ("coarse", "fine") if r.using_fine else ("coarse",)
    sum((res[lv].rgb * grgb.cuda()).sum() + (res[lv].depth * gdep.cuda()).sum() for lv in lvls).backward()
    ro = rays.clone().requires_grad_(True)
    n = O.RenderNoise(noise["coarse"], noise["fine_u"], noise["fine_jitter"], noise["depth"])
    ref = O.render(H.oracle_scene(scene), synth.mlp_state(1), synth.mlp_state(2), ro, n, n_coarse=kc, n_fine=r.n_fine,
                   n_fine_depth=kfd, depth_std=0.5, white_bkgd=r.white_bkgd, lindisp=r.lindisp, grad=True)
    sum((ref[lv]["rgb"] * grgb).sum() + (ref[lv]["depth"] * gdep).sum() for lv in lvls).backward()
    if r.using_fine:
        near, far = rays[..., 6:7], rays[..., 7:8]
        raw = ref["coarse"]["depth"].detach()[..., None] + noise["depth"].reshape(2, B, -1) * 0.5
        assert (raw < near).any() and (raw > far).any()
    errs = {name: rel_err(rc.grad[..., sl], ro.grad[..., sl]) for name, sl in
            (("origin", slice(0, 3)), ("direction", slice(3, 6)), ("near", slice(6, 7)), ("far", slice(7, 8)))}
    print(f"\nRAYGRAD {case}: " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    for name, e in errs.items():
        assert e <= 1e-2, (case, name, e)


def test_yolo_render_ray_grads(lib):
    """YoloRenderer on the training path with the rays requiring grad: coarse samples only."""
    from pixel_nerf_yolo_b200.render import YoloRenderer
    m = Case(LAYOUTS["yolo"], 1, 3, yolo=True)
    m.net.set_cameras(m.cams[0].cuda(), m.cams[1].cuda(), m.scene["image_wh"], m.cams[2].cuda())
    m.net.train_precision = "fp32"
    B, Kc = 48, 32
    rays = H.rays_subset(1, B, seed=21)[0].contiguous()
    noise = torch.rand(rays.shape[0], Kc, generator=torch.Generator().manual_seed(3))
    r = YoloRenderer(Kc, 1024, 1, 3)
    r.bind_net(m.net)
    r.noise_override = noise.cuda()
    gres = torch.randn(rays.shape[0], 3, 7, generator=torch.Generator().manual_seed(4))
    rc = rays.cuda().requires_grad_(True)
    (r(rc) * gres.cuda()).sum().backward()
    sc = O.encode_cameras(m.scene["latent"], m.cams[0].reshape(1, 3, 4, 4), m.cams[1], m.scene["image_wh"], m.cams[2],
                          yolo=True)
    ro = rays.clone().requires_grad_(True)
    with ZO.switched(num_freqs=6, freq_factor=FF, **m.sw):
        ref = O.yolo_render(sc, m.state, ro, noise, n_coarse=Kc, num_anchors=3, grad=True, n_blocks=SHAPE["n_blocks"],
                            combine_layer=SHAPE["combine_layer"])
    (ref * gres).sum().backward()
    errs = {name: rel_err(rc.grad[:, sl], ro.grad[:, sl]) for name, sl in
            (("origin", slice(0, 3)), ("direction", slice(3, 6)), ("near", slice(6, 7)), ("far", slice(7, 8)))}
    print("\nYOLO RAYGRAD " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    for name, e in errs.items():
        assert e <= 1e-2, (name, e)


def test_config3_step_with_source_pose_grads(lib):
    """A config-3-shaped training step (4 objects x 128 rays, 3 source views, 64 + 32 samples, both networks and the maps
    training, tcgen05 arithmetic) with the source camera-to-world poses requiring grad: the pose gradient against autograd
    over the oracle's render with the bf16-operand emulation, and the parameter gradients against the same step without
    camera gradients."""
    import numpy as np
    scene = H.make_scene_dict(num_objs=4, num_views=3, feat=32)
    rays = H.rays_subset(4, 128, seed=1)
    noise = H.make_noise(512, seed=2)
    gt = torch.rand(4, 128, 3, generator=torch.Generator().manual_seed(3))

    def step(pose_grad):
        net = H.build_net(scene, precision="bf16", train=True)
        net.train_precision = "bf16"
        poses = scene["poses"].reshape(-1, 4, 4).cuda().requires_grad_(pose_grad)
        net.set_cameras(poses, scene["focal"].cuda(), scene["image_wh"])
        r = _renderer().train()
        r.noise_override = {k: v.cuda() for k, v in noise.items()}
        res = r(net, rays.cuda())
        loss = ((res.coarse.rgb - gt.cuda()) ** 2).mean() + ((res.fine.rgb - gt.cuda()) ** 2).mean()
        net.last_bwd_launches = 0
        loss.backward()
        grads = {n: p.grad.detach().clone() for n, p in net.named_parameters() if p.grad is not None}
        return poses.grad, grads, (net.last_launches, net.last_bwd_launches)

    d_poses, grads_cam, launches_cam = step(True)
    _, grads_a, launches_a = step(False)
    assert launches_cam[0] == launches_a[0]                 # the forward is the same sequence
    ref_poses = scene["poses"].reshape(-1, 4, 4).clone().requires_grad_(True)
    sc = O.encode_cameras(scene["latent"], ref_poses.reshape(4, 3, 4, 4), scene["focal"], scene["image_wh"])
    n = O.RenderNoise(noise["coarse"], noise["fine_u"], noise["fine_jitter"], noise["depth"])
    ref = O.render(sc, synth.mlp_state(1), synth.mlp_state(2), rays, n, grad=True, emulate_bf16=True)
    loss = ((ref["coarse"]["rgb"] - gt) ** 2).mean() + ((ref["fine"]["rgb"] - gt) ** 2).mean()
    loss.backward()
    e = rel_err(d_poses, ref_poses.grad)
    print(f"\nCONFIG3 pose grad rel-norm err {e:.2e}")
    assert e <= BOUND["bf16"], e
    for name in grads_a:          # parameter gradients with and without the pose input: same within bf16 accumulation order
        np.testing.assert_allclose(grads_cam[name].cpu().numpy(), grads_a[name].cpu().numpy(),
                                   atol=1e-3 * grads_a[name].abs().max().item() + 1e-12, rtol=0)
