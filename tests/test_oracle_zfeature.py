"""PixelNeRFNet's z-feature switches on the CPU: use_viewdirs, use_code_viewdirs, normalize_z, use_xyz, use_code and
code.include_input.

The z-feature is the non-latent part of each MLP input row.  For every combination of the six switches this checks the width
(``d_in``), the ``code`` module and the state_dict the drop-in builds against the reference's rule (models.py:16-90), the width
the C library computes from the scene flags (``pnr_zfeat_width``), and the z-feature the oracle feeds its ResnetFC against a
literal transcription of models.py:183-209 (tests/zfeature_oracle.py, which with the default switches is the golden-pinned
oracle bit for bit).  The GPU side is tests/test_gpu_zfeature.py.
"""
import copy
import itertools

import pytest
import torch

import helpers as H
import pixel_nerf_yolo_b200.synth as synth
import zfeature_oracle as ZO
from oracle import pixelnerf_oracle as O

SWITCHES = ("use_viewdirs", "use_code_viewdirs", "normalize_z", "use_xyz", "use_code", "include_input")
COMBOS = [dict(zip(SWITCHES, v)) for v in itertools.product((True, False), repeat=len(SWITCHES))]
DEFAULT = ZO.DEFAULT


def combo_id(sw):
    return "-".join(k for k in SWITCHES if sw[k]) or "none"


def reference_d_in(sw, num_freqs):
    """models.py:16-90, restated: (d_in, width of the code module's input or None)."""
    d_in = 3 if sw["use_xyz"] else 1
    if sw["use_viewdirs"] and sw["use_code_viewdirs"]:
        d_in += 3
    code_in = None
    if sw["use_code"] and d_in > 0:
        code_in = d_in
        d_in = d_in * (2 * num_freqs + (1 if sw["include_input"] else 0))
    if sw["use_viewdirs"] and not sw["use_code_viewdirs"]:
        d_in += 3
    return d_in, code_in


def model_conf(sw, num_freqs=6, d_hidden=64):
    conf = copy.deepcopy(H.MODEL_CONF)
    conf.update({k: v for k, v in sw.items() if k != "include_input"})
    conf["code"] = {"num_freqs": num_freqs, "freq_factor": 1.5, "include_input": sw["include_input"]}
    conf["encoder"]["backbone"] = "resnet18"
    for k in ("mlp_coarse", "mlp_fine"):
        conf[k].update(d_hidden=d_hidden, n_blocks=2, combine_layer=1)
    return conf


def make(sw, num_freqs=6):
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.model import make_model
    return make_model(ConfigTree.from_dict(model_conf(sw, num_freqs)))


@pytest.fixture(scope="module")
def lib():
    from pixel_nerf_yolo_b200 import _lib, build
    build.build()
    return _lib.load()


@pytest.mark.parametrize("num_freqs", [4, 6, 9])
@pytest.mark.parametrize("sw", COMBOS, ids=combo_id)
def test_width_code_and_state_dict(lib, sw, num_freqs):
    """d_in, the presence of ``code`` and the state_dict names and shapes follow the reference; the C library's width of the
    scene flags equals d_in; a z-feature wider than one K = 64 slab is refused at construction, naming d_in and the limit."""
    d_in, code_in = reference_d_in(sw, num_freqs)
    if d_in > 64:
        with pytest.raises(NotImplementedError, match=f"d_in={d_in} .*at most 64"):
            make(sw, num_freqs)
        return
    net = make(sw, num_freqs)
    assert net.d_in == d_in
    assert lib.pnr_zfeat_width(net.zf_flags, num_freqs) == d_in
    sd = net.state_dict()
    assert hasattr(net, "code") == (code_in is not None)
    assert ("code._freqs" in sd) == ("code._phases" in sd) == (code_in is not None)
    if code_in is not None:
        assert net.code.d_in == code_in and net.code.d_out == d_in - (3 if sw["use_viewdirs"] and not sw["use_code_viewdirs"] else 0)
        assert tuple(sd["code._freqs"].shape) == (1, 2 * num_freqs, 1) and tuple(sd["code._phases"].shape) == (1, 2 * num_freqs, 1)
        assert net.code_args() == (num_freqs, 1.5)
    else:
        assert net.code_args() == (0, 0.0)
    for mlp in ("mlp_coarse", "mlp_fine"):
        state = synth.mlp_state(0, d_in=d_in, d_hidden=64, n_blocks=2, combine_layer=1)
        for k, v in state.items():
            assert tuple(sd[f"{mlp}.{k}"].shape) == tuple(v.shape), (mlp, k)
    # load_state_dict(strict=True) works both ways with a state of the same switches, and not across the use_code boundary
    net.load_state_dict(copy.deepcopy(sd), strict=True)
    other = make({**sw, "use_code": not sw["use_code"]}, num_freqs) if reference_d_in({**sw, "use_code": not sw["use_code"]},
                                                                                      num_freqs)[0] <= 64 else None
    if other is not None:
        with pytest.raises(RuntimeError):
            other.load_state_dict(sd, strict=True)


def test_flag_bits_are_the_header_values(lib):
    from pixel_nerf_yolo_b200 import _lib
    import os
    import re
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "pixelnerf_b200.h")).read()
    for name in ("NO_VIEWDIRS", "CODE_VIEWDIRS", "CAM_COORDS", "Z_ONLY", "NO_CODE", "NO_CODE_INPUT"):
        value = int(re.search(rf"#define PNR_SCENE_ZF_{name} (\d+)", header).group(1))
        assert getattr(_lib, f"SCENE_ZF_{name}") == value, name
    assert lib.pnr_zfeat_width(0, 6) == 42 and lib.pnr_zfeat_width(0, 9) == 60


@pytest.mark.parametrize("what,conf", [("use_encoder=False", {"use_encoder": False}),
                                       ("use_global_encoder=True", {"use_global_encoder": True})])
def test_unbuilt_networks_are_refused(what, conf):
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.model import make_model
    c = model_conf(DEFAULT)
    c.update(conf)
    with pytest.raises(NotImplementedError, match=what):
        make_model(ConfigTree.from_dict(c))


def test_refusal_example_from_the_switches():
    """use_code_viewdirs with use_xyz at 6 frequencies: PE of 6 values, 78 wide."""
    with pytest.raises(NotImplementedError, match="d_in=78 .*at most 64"):
        make({**DEFAULT, "use_code_viewdirs": True})


# ------------------------------------------------------------------------------------------------ the oracle's z-feature
def _scene_points(num_views=2, P=37, seed=11):
    scene = H.make_scene_dict(num_views=num_views, C=64, feat=8)
    sc = H.oracle_scene(scene)
    g = torch.Generator().manual_seed(seed)
    xyz = (torch.rand(1, P, 3, generator=g) - 0.5) * 0.9
    dirs = torch.nn.functional.normalize(torch.randn(1, P, 3, generator=g), dim=-1)
    return sc, xyz, dirs


def transcribed_zfeature(sc, xyz, dirs, sw, num_freqs, freq_factor):
    """models.py:183-209 written out, one view at a time: x_rot = R x, x_cam = R x + t."""
    rows = []
    for v in range(sc.poses.shape[0]):
        R, t = sc.poses[v, :, :3], sc.poses[v, :, 3]
        x_rot = (R @ xyz[0].unsqueeze(-1))[..., 0]
        x_cam = x_rot + t
        code = lambda x: O.positional_encoding(x, num_freqs, freq_factor, sw["include_input"])
        if sw["use_xyz"]:
            zf = x_rot if sw["normalize_z"] else x_cam
        else:
            zf = -(x_rot if sw["normalize_z"] else x_cam)[..., 2:3]
        if sw["use_code"] and not sw["use_code_viewdirs"]:
            zf = code(zf)
        if sw["use_viewdirs"]:
            zf = torch.cat((zf, (R @ dirs[0].unsqueeze(-1))[..., 0]), dim=1)
        if sw["use_code"] and sw["use_code_viewdirs"]:
            zf = code(zf)
        rows.append(zf)
    return torch.cat(rows)


def oracle_zfeature(sc, mlp, xyz, dirs, C, **kw):
    """The z-feature columns of the MLP input ``zfeature_oracle.field_forward(sc, mlp, xyz, dirs, **kw)`` builds."""
    seen = {}
    saved = O.resnetfc_forward

    def spy(p, zx, *a, **k):
        seen["zx"] = zx.detach().clone()
        return saved(p, zx, *a, **k)
    O.resnetfc_forward = spy
    try:
        ZO.field_forward(sc, mlp, xyz, dirs, **kw)
    finally:
        O.resnetfc_forward = saved
    return seen["zx"][:, C:]


@pytest.mark.parametrize("num_freqs", [4, 6, 9])
@pytest.mark.parametrize("sw", COMBOS, ids=combo_id)
def test_oracle_zfeature_is_the_transcription(sw, num_freqs):
    d_in, _ = reference_d_in(sw, num_freqs)
    sc, xyz, dirs = _scene_points()
    mlp = synth.mlp_state(3, d_in=d_in, d_latent=64, d_hidden=64, n_blocks=2, combine_layer=1)
    zf = oracle_zfeature(sc, mlp, xyz, dirs if sw["use_viewdirs"] else None, 64, n_blocks=2, combine_layer=1, num_freqs=num_freqs,
                         freq_factor=1.5, **sw)
    want = transcribed_zfeature(sc, xyz, dirs, sw, num_freqs, 1.5)
    assert zf.shape == (2 * 37, d_in)
    assert torch.equal(zf, want)


@pytest.mark.parametrize("yolo", [False, True])
def test_switched_oracle_defaults_are_the_oracle(yolo):
    """With the default switches the switched restatement is the golden-pinned oracle bit for bit, and both are the layout
    [PE(R x), R d] written out."""
    sc, xyz, dirs = _scene_points(num_views=3, P=53)
    mlp = synth.mlp_state(4, d_in=42, d_latent=64, d_hidden=64, n_blocks=2, combine_layer=1)
    out = O.field_forward(sc, mlp, xyz, dirs, n_blocks=2, combine_layer=1, yolo=yolo)
    assert torch.equal(out, ZO.field_forward(sc, mlp, xyz, dirs, n_blocks=2, combine_layer=1, yolo=yolo))
    assert torch.equal(out, ZO.field_forward(sc, mlp, xyz, dirs, n_blocks=2, combine_layer=1, yolo=yolo, **DEFAULT))
    if yolo:
        return
    # the pre-switch construction, written out
    NS, P = 3, 53
    R = sc.poses[:, None, :3, :3]
    x_rot = torch.matmul(R, xyz.expand(NS, P, 3).unsqueeze(-1))[..., 0]
    x_cam = x_rot + sc.poses[:, None, :3, 3]
    zf = torch.cat((O.positional_encoding(x_rot.reshape(-1, 3), 6, 1.5),
                    torch.matmul(R, dirs.expand(NS, P, 3).unsqueeze(-1)).reshape(-1, 3)), dim=1)
    uv = -x_cam[:, :, :2] / x_cam[:, :, 2:] * sc.focal.unsqueeze(1) + sc.c.unsqueeze(1)
    lat = O.bilinear_index(sc.latent, uv, sc.latent_scaling, sc.image_shape).transpose(1, 2).reshape(-1, 64)
    raw = O.resnetfc_forward(mlp, torch.cat((lat, zf), dim=-1), 64, 2, 1, (NS, P)).reshape(1, P, 4)
    ref = torch.cat((O._f64(torch.sigmoid, raw[..., :3]), torch.relu(raw[..., 3:4])), dim=-1)
    assert torch.equal(out, ref)
    assert torch.equal(oracle_zfeature(sc, mlp, xyz, dirs, 64, n_blocks=2, combine_layer=1), zf)


def test_bf16_reference_runs_the_switched_network():
    """Inside ``zfeature_oracle.switched`` the oracle's callers run the switched network: bf16_field_reference with rounding
    off is the switched oracle, and O.field_forward is the golden-pinned one again afterwards."""
    import bf16_field_reference as BR
    sw = dict(use_viewdirs=False, use_code_viewdirs=False, normalize_z=False, use_xyz=False, use_code=True, include_input=False)
    d_in, _ = reference_d_in(sw, 4)
    sc, xyz, dirs = _scene_points()
    mlp = synth.mlp_state(5, d_in=d_in, d_latent=64, d_hidden=64, n_blocks=2, combine_layer=1)
    zkw = dict(num_freqs=4, freq_factor=1.5, **sw)
    with ZO.switched(**zkw):
        a = BR.field_forward_bf16(sc, mlp, xyz, None, rounding=False, projected=False, n_blocks=2, combine_layer=1)
        b = BR.field_forward_bf16(sc, mlp, xyz, None, projected=False, n_blocks=2, combine_layer=1)
    assert torch.equal(a, ZO.field_forward(sc, mlp, xyz, None, n_blocks=2, combine_layer=1, **zkw))
    assert not torch.equal(a, b)
    assert O.field_forward is ZO._field_forward
