"""CPU-side tests: config parsing, C-ABI surface, sharding host logic (gloo, world_size 2), API shape."""
import ctypes
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_hocon_subset_parser(tmp_path):
    from pixel_nerf_yolo_b200 import conf
    (tmp_path / "base.conf").write_text(
        "# comment\nmodel {\n  use_xyz = True  # trailing\n  code { num_freqs = 6\n freq_factor = 1.5 }\n"
        "  mlp_coarse { type = resnet\n n_blocks = 3 }\n}\nrenderer { sched = []\n white_bkgd = True }\n")
    (tmp_path / "exp").mkdir()
    (tmp_path / "exp" / "child.conf").write_text(
        'include required("../base.conf")\nmodel {\n mlp_coarse{\n n_blocks = 5\n combine_layer = 3 }\n}\n'
        "yolo { anchors = [\n [[0.02, 0.03], [0.04, 0.07]],\n [[0.07, 0.15], [0.15, 0.11]]\n ]\n scale = [0.5, 0.47407] }\n")
    c = conf.parse_file(str(tmp_path / "exp" / "child.conf"))
    assert c["model.mlp_coarse.n_blocks"] == 5 and c["model"]["mlp_coarse"].get_string("type") == "resnet"
    assert c.get_int("model.mlp_coarse.combine_layer") == 3 and c["model"].get_bool("use_xyz") is True
    assert c["model.code"].get_float("freq_factor") == 1.5 and c.get_list("renderer.sched") == []
    assert c["yolo.anchors"][1][0] == [0.07, 0.15] and c["yolo"].get_list("scale") == [0.5, 0.47407]
    assert "model.mlp_fine" not in c and c.get_int("model.missing", 7) == 7


def test_dotmap_contract():
    from pixel_nerf_yolo_b200.conf import DotMap
    d = DotMap(coarse=DotMap(rgb=1))
    assert len(d.fine) == 0 and d.coarse.rgb == 1 and d.toDict() == {"coarse": {"rgb": 1}, "fine": {}}


def test_library_exports_every_declared_symbol():
    """The C-ABI library loads (no GPU needed) and exports exactly what include/pixelnerf_b200.h declares."""
    from pixel_nerf_yolo_b200 import _lib, build
    build.build()
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "pixelnerf_b200.h")).read()
    declared = set(re.findall(r"\b(pnr_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.pnr_version() == 3
    # struct layouts agree with the header (sizes computed by the C compiler)
    src = '#include "pixelnerf_b200.h"\n#include <stdio.h>\nint main(){printf("%zu %zu %zu %zu %zu",sizeof(pnr_scene),sizeof(pnr_points),sizeof(pnr_mlp_params),sizeof(pnr_mlp_grads),sizeof(pnr_render_args));}'
    exe = os.path.join(ROOT, "pixel-nerf-yolo_b200", "csrc", "build", "sizes")
    subprocess.run(["gcc", "-x", "c", "-", "-I", os.path.join(ROOT, "include"), "-o", exe], input=src.encode(), check=True)
    sizes = [int(x) for x in subprocess.check_output([exe]).split()]
    assert sizes == [ctypes.sizeof(_lib.Scene), ctypes.sizeof(_lib.Points), ctypes.sizeof(_lib.MlpParams), ctypes.sizeof(_lib.MlpGrads), ctypes.sizeof(_lib.RenderArgs)]


def test_no_silent_cpu_fallback():
    """Without a GPU the product path must raise, not compute on the CPU."""
    if torch.cuda.is_available():
        pytest.skip("GPU box")
    from pixel_nerf_yolo_b200.render import NeRFRenderer
    from pixel_nerf_yolo_b200.model.code import PositionalEncoding
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        NeRFRenderer(64, 32, 16)(object(), torch.zeros(1, 4, 8))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        PositionalEncoding(6, 3, 1.5)(torch.zeros(3, 3))


def test_unsupported_options_raise():
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.model.resnetfc import ResnetFC
    from pixel_nerf_yolo_b200.model.encoder import SpatialEncoder
    from pixel_nerf_yolo_b200.render.render_util import make_renderer
    with pytest.raises(NotImplementedError):
        ResnetFC(42, 4, d_latent=512, d_hidden=512, combine_type="max")
    with pytest.raises(NotImplementedError):
        ResnetFC(42, 4, d_latent=512, d_hidden=512, beta=100.0)
    with pytest.raises(NotImplementedError):
        SpatialEncoder("resnet34", pretrained=False, index_padding="border")
    with pytest.raises(NotImplementedError):
        make_renderer(ConfigTree.from_dict({"renderer": {"type": "volsdf"}}))
    from pixel_nerf_yolo_b200.render import YoloRenderer
    y = make_renderer(ConfigTree.from_dict({"renderer": {"type": "yolo", "n_coarse": 128},
                                            "model": {"mlp_coarse": {"num_anchors_per_scale": 3}}}))
    assert isinstance(y, YoloRenderer) and (y.n_coarse, y.num_anchors_per_scale) == (128, 3)
    with pytest.raises(RuntimeError):
        y(torch.zeros(4, 8))                          # no network bound


def test_model_api_and_state_dict_names():
    from helpers import MODEL_CONF
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.model import make_model
    from pixel_nerf_yolo_b200.render import NeRFRenderer
    import pixel_nerf_yolo_b200.synth as synth
    net = make_model(ConfigTree.from_dict(MODEL_CONF))
    sd = net.state_dict()
    assert (net.d_in, net.d_latent, net.d_out) == (42, 512, 4)
    for mlp in ("mlp_coarse", "mlp_fine"):
        for k, v in synth.mlp_state(0).items():
            assert tuple(sd[f"{mlp}.{k}"].shape) == tuple(v.shape)
    assert "code._freqs" in sd and "code._phases" in sd and "poses" not in sd and "encoder.latent" not in sd
    assert sum(p.numel() for p in net.parameters()) == 28161864          # SURVEY.md section 3.3
    r = NeRFRenderer.from_conf(ConfigTree.from_dict({"n_coarse": 64, "n_fine": 32, "n_fine_depth": 16, "sched": []}))
    assert set(r.state_dict()) == {"iter_idx", "last_sched"} and r.using_fine and r.sched is None


def test_shard_bounds_cover_and_align():
    from pixel_nerf_yolo_b200.dist import shard_bounds
    for n in (0, 1, 31, 32, 33, 2048, 16384, 16385, 409600):
        for world in (1, 2, 3, 4, 8):
            b = shard_bounds(n, world)
            assert b[0][0] == 0 and b[-1][1] == n and all(b[i][1] == b[i + 1][0] for i in range(world - 1))
            assert all(s % 32 == 0 for s, _ in b if s < n)
            sizes = [e - s for s, e in b]
            assert max(sizes) - min(sizes) < 2 * 32 or n < 32 * world   # last slice is clipped to n


def test_sharded_render_two_ranks_gloo_matches_single():
    """world_size-2 gloo run of ShardedRenderer: gathered output == the unsharded render, bit for bit."""
    import socket
    script = os.path.join(ROOT, "tests", "_gloo_worker.py")
    with socket.socket() as sk:                      # a free rendezvous port
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port), script],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "GLOO_SHARD_OK" in r.stdout


def test_sched_step_follows_reference_schedule():
    """nerf.py:324-344: sched = [iteration thresholds, n_coarse values, n_fine values]; the persistent buffers iter_idx /
    last_sched carry the position through a checkpoint (forward re-reads the resolution from last_sched, nerf.py:271-273)."""
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.render import NeRFRenderer
    conf = {"n_coarse": 64, "n_fine": 32, "n_fine_depth": 16, "sched": [[2, 5], [96, 128], [48, 64]]}
    r = NeRFRenderer.from_conf(ConfigTree.from_dict(conf))
    seen = []
    for _ in range(6):
        r.sched_step()
        seen.append((int(r.iter_idx), int(r.last_sched), r.n_coarse, r.n_fine))
    assert seen == [(1, 0, 64, 32), (2, 1, 96, 48), (3, 1, 96, 48), (4, 1, 96, 48), (5, 2, 128, 64), (6, 2, 128, 64)]
    r.sched_step(10)                                    # past the last threshold: nothing more to change
    assert (int(r.last_sched), r.n_coarse, r.n_fine) == (2, 128, 64)
    r2 = NeRFRenderer.from_conf(ConfigTree.from_dict(conf))
    r2.load_state_dict(r.state_dict())
    assert int(r2.iter_idx) == 16 and int(r2.last_sched) == 2 and r2.n_coarse == 64     # restored lazily, at the next forward
    r3 = NeRFRenderer.from_conf(ConfigTree.from_dict(conf))
    r3.sched_step(3)                                    # a multi-iteration step crosses one threshold
    assert (int(r3.last_sched), r3.n_coarse, r3.n_fine) == (1, 96, 48)
    none = NeRFRenderer.from_conf(ConfigTree.from_dict({"n_coarse": 64, "sched": []}))
    none.sched_step()
    assert int(none.iter_idx) == 0 and none.sched is None


def test_state_dict_is_checkpoint_compatible_with_reference():
    """A checkpoint written by the reference's trainer loads with strict=True: same names, shapes and dtypes as the
    unmodified reference's state_dict (manifest generated by tests/golden/make_golden_state_dict.py), same PE buffers."""
    import json
    from helpers import MODEL_CONF, RENDER_CONF
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.model import make_model
    from pixel_nerf_yolo_b200.render import NeRFRenderer
    man = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_state_dict.json")))
    net = make_model(ConfigTree.from_dict(MODEL_CONF))
    sd = net.state_dict()
    ours = {k: [list(v.shape), str(v.dtype)] for k, v in sd.items()}
    assert set(ours) == set(man["model"]), (sorted(set(ours) - set(man["model"]))[:5], sorted(set(man["model"]) - set(ours))[:5])
    assert ours == man["model"]
    assert sd["code._freqs"].flatten().tolist() == man["code._freqs"]
    assert sd["code._phases"].flatten().tolist() == man["code._phases"]
    assert sum(p.numel() for p in net.parameters()) == man["n_params"]
    r = NeRFRenderer.from_conf(ConfigTree.from_dict(RENDER_CONF))
    assert {k: [list(v.shape), str(v.dtype)] for k, v in r.state_dict().items()} == man["renderer"]
    # a synthetic "reference checkpoint" with exactly the manifest's entries loads strictly
    import torch
    fake = {k: torch.zeros(shape, dtype=getattr(torch, dt.split(".")[1])) for k, (shape, dt) in man["model"].items()}
    net.load_state_dict(fake, strict=True)


def test_render_state_key_tracks_generations():
    """MultiDeviceRenderer / the prepared render arguments decide "did anything change" from explicit generation counters
    (a new encode, new cameras, new weights), never from pointer identity, which the caching allocator re-issues (ABA)."""
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.dist import MultiDeviceRenderer
    from pixel_nerf_yolo_b200.model import make_model
    from pixel_nerf_yolo_b200.render import NeRFRenderer
    import pixel_nerf_yolo_b200.synth as synth
    conf = {"use_encoder": True, "use_xyz": True, "use_code": True, "code": {"num_freqs": 6, "freq_factor": 1.5, "include_input": True},
            "use_viewdirs": True, "use_code_viewdirs": False,
            "mlp_coarse": {"type": "resnet", "n_blocks": 5, "d_hidden": 512, "d_out": 4, "combine_layer": 3, "combine_type": "average"},
            "mlp_fine": {"type": "resnet", "n_blocks": 5, "d_hidden": 512, "d_out": 4, "combine_layer": 3, "combine_type": "average"},
            "encoder": {"backbone": "resnet34", "pretrained": False, "num_layers": 4, "index_padding": "zeros"}}
    net = make_model(ConfigTree.from_dict(conf)).eval()
    scene = synth.scene_config1(seed=1, num_views=3, feat=8)
    net.num_objs, net.num_views_per_obj = 1, 3
    net.encoder.set_latent(scene["latent"])
    net.set_cameras(scene["poses"].reshape(-1, 4, 4), scene["focal"], scene["image_wh"])
    md = MultiDeviceRenderer(NeRFRenderer(64, 32, 16).bind_parallel(net, None, simple_output=True), [0, 1])
    k0 = md.state_key()
    assert md.state_key() == k0
    # same storage, same version, new content: pointer identity would not notice a re-encode into a recycled buffer
    lat = scene["latent"]
    net.encoder.set_latent(lat)
    k1 = md.state_key()
    assert k1 != k0
    net.set_cameras(scene["poses"].reshape(-1, 4, 4), scene["focal"], scene["image_wh"])
    k2 = md.state_key()
    assert k2 != k1
    with torch.no_grad():
        net.mlp_coarse.lin_in.bias.add_(1.0)                      # optimizer-style in-place step
    k3 = md.state_key()
    assert k3 != k2
    net.mlp_fine.lin_out.weight.data.mul_(2.0)                    # behind autograd's back: explicit invalidate()
    assert md.state_key() == k3
    net.mlp_fine.invalidate()
    k4 = md.state_key()
    assert k4 != k3
    net.mlp_coarse.load_state_dict(synth.mlp_state(3))
    assert md.state_key() != k4
    md._key = md.state_key()
    md.invalidate()
    assert md._key is None
    # a call that would record a backward pass is refused (the replicas' gradients are not reduced onto `net`)
    with pytest.raises(NotImplementedError, match="inference driver"):
        md(torch.zeros(1, 4, 8))
