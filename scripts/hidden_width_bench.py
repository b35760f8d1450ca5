"""Render and training-step time of the benchmarked network at ResnetFC hidden widths 128 / 256 / 512, on one GPU.

* render: bench.py's workload (16 384-ray 3-view 128x128 image, 64 coarse + 32 fine samples, bf16 tensor-core path through the
  single-call render) with the hidden width changed, synthetic weights of that width.  At d_hidden <= 256 the field kernel runs
  the one-tile variant (network zero-padded to 256 features) and, the latent (512) being wider than the network, gathers the
  lin_z pre-projections of the maps;
* train: bench.py's config-3 training step (4 objects x 128 rays, 3 views, forward + backward) on the tcgen05 arithmetic.

Each step is timed with CUDA events with the L2 overwritten (256 MiB write) before it; the widths are alternated step by step
in one process so that they see the same machine state.  The device name and power limit are read with nvidia-smi in the same
run.

    python scripts/hidden_width_bench.py --steps 20 --warmup 3 --out /tmp/r04_hidden_width.json
"""
import argparse
import copy
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench as B  # noqa: E402

WIDTHS = (128, 256, 512)


def model_conf(d_hidden):
    conf = copy.deepcopy(B.MODEL_CONF)
    for k in ("mlp_coarse", "mlp_fine"):
        conf[k]["d_hidden"] = d_hidden
    return conf


def build_render(d_hidden, device):
    """bench.build_ours at another hidden width: the render module bound to its network, and the rays."""
    import pixel_nerf_yolo_b200.synth as synth
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.model import make_model
    from pixel_nerf_yolo_b200.render import NeRFRenderer
    scene, images, rays = B.scene_inputs()
    torch.manual_seed(0)
    net = make_model(ConfigTree.from_dict(model_conf(d_hidden))).eval()
    net.mlp_coarse.load_state_dict(synth.mlp_state(1, d_hidden=d_hidden))
    net.mlp_fine.load_state_dict(synth.mlp_state(2, d_hidden=d_hidden))
    net = net.to(device).requires_grad_(False)
    with torch.no_grad():
        net.encode(images.to(device), scene["poses"].to(device), scene["focal"].to(device))
        lat = net.encoder.latent
        net.encoder.set_latent(lat / lat.std())
    renderer = NeRFRenderer(B.KC, B.KF, B.KFD, depth_std=0.01, white_bkgd=True, eval_batch_size=50000).eval().to(device)
    render_par = renderer.bind_parallel(net, None, simple_output=True).eval()
    rays = rays.to(device)

    def step():
        with torch.no_grad():
            return render_par(rays)
    return step, net.projects_latent()


def build_train(d_hidden, device):
    """bench.train_step_block's step at another hidden width, tcgen05 arithmetic."""
    import pixel_nerf_yolo_b200.synth as synth
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.model import make_model
    from pixel_nerf_yolo_b200.render import NeRFRenderer
    scene = synth.scene_config1(seed=5, num_views=B.NS, C=B.C_LAT, size=B.SIZE, feat=64, num_objs=4)
    net = make_model(ConfigTree.from_dict(model_conf(d_hidden)))
    net.mlp_coarse.load_state_dict(synth.mlp_state(1, d_hidden=d_hidden))
    net.mlp_fine.load_state_dict(synth.mlp_state(2, d_hidden=d_hidden))
    net = net.to(device).train()
    net.num_objs, net.num_views_per_obj = 4, B.NS
    lat = scene["latent"].to(device).clone().requires_grad_(True)
    net.encoder.set_latent(lat)
    net.set_cameras(scene["poses"].reshape(-1, 4, 4).to(device), scene["focal"].to(device), scene["image_wh"])
    net.train_precision = "bf16"
    allr = torch.cat([synth.target_rays(B.SIZE, 15.0 + 20 * s, -10.0) for s in range(4)])
    pick = torch.from_numpy(np.random.default_rng(1).choice(B.SIZE * B.SIZE, 128, replace=False)).long()
    rays = allr[:, pick].contiguous().to(device)
    gt = torch.rand(4, 128, 3, device=device)
    params = list(net.mlp_coarse.parameters()) + list(net.mlp_fine.parameters())
    r = NeRFRenderer(B.KC, B.KF, B.KFD, white_bkgd=True).train().to(device)

    def step():
        for p in params:
            p.grad = None
        lat.grad = None
        res = r(net, rays)
        loss = ((res.coarse.rgb - gt) ** 2).mean() + ((res.fine.rgb - gt) ** 2).mean()
        loss.backward()
    return step


def gpu_info(index):
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", str(index)],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "sm_clock_max": clock}
    except Exception as e:   # the numbers are still reported, without the card's settings
        return {"name": torch.cuda.get_device_name(index), "power_limit": None, "error": str(e)}


def alternate(steps_by_width, n, flush):
    """n rounds; in each round every width runs one step after an L2 flush.  -> {width: [ms, ...]}"""
    ms = {w: [] for w in steps_by_width}
    for _ in range(n):
        for w, fn in steps_by_width.items():
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms[w].append(e0.elapsed_time(e1))
    return ms


def summary(ms, work):
    med = statistics.median(ms)
    return {"ms_median": round(med, 3), "ms_min": round(min(ms), 3), "ms_max": round(max(ms), 3), "steps": len(ms),
            "rays_per_s": round(work / (med * 1e-3))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("hidden_width_bench.py: no CUDA device")
    device = torch.device("cuda", 0)
    torch.cuda.set_device(device)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    render, projected = {}, {}
    for w in WIDTHS:
        render[w], projected[w] = build_render(w, device)
    train = {w: build_train(w, device) for w in WIDTHS}
    alternate(render, args.warmup, flush)
    alternate(train, args.warmup, flush)
    ms_render = alternate(render, args.steps, flush)
    ms_train = alternate(train, args.steps, flush)
    rays = B.SIZE * B.SIZE
    res = {
        "device": gpu_info(0),
        "render": {"workload": B.WORKLOAD.replace("bf16 ResnetFC", "bf16 ResnetFC at d_hidden = w"),
                   **{str(w): {**summary(ms_render[w], rays), "lin_z_pre_projected": projected[w],
                               "field_kernel_variant": "MT = 1 (Hp = 256)" if w <= 256 else "MT = 2 (Hp = 512)"} for w in WIDTHS}},
        "train": {"workload": "config3: train step, 4 objects x 128 rays, 3 views, 64+32 samples, forward + backward, tcgen05 "
                              "arithmetic (train_precision bf16)",
                  **{str(w): summary(ms_train[w], 512) for w in WIDTHS}},
        "l2": "flushed before every timed step (256 MiB write); widths alternated step by step",
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
