"""Render time of the two view-pooling settings of ResnetFC next to the benchmarked one, on one GPU.

Three full 128x128 renders (16 384 rays, 64 coarse + 32 fine samples = 160 field points per ray, bf16 tensor-core path through
the single-call render), timed with CUDA events, the L2 overwritten (256 MiB write) before every timed step, the three
configurations alternated step by step in one process so that they see the same machine state:

  single : one source view, the 3-block network of conf/default.conf (no combine_layer: no pooling, lin_z before every block)
  max    : 3 source views, 5 blocks, combine_layer 3, combine_type max
  average: the same network with combine_type average (the network shape of bench.py; synthetic weights and feature maps here)

FLOPs are algorithmic, from the shapes (2 per multiply-add of every Linear; a pooled network runs blocks [0, combine_layer) and
lin_z once per (point, view) and the rest once per point; without pooling every block runs once per point).

    python scripts/pooling_bench.py --steps 30 --warmup 5 --out /tmp/pooling_bench.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SIZE, KC, KF, KFD = 128, 64, 32, 16
H, D_IN, C_LAT, D_OUT = 512, 42, 512, 4
CONFIGS = {   # name -> (source views, mlp conf)
    "single": (1, {"n_blocks": 3}),
    "max": (3, {"n_blocks": 5, "combine_layer": 3, "combine_type": "max"}),
    "average": (3, {"n_blocks": 5, "combine_layer": 3, "combine_type": "average"}),
}


def flop_per_point(ns, n_blocks, combine_layer=1000):
    cl = min(combine_layer, n_blocks)
    per_view = D_IN * H + cl * (C_LAT * H + 2 * H * H)             # lin_in, then lin_z + fc_0 + fc_1 of blocks [0, cl)
    return 2 * (ns * per_view + (n_blocks - cl) * 2 * H * H + H * D_OUT)


def build(name, device):
    import pixel_nerf_yolo_b200.synth as synth
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.model import make_model
    ns, mlp = CONFIGS[name]
    mlp_conf = {"type": "resnet", "d_hidden": H, "d_out": D_OUT, **mlp}
    conf = {"use_encoder": True, "use_global_encoder": False, "use_xyz": True, "use_code": True,
            "code": {"num_freqs": 6, "freq_factor": 1.5, "include_input": True}, "use_viewdirs": True, "use_code_viewdirs": False,
            "mlp_coarse": mlp_conf, "mlp_fine": mlp_conf,
            "encoder": {"backbone": "resnet34", "pretrained": False, "num_layers": 4, "index_padding": "zeros"}}
    net = make_model(ConfigTree.from_dict(conf)).eval()
    shape = dict(n_blocks=mlp["n_blocks"], combine_layer=mlp.get("combine_layer", 1000))
    net.mlp_coarse.load_state_dict(synth.mlp_state(1, **shape))
    net.mlp_fine.load_state_dict(synth.mlp_state(2, **shape))
    net = net.to(device).requires_grad_(False)
    scene = synth.scene_config1(seed=0, num_views=ns, C=C_LAT, size=SIZE)
    net.num_objs, net.num_views_per_obj = 1, ns
    net.encoder.set_latent(scene["latent"].to(device))
    net.set_cameras(scene["poses"].reshape(-1, 4, 4).to(device), scene["focal"].to(device), scene["image_wh"])
    return net, flop_per_point(ns, mlp["n_blocks"], mlp.get("combine_layer", 1000)) * (KC + KC + KF) * SIZE * SIZE


def gpu_identity():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": power, "sm_clock_max": clock}
    except Exception as e:          # the measurement stands without it, but says so
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"not read ({e})", "sm_clock_max": "not read"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pooling_bench.py: no CUDA device (the render path has no CPU fallback)")
    from pixel_nerf_yolo_b200.render import NeRFRenderer
    import pixel_nerf_yolo_b200.synth as synth
    device = torch.device("cuda", 0)
    torch.cuda.set_device(device)
    nets = {n: build(n, device) for n in CONFIGS}
    renderer = NeRFRenderer(KC, KF, KFD, depth_std=0.01, white_bkgd=True, eval_batch_size=50000).eval().to(device)
    rays = synth.target_rays(SIZE, theta=15.0, phi=-10.0).to(device)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
    torch.manual_seed(0)
    times = {n: [] for n in CONFIGS}
    with torch.no_grad():
        for n, (net, _) in nets.items():                              # every shape warmed up before anything is timed
            for _ in range(args.warmup):
                renderer(net, rays)
        torch.cuda.synchronize()
        for _ in range(args.steps):
            for n, (net, _) in nets.items():
                flush.fill_(1)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                res = renderer(net, rays)
                e1.record()
                e1.synchronize()
                times[n].append(e0.elapsed_time(e1))
                assert torch.isfinite(res.fine.rgb).all()
    result = {"what": "full 128x128 render (16384 rays, 64+32 samples), bf16 tensor-core path, L2 flushed between steps, "
                      "configurations alternated step by step; ms per image from CUDA events", **gpu_identity(),
              "steps": args.steps, "warmup": args.warmup, "configs": {}}
    for n, (net, flop) in nets.items():
        t = sorted(times[n])
        med = statistics.median(t)
        result["configs"][n] = {"source_views": CONFIGS[n][0], "mlp": CONFIGS[n][1], "ms_median": round(med, 4),
                                "ms_min": round(t[0], 4), "ms_max": round(t[-1], 4), "gflop_per_image": round(flop / 1e9, 3),
                                "tflops_at_median": round(flop / (med * 1e-3) / 1e12, 1)}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
