"""Cost of camera gradients on the BASELINE config-3 training step (4 objects x 128 rays, 3 source views, 64 + 32 samples,
forward + backward of the render, both networks and the maps training), against a parent build of the library.

    python scripts/camera_grad_bench.py --parent PARENT_TREE [--rounds 3] [--steps 20] [--out results.json]

PARENT_TREE is a checkout of the parent commit with its library built.  Each round runs three arms, one process each, in an
order that rotates from round to round: the parent tree without camera gradients, this tree without them, and this tree with
the source camera-to-world poses and the focal length requiring grad.  Every process sets the cameras once per step (as
``encode`` does), times ``--steps`` steps per training arithmetic with CUDA events after one warm-up step, and dumps the
gradients of one seeded step.  The summary gives the median step time per (tree, mode, arithmetic) over the rounds, the kernel
launches of the backward pass, and how far the parameter / map gradients without camera gradients are from the parent's, next
to how far two parent runs are apart.  Card name and power limit are recorded beside the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PRECISIONS = ("fp32", "tf32", "bf16")


def worker(tree, mode, steps, dump):
    sys.path.insert(0, tree)
    sys.path.insert(0, os.path.join(tree, "tests"))
    import numpy as np
    import torch
    import helpers as H
    from pixel_nerf_yolo_b200.conf import ConfigTree
    from pixel_nerf_yolo_b200.render import NeRFRenderer
    dev = torch.device("cuda", 0)
    scene = H.make_scene_dict(num_objs=4, num_views=3, feat=64)
    net = H.build_net(scene, device=dev, precision="bf16", train=True)
    lat = scene["latent"].to(dev).clone().requires_grad_(True)
    net.encoder.set_latent(lat)
    rays = H.rays_subset(4, 128, seed=1).to(dev)
    noise = {k: v.to(dev) for k, v in H.make_noise(512, seed=2).items()}
    gt = torch.rand(4, 128, 3, generator=torch.Generator().manual_seed(3)).to(dev)
    r = NeRFRenderer.from_conf(ConfigTree.from_dict(dict(H.RENDER_CONF))).train().to(dev)
    r.noise_override = noise
    params = list(net.parameters())
    c2w = scene["poses"].reshape(-1, 4, 4).to(dev)
    focal = scene["focal"].to(dev)
    cams = mode == "cams"
    res = {"tree": tree, "mode": mode}

    def step():
        for p in params:
            p.grad = None
        lat.grad = None
        poses, f = c2w.clone().requires_grad_(cams), focal.clone().requires_grad_(cams)
        net.set_cameras(poses, f, scene["image_wh"])
        net.last_bwd_launches = 0
        out = r(net, rays)
        loss = ((out.coarse.rgb - gt) ** 2).mean() + ((out.fine.rgb - gt) ** 2).mean()
        loss.backward()
        return poses, f

    for prec in PRECISIONS:
        net.train_precision = prec
        step()
        torch.cuda.synchronize()
        ms = []
        for _ in range(steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        poses, f = step()
        torch.cuda.synchronize()
        res[prec] = {"ms": sorted(ms)[len(ms) // 2], "fwd_launches_last_field": net.last_launches,
                     "bwd_launches": net.last_bwd_launches}
        arrays = {f"{prec}/{n}": p.grad.cpu().numpy() for n, p in net.named_parameters() if p.grad is not None}
        arrays[f"{prec}/latent"] = lat.grad.cpu().numpy()
        if cams:
            arrays[f"{prec}/d_poses"] = poses.grad.cpu().numpy()
            arrays[f"{prec}/d_focal"] = f.grad.cpu().numpy()
        np.savez(dump + f".{prec}.npz", **arrays)
    print(json.dumps(res))


def run(tree, mode, steps, dump):
    cmd = [sys.executable, os.path.abspath(__file__), "--worker", tree, "--mode", mode, "--steps", str(steps), "--dump", dump]
    out = subprocess.run(cmd, check=True, capture_output=True, text=True).stdout
    return json.loads(out.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent", help="parent commit's tree, library built")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", default=None)
    ap.add_argument("--mode", default="plain", choices=("plain", "cams"))
    ap.add_argument("--dump", default=None)
    a = ap.parse_args()
    if a.worker:
        worker(a.worker, a.mode, a.steps, a.dump)
        return
    import numpy as np
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    arms = [("parent", os.path.abspath(a.parent), "plain"), ("this", HERE, "plain"), ("this", HERE, "cams")]
    tmp = tempfile.mkdtemp(prefix="camgrad_")
    rows = []
    for rnd in range(a.rounds):
        for name, tree, mode in arms[rnd % 3:] + arms[:rnd % 3]:       # each arm leads one round in three
            r = run(tree, mode, a.steps, os.path.join(tmp, f"{name}-{mode}-{rnd}"))
            r["name"], r["round"] = name, rnd
            rows.append(r)
            print(json.dumps({k: r[k] for k in ("name", "mode", "round")} | {p: r[p] for p in PRECISIONS}), flush=True)
    summary = {"card": q.stdout.strip() or torch.cuda.get_device_name(0), "steps_per_arm": a.steps, "rounds": a.rounds}
    for name, _, mode in arms:
        for prec in PRECISIONS:
            ms = [r[prec]["ms"] for r in rows if r["name"] == name and r["mode"] == mode]
            summary[f"{name}/{mode}/{prec}"] = {"median_ms": sorted(ms)[len(ms) // 2], "per_round_ms": ms,
                                                "bwd_launches": rows[[i for i, r in enumerate(rows) if r["name"] == name
                                                                      and r["mode"] == mode][0]][prec]["bwd_launches"]}

    def diff(x, y):
        """(bit for bit equal, largest max|a - b| / max|b| over the gradient tensors)"""
        ax, ay = np.load(x), np.load(y)
        if sorted(ax.files) != sorted(ay.files):
            return False, float("inf")
        worst = max(float(np.abs(ax[k] - ay[k]).max() / max(np.abs(ay[k]).max(), 1e-30)) for k in ax.files)
        return all(np.array_equal(ax[k], ay[k]) for k in ax.files), worst
    # the split-K weight gradients and the feature-map gradient are reduced with atomics, so even two parent runs need not agree
    # bit for bit: the parent-vs-parent spread is the yardstick of the this-vs-parent difference
    for prec in PRECISIONS:
        f = lambda n, m, rnd: os.path.join(tmp, f"{n}-{m}-{rnd}.{prec}.npz")
        summary[f"gradients/{prec}"] = {
            "this_plain_vs_parent": [diff(f("this", "plain", k), f("parent", "plain", k)) for k in range(a.rounds)],
            "parent_vs_parent": [diff(f("parent", "plain", k), f("parent", "plain", 0)) for k in range(1, a.rounds)]}
    print(json.dumps(summary, indent=1))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump({"summary": summary, "runs": rows}, fh, indent=1)


if __name__ == "__main__":
    main()
