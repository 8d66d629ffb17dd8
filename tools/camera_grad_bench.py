#!/usr/bin/env python
"""Cost of camera gradients: one view's backward with and without them.

    python tools/camera_grad_bench.py [--rounds 50] [--out FILE]

Two shapes:
  * c2: bench.py's C2 model, one view at 980x545 through render() (decode + rasterizer).  Per round, one forward with a
    plain camera and one whose world_view_transform, full_proj_transform and camera_center require grad (the order
    alternates round by round); only loss.backward() is timed, with CUDA events around it.
  * c5_1M: 1 M Gaussians fed straight to the rasterizer at 3840x2160 (BASELINE.md's C5 shape), the rasterizer's
    backward (rasterize_backward_state) on one forward's workspaces, with and without camera=True, alternating.
Prints one JSON line with the median (and quartiles) of each, their ratio, the GPU's name and its power limit.
Needs a GPU."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, limit = [s.strip() for s in out[torch.cuda.current_device()].split(",")]
        return {"gpu": name, "power_limit": limit}
    except Exception as e:
        return {"gpu": torch.cuda.get_device_name(), "power_limit": f"unknown ({type(e).__name__})"}


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def summary(ms):
    q = np.percentile(ms, [25, 50, 75])
    return {"p25": round(float(q[0]), 4), "median": round(float(q[1]), 4), "p75": round(float(q[2]), 4)}


def bench_c2(rounds):
    import bench
    from splatco_b200.gaussian_renderer import prefilter_voxel, render
    cfg = dict(bench.WORKLOADS["c2"])
    bench.LEVEL = 2
    dev = torch.device("cuda")
    pc = bench.build_model(cfg, dev)
    cams, _ = bench.build_views(cfg)
    cam = cams[0].to(dev)
    bg = torch.ones(3, device=dev)
    g = torch.Generator(device=dev).manual_seed(0)
    dC = torch.randn(3, cfg["H"], cfg["W"], device=dev, generator=g) / (3 * cfg["H"] * cfg["W"])

    def camera(grad):
        c = cam.to(dev)
        if grad:
            c.world_view_transform = c.world_view_transform.clone().requires_grad_()
            c.full_proj_transform = c.full_proj_transform.clone().requires_grad_()
            c.camera_center = c.camera_center.clone().requires_grad_()
        return c

    ms = {False: [], True: []}
    for i in range(rounds + 5):                       # the first 5 rounds warm up
        for grad in ((False, True) if i % 2 == 0 else (True, False)):
            c = camera(grad)
            for p in pc.parameters():
                p.grad = None
            img = render(c, pc, bench.PIPE, bg, visible_mask=prefilter_voxel(c, pc, bench.PIPE, bg))["render"]
            torch.cuda.synchronize()
            t = timed(lambda: img.backward(dC))
            if grad:
                assert c.world_view_transform.grad is not None and c.camera_center.grad is not None
            if i >= 5:
                ms[grad].append(t)
    return {"c2_view_backward_ms": summary(ms[False]), "c2_view_backward_camera_ms": summary(ms[True]),
            "c2_ratio": round(float(np.median(ms[True]) / np.median(ms[False])), 4)}


def bench_c5(rounds):
    from splatco_b200.diff_gaussian_rasterization import rasterize_backward_state, rasterize_forward_state
    from splatco_b200.synthetic import random_gaussians, ring_cameras
    from tests.util import settings_for
    W, H, M = 3840, 2160, 1_000_000
    cam = ring_cameras(3, W, H)[1]
    ins = [t.cuda() for t in random_gaussians(M, cam, 1, sigma_px=(0.5, 4.0))]
    st = settings_for(cam, [1.0, 1.0, 1.0])
    with torch.no_grad():
        _, radii, state = rasterize_forward_state(*ins, st)
    g = torch.Generator(device="cuda").manual_seed(0)
    dC = torch.randn(3, H, W, device="cuda", generator=g) / (3 * H * W)
    ms = {False: [], True: []}
    for i in range(rounds + 5):
        for cam_grad in ((False, True) if i % 2 == 0 else (True, False)):
            t = timed(lambda: rasterize_backward_state(state, dC, ins[0], ins[3], ins[4], st, camera=cam_grad))
            if i >= 5:
                ms[cam_grad].append(t)
    return {"c5_1M_gaussians_visible": int((radii > 0).sum()), "c5_raster_backward_ms": summary(ms[False]),
            "c5_raster_backward_camera_ms": summary(ms[True]),
            "c5_ratio": round(float(np.median(ms[True]) / np.median(ms[False])), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=50, help="timed rounds of each variant (>= 20)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("camera_grad_bench: needs a CUDA device")
    if args.rounds < 20:
        sys.exit("camera_grad_bench: --rounds must be >= 20")
    res = {"rounds": args.rounds}
    res.update(gpu_info())
    res.update(bench_c2(args.rounds))
    res.update(bench_c5(args.rounds))
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
