#!/usr/bin/env python
"""Cost of the depth / alpha maps at the C2 view shape (bench.py's `c2` workload, one view, 980x545).

    python tools/depth_alpha_bench.py [--launches 200] [--out FILE]

Builds the C2 model, decodes one view and rasterizes it once, then times on the SAME workspaces, alternating the two
members of each pair launch by launch with CUDA events around each launch:
    splatco_blend_fwd       vs splatco_blend_fwd_depth_alpha
    splatco_blend_bwd       vs splatco_blend_bwd_depth_alpha    (all three upstream maps non-NULL)
    splatco_preprocess_bwd  vs splatco_preprocess_bwd_depth
and prints one JSON line with the median (and quartiles) of each, their ratio, the GPU's name and its power limit.
The gradient buffers are zeroed before every backward launch, outside the timed window.  Needs a GPU."""
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
    except Exception as e:                              # the name at least comes from torch
        return {"gpu": torch.cuda.get_device_name(), "power_limit": f"unknown ({type(e).__name__})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=200, help="timed launches of each kernel (>= 50)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("depth_alpha_bench: needs a CUDA device")
    if args.launches < 50:
        sys.exit("depth_alpha_bench: --launches must be >= 50")
    import bench
    from splatco_b200 import _lib
    from splatco_b200._lib import check, ptr
    from splatco_b200.diff_gaussian_rasterization import rasterize_forward_state
    from splatco_b200.gaussian_renderer import _settings, generate_neural_gaussians, prefilter_voxel

    cfg = dict(bench.WORKLOADS["c2"])
    bench.LEVEL = 2
    dev = torch.device("cuda")
    pc = bench.build_model(cfg, dev)
    cams, _ = bench.build_views(cfg)
    cam = cams[0].to(dev)
    bg = torch.ones(3, device=dev)
    with torch.no_grad():
        vm = prefilter_voxel(cam, pc, bench.PIPE, bg)
        xyz, color, opacity, scaling, rot, _, _ = generate_neural_gaussians(cam, pc, vm, is_training=True)
        st_ = _settings(cam, bench.PIPE, bg, 1.0)
        img, radii, st = rasterize_forward_state(xyz, color, opacity, scaling, rot, st_)
    torch.cuda.synchronize()
    L = _lib.lib()
    P, R, H, W = st.P, st.RL, st.H, st.W
    stream = _lib.raw_stream(dev)
    view, proj = st_.viewmatrix.float().contiguous(), st_.projmatrix.float().contiguous()
    g = torch.Generator(device=dev).manual_seed(0)
    dC = torch.randn(3, H, W, device=dev, generator=g) / (3 * H * W)
    dD = torch.randn(H, W, device=dev, generator=g) / (H * W)
    dA = torch.randn(H, W, device=dev, generator=g) / (H * W)
    out_c, out_d, out_a = torch.empty(3, H, W, device=dev), torch.empty(H, W, device=dev), torch.empty(H, W, device=dev)
    gbuf = torch.zeros(11 * P, device=dev)
    g2, gc, go, gcol, gz = gbuf.split_with_sizes([3 * P, 3 * P, P, 3 * P, P])
    g3 = torch.empty(P, 3, device=dev)
    gs = torch.empty(P, 3, device=dev)
    gq = torch.empty(P, 4, device=dev)
    scl = scaling.contiguous()

    calls = {
        "blend_fwd": lambda: check(L.splatco_blend_fwd(R, H, W, ptr(bg), ptr(st.geom), ptr(st.binning), ptr(st.image),
                                                       ptr(out_c), stream), "blend_fwd"),
        "blend_fwd_depth_alpha": lambda: check(L.splatco_blend_fwd_depth_alpha(
            R, H, W, ptr(bg), ptr(st.geom), ptr(st.binning), ptr(st.image), ptr(out_c), ptr(out_d), ptr(out_a), stream),
            "blend_fwd_depth_alpha"),
        "blend_bwd": lambda: check(L.splatco_blend_bwd(P, R, H, W, ptr(bg), ptr(st.geom), ptr(st.binning), ptr(st.image),
                                                       ptr(dC), ptr(g2), ptr(gc), ptr(go), ptr(gcol), stream), "blend_bwd"),
        "blend_bwd_depth_alpha": lambda: check(L.splatco_blend_bwd_depth_alpha(
            P, R, H, W, ptr(bg), ptr(st.geom), ptr(st.binning), ptr(st.image), ptr(dC), ptr(dD), ptr(dA), ptr(g2), ptr(gc),
            ptr(go), ptr(gcol), ptr(gz), stream), "blend_bwd_depth_alpha"),
        "preprocess_bwd": lambda: check(L.splatco_preprocess_bwd(
            P, ptr(xyz), ptr(scl), 3, ptr(rot), 1.0, ptr(view), ptr(proj), float(st_.tanfovx), float(st_.tanfovy), H, W,
            ptr(st.radii), ptr(g2), ptr(gc), ptr(g3), ptr(gs), ptr(gq), stream), "preprocess_bwd"),
        "preprocess_bwd_depth": lambda: check(L.splatco_preprocess_bwd_depth(
            P, ptr(xyz), ptr(scl), 3, ptr(rot), 1.0, ptr(view), ptr(proj), float(st_.tanfovx), float(st_.tanfovy), H, W,
            ptr(st.radii), ptr(g2), ptr(gc), ptr(g3), ptr(gs), ptr(gq), ptr(gz), stream), "preprocess_bwd_depth"),
    }
    zero_first = {"blend_bwd", "blend_bwd_depth_alpha"}
    pairs = [("blend_fwd", "blend_fwd_depth_alpha"), ("blend_bwd", "blend_bwd_depth_alpha"),
             ("preprocess_bwd", "preprocess_bwd_depth")]
    res = {"workload": "c2 (one view)", "H": H, "W": W, "gaussians": P, "instances": st.R, "launches": args.launches}
    res.update(gpu_info())
    for a, b in pairs:
        ms = {a: [], b: []}
        for i in range(args.launches + 10):                     # the first 10 rounds warm up
            for k in ((a, b) if i % 2 == 0 else (b, a)):
                if k in zero_first:
                    gbuf.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                calls[k]()
                e1.record()
                e1.synchronize()
                if i >= 10:
                    ms[k].append(e0.elapsed_time(e1))
        for k in (a, b):
            q = np.percentile(ms[k], [25, 50, 75])
            res[k + "_ms"] = {"p25": round(float(q[0]), 4), "median": round(float(q[1]), 4), "p75": round(float(q[2]), 4)}
        res[f"{b}_over_{a}"] = round(res[b + "_ms"]["median"] / res[a + "_ms"]["median"], 4)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
