#!/usr/bin/env python
"""Cost of antialiasing (GaussianRasterizationSettings(..., antialiasing=True)) on two shapes: the C2 view (bench.py's
`c2` workload, one decoded view, 980x545) and 1 M synthetic Gaussians at 3840x2160.

    python tools/antialiasing_bench.py [--launches 100] [--out FILE]

For each shape it rasterizes once with antialiasing off and once on, then times on those workspaces, alternating the
two members of each pair launch by launch with CUDA events around each launch:
    splatco_preprocess_fwd  vs splatco_preprocess_fwd_aa
    splatco_blend_fwd       on the plain vs the antialiased geometry record (the record opacity changes the live pairs)
    splatco_blend_bwd       likewise
    splatco_preprocess_bwd  vs splatco_preprocess_bwd_aa
    the rasterizer's forward + backward (GaussianRasterizer, colour loss), off vs on
and prints one JSON line with the median (and quartiles) of each, the on/off ratios, the GPU's name and its power
limit.  Gradient buffers are reset before every backward launch, outside the timed window.  Needs a GPU."""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.depth_alpha_bench import gpu_info  # noqa: E402


def c2_inputs(dev):
    import bench
    from splatco_b200.gaussian_renderer import _settings, generate_neural_gaussians, prefilter_voxel
    cfg = dict(bench.WORKLOADS["c2"])
    bench.LEVEL = 2
    pc = bench.build_model(cfg, dev)
    cams, _ = bench.build_views(cfg)
    cam = cams[0].to(dev)
    bg = torch.ones(3, device=dev)
    with torch.no_grad():
        vm = prefilter_voxel(cam, pc, bench.PIPE, bg)
        xyz, color, opacity, scaling, rot, _, _ = generate_neural_gaussians(cam, pc, vm, is_training=True)
    return [t.detach().contiguous() for t in (xyz, color, opacity, scaling, rot)], _settings(cam, bench.PIPE, bg, 1.0)


def synthetic_inputs(dev, M=1_000_000, W=3840, H=2160):
    from tests.util import scene, settings_for
    cam, means, colors, opac, scales, rots = scene(M, W, H, 11, sigma_px=(0.3, 4.0))
    return [t.to(dev).contiguous() for t in (means, colors, opac, scales, rots)], settings_for(cam, [1.0, 1.0, 1.0])


def time_pairs(calls, pairs, launches, reset):
    res = {}
    for a, b in pairs:
        ms = {a: [], b: []}
        for i in range(launches + 10):                          # the first 10 rounds warm up
            for k in ((a, b) if i % 2 == 0 else (b, a)):
                if k in reset:
                    reset[k]()
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
    return res


def measure(ins, settings, launches):
    from splatco_b200 import _lib
    from splatco_b200._lib import check, ptr
    from splatco_b200.diff_gaussian_rasterization import GaussianRasterizer, rasterize_forward_state
    dev = ins[0].device
    xyz, color, opacity, scaling, rot = ins
    s_off, s_on = settings._replace(antialiasing=False), settings._replace(antialiasing=True)
    with torch.no_grad():
        _, _, st0 = rasterize_forward_state(*ins, s_off)
        _, _, st1 = rasterize_forward_state(*ins, s_on)
    torch.cuda.synchronize()
    assert st0.R == st1.R and torch.equal(st0.radii, st1.radii)
    L = _lib.lib()
    P, R, H, W = st0.P, st0.RL, st0.H, st0.W
    stream = _lib.raw_stream(dev)
    bg = settings.bg.float().contiguous()
    view, proj = settings.viewmatrix.float().contiguous(), settings.projmatrix.float().contiguous()
    tx, ty = float(settings.tanfovx), float(settings.tanfovy)
    geom = torch.empty_like(st0.geom)
    radii = torch.empty_like(st0.radii)
    g = torch.Generator(device=dev).manual_seed(0)
    dC = torch.randn(3, H, W, device=dev, generator=g) / (3 * H * W)
    out_c = torch.empty(3, H, W, device=dev)
    gbuf = torch.zeros(10 * P, device=dev)
    g2, gc, go, gcol = gbuf.split_with_sizes([3 * P, 3 * P, P, 3 * P])
    with torch.no_grad():                                       # the blend gradients of the antialiased view
        check(L.splatco_blend_bwd(P, R, H, W, ptr(bg), ptr(st1.geom), ptr(st1.binning), ptr(st1.image), ptr(dC),
                                  ptr(g2), ptr(gc), ptr(go), ptr(gcol), stream), "blend_bwd")
    go_saved = go.clone()
    g3, gs, gq = torch.empty(P, 3, device=dev), torch.empty(P, 3, device=dev), torch.empty(P, 4, device=dev)
    pre = lambda name: (lambda: check(getattr(L, name)(
        P, ptr(xyz), ptr(scaling), 3, ptr(rot), ptr(opacity), ptr(color), 1.0, ptr(view), ptr(proj), tx, ty, H, W,
        ptr(radii), ptr(geom), None, stream), name))
    blend_f = lambda s: (lambda: check(L.splatco_blend_fwd(R, H, W, ptr(bg), ptr(s.geom), ptr(s.binning), ptr(s.image),
                                                           ptr(out_c), stream), "blend_fwd"))
    blend_b = lambda s: (lambda: check(L.splatco_blend_bwd(P, R, H, W, ptr(bg), ptr(s.geom), ptr(s.binning),
                                                           ptr(s.image), ptr(dC), ptr(g2), ptr(gc), ptr(go), ptr(gcol),
                                                           stream), "blend_bwd"))
    pre_args = lambda: (P, ptr(xyz), ptr(scaling), 3, ptr(rot), 1.0, ptr(view), ptr(proj), tx, ty, H, W,
                        ptr(st1.radii), ptr(g2), ptr(gc), ptr(g3), ptr(gs), ptr(gq))
    leaves = [t.clone().requires_grad_() for t in ins]

    def raster(s):
        def run():
            img, _ = GaussianRasterizer(s)(means3D=leaves[0], means2D=torch.zeros_like(leaves[0]), shs=None,
                                           colors_precomp=leaves[1], opacities=leaves[2], scales=leaves[3],
                                           rotations=leaves[4], cov3D_precomp=None)
            img.backward(dC)
        return run
    calls = {
        "preprocess_fwd": pre("splatco_preprocess_fwd"), "preprocess_fwd_aa": pre("splatco_preprocess_fwd_aa"),
        "blend_fwd": blend_f(st0), "blend_fwd_aa": blend_f(st1),
        "blend_bwd": blend_b(st0), "blend_bwd_aa": blend_b(st1),
        "preprocess_bwd": lambda: check(L.splatco_preprocess_bwd(*pre_args(), stream), "preprocess_bwd"),
        "preprocess_bwd_aa": lambda: check(L.splatco_preprocess_bwd_aa(*pre_args(), ptr(opacity), ptr(go), None, None,
                                                                       None, None, stream), "preprocess_bwd_aa"),
        "raster_fwd_bwd": raster(s_off), "raster_fwd_bwd_aa": raster(s_on),
    }
    clear_grads = lambda: [setattr(x, "grad", None) for x in leaves]
    reset = {"blend_bwd": gbuf.zero_, "blend_bwd_aa": gbuf.zero_, "preprocess_bwd": lambda: go.copy_(go_saved),
             "preprocess_bwd_aa": lambda: go.copy_(go_saved), "raster_fwd_bwd": clear_grads,
             "raster_fwd_bwd_aa": clear_grads}
    pairs = [(k, k + "_aa") for k in ("preprocess_fwd", "blend_fwd", "blend_bwd", "preprocess_bwd", "raster_fwd_bwd")]
    res = {"H": H, "W": W, "gaussians": P, "instances": st0.R}
    res.update(time_pairs(calls, pairs, launches, reset))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=100, help="timed launches of each member of a pair (>= 30)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("antialiasing_bench: needs a CUDA device")
    if args.launches < 30:
        sys.exit("antialiasing_bench: --launches must be >= 30")
    dev = torch.device("cuda")
    res = {"launches": args.launches}
    res.update(gpu_info())
    res["c2"] = measure(*c2_inputs(dev), args.launches)
    res["synthetic_1M_3840x2160"] = measure(*synthetic_inputs(dev), args.launches)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
