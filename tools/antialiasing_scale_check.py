#!/usr/bin/env python
"""What antialiasing is for: a render at a quarter of the resolution should look like the full-resolution render
averaged over 4x4 pixel blocks.

    python tools/antialiasing_scale_check.py [--W 1920 --H 1088 --M 300000] [--out FILE]

Renders a scene of Gaussians 0.4-2 px wide at W x H (0.1-0.5 px at W/4 x H/4, the same field of view, so the focal
length scales by 1/4) and compares the W/4 x H/4 render with the 4x4 box average of the W x H render, both with
antialiasing off and both with it on.  Prints one JSON line with the mean and max absolute errors of each setting, the
GPU's name and its power limit.  Needs a GPU."""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.depth_alpha_bench import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--W", type=int, default=1920)
    ap.add_argument("--H", type=int, default=1088)
    ap.add_argument("--M", type=int, default=300_000)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.W % 4 or args.H % 4:
        sys.exit("antialiasing_scale_check: W and H must be multiples of 4")
    if not torch.cuda.is_available():
        sys.exit("antialiasing_scale_check: needs a CUDA device")
    from splatco_b200.diff_gaussian_rasterization import GaussianRasterizer
    from splatco_b200.synthetic import ring_cameras
    from tests.test_oracle_antialiasing import box4, scale_scene
    from tests.util import settings_for
    cam_hi, *ins = scale_scene(args.M, args.W, args.H, 3)
    cam_lo = ring_cameras(3, args.W // 4, args.H // 4)[1]
    ins = [t.cuda() for t in ins]
    res = {"W": args.W, "H": args.H, "gaussians": args.M}
    res.update(gpu_info())
    for aa in (False, True):
        imgs = []
        for cam in (cam_hi, cam_lo):
            st = settings_for(cam, [0.0, 0.0, 0.0])._replace(antialiasing=aa)
            with torch.no_grad():
                img, _ = GaussianRasterizer(st)(means3D=ins[0], means2D=torch.zeros_like(ins[0]), shs=None,
                                                colors_precomp=ins[1], opacities=ins[2], scales=ins[3], rotations=ins[4],
                                                cov3D_precomp=None)
            imgs.append(img.cpu().numpy())
        d = np.abs(imgs[1] - box4(imgs[0]))
        key = "aa_on" if aa else "aa_off"
        res[key] = {"mean_abs_err": round(float(d.mean()), 5), "max_abs_err": round(float(d.max()), 4),
                    "mean_low_res": round(float(imgs[1].mean()), 4), "mean_full_res": round(float(imgs[0].mean()), 4)}
    res["err_off_over_on"] = round(res["aa_off"]["mean_abs_err"] / res["aa_on"]["mean_abs_err"], 2)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
