#!/usr/bin/env python
"""Pose refinement with the camera gradients: render() recovers a perturbed camera pose.

    python tools/pose_refine_check.py [--steps 300] [--rot-deg 0.2] [--trans-frac 0.005] [--out FILE]

bench.py's C1 model (10k anchors x 10 offsets, 256x256) is rendered at a true pose to give the target image.  The
camera is then x_cam = exp(delta) x_cam_true (delta = (omega, t) in se(3)), starting from a delta that rotates by
--rot-deg degrees and moves by --trans-frac of the mean anchor depth.  Only delta is optimised (Adam on an L1 image
loss, the model frozen); world_view_transform, full_proj_transform and camera_center are rebuilt from it every step, so
the gradient reaches delta through the rasterizer's projection and through the decode's view direction.  Prints one
JSON line with the rotation and translation error before and after.  This shows the feature doing its job; it is not
a unit test.  Needs a GPU."""
import argparse
import json
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def se3_exp(delta):
    w, t = delta[:3], delta[3:]
    z = delta.new_zeros(())
    X = torch.stack([torch.stack([z, -w[2], w[1], t[0]]), torch.stack([w[2], z, -w[0], t[1]]),
                     torch.stack([-w[1], w[0], z, t[2]]), torch.stack([z, z, z, z])])
    return torch.linalg.matrix_exp(X)


def pose_error(delta):
    """(rotation angle in degrees, translation norm) of exp(delta): the distance of the camera from the true one."""
    T = se3_exp(delta.detach())
    c = ((T[0, 0] + T[1, 1] + T[2, 2] - 1.0) * 0.5).clamp(-1.0, 1.0)
    return math.degrees(float(torch.arccos(c))), float(T[:3, 3].norm())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--rot-deg", type=float, default=0.2)
    ap.add_argument("--trans-frac", type=float, default=0.005)
    ap.add_argument("--lr", type=float, default=2e-3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("pose_refine_check: needs a CUDA device")
    import bench
    from types import SimpleNamespace
    from splatco_b200.gaussian_renderer import prefilter_voxel, render
    cfg = dict(bench.WORKLOADS["c1"])
    bench.LEVEL = 2
    dev = torch.device("cuda")
    pc = bench.build_model(cfg, dev)
    pc.feat_planes.Q0 = 0.0
    for p in pc.parameters():
        p.requires_grad_(False)
    pc.eval()                                  # BatchNorm on its running statistics: the scene does not move with the view
    cams, _ = bench.build_views(cfg)
    cam = cams[1 % len(cams)].to(dev)
    wv0, full0 = cam.world_view_transform.double(), cam.full_proj_transform.double()
    proj = torch.linalg.solve(wv0, full0)
    bg = torch.ones(3, device=dev)

    def camera(delta):
        wv = wv0 @ se3_exp(delta).transpose(0, 1)            # world->camera: exp(delta) after the true transform
        return SimpleNamespace(uid=0, image_width=cam.image_width, image_height=cam.image_height, FoVx=cam.FoVx,
                               FoVy=cam.FoVy, world_view_transform=wv.float(), full_proj_transform=(wv @ proj).float(),
                               camera_center=torch.linalg.inv(wv)[3, :3].float())

    def image(delta):
        c = camera(delta)
        return render(c, pc, bench.PIPE, bg, visible_mask=prefilter_voxel(c, pc, bench.PIPE, bg))["render"]

    with torch.no_grad():
        target = image(torch.zeros(6, dtype=torch.float64, device=dev))
        anchors = torch.cat([pc.get_anchor, torch.ones(pc.get_anchor.shape[0], 1, device=dev)], 1).double() @ wv0
        depth = float(anchors[:, 2][anchors[:, 2] > 0.2].mean())
    g = torch.Generator().manual_seed(0)
    axis = torch.randn(3, generator=g, dtype=torch.float64)
    move = torch.randn(3, generator=g, dtype=torch.float64)
    delta0 = torch.cat([axis / axis.norm() * math.radians(args.rot_deg), move / move.norm() * args.trans_frac * depth])
    delta = delta0.clone().to(dev).requires_grad_()
    opt = torch.optim.Adam([delta], lr=args.lr)
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, args.steps, eta_min=args.lr * 1e-2)
    rot0, tr0 = pose_error(delta)
    loss0 = None
    for _ in range(args.steps):
        opt.zero_grad(set_to_none=True)
        loss = (image(delta) - target).abs().mean()
        loss.backward()
        opt.step()
        sched.step()
        loss0 = float(loss.detach()) if loss0 is None else loss0
    with torch.no_grad():
        loss1 = float((image(delta) - target).abs().mean())
    rot1, tr1 = pose_error(delta)
    res = {"workload": "c1 (one view, model frozen, eval mode)", "steps": args.steps, "mean_depth": round(depth, 4),
           "rot_err_deg_before": round(rot0, 5), "rot_err_deg_after": round(rot1, 5),
           "trans_err_before": round(tr0, 6), "trans_err_after": round(tr1, 6),
           "l1_before": round(loss0, 6), "l1_after": round(loss1, 6)}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
