"""CPU tests of the camera-gradient references (tests/camera_grad_ref.py), the closed forms the GPU kernels implement:

* dL/dviewmatrix and dL/dprojmatrix of the preprocess: the per-Gaussian closed form summed in fp64 equals autograd
  through oracle/composite_torch.project, with and without a depth term, and on a scene where half the Gaussians are
  beyond the 1.3 tanfov clamp;
* dL/dcamera_center of the decode: minus the sum over visible anchors of the direction / distance gradient the decode
  backward adds to dL/danchor equals autograd of oracle/decode_oracle.decode with respect to cam_center."""
import os

import numpy as np
import pytest
import torch

from oracle import decode_oracle as D
from splatco_b200.synthetic import ring_cameras
from tests.camera_grad_ref import camera_terms, clamp_scene, project_camera_grads
from tests.util import scene, tans

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
UNUSED = [3, 7, 11, 15, 16 + 2, 16 + 6, 16 + 10, 16 + 14]


def _upstream(P, W, H, seed, depth):
    g = np.random.default_rng(seed)
    g2 = g.normal(size=(P, 3)) * np.array([0.5 * W, 0.5 * H, 0.0]) * 1e-3
    gc = g.normal(size=(P, 3)) * 1e-2
    gd = g.normal(size=P) * 1e-2 if depth else None
    return g2, gc, gd


@pytest.mark.parametrize("depth", [False, True])
@pytest.mark.parametrize("kind", ["random", "clamped"])
def test_closed_form_equals_autograd_through_project(kind, depth):
    W, H, P = 128, 96, 600
    if kind == "random":
        cam, means, colors, opac, scales, rots = scene(P, W, H, 5, sigma_px=(0.5, 8.0))
    else:
        cam = ring_cameras(3, W, H)[1]
        means, colors, opac, scales, rots = clamp_scene(cam, P, 5)
    tx, ty = tans(cam)
    view, proj = cam.world_view_transform.numpy(), cam.full_proj_transform.numpy()
    pv = np.concatenate([means.numpy(), np.ones((P, 1), np.float32)], 1).astype(np.float64) @ view.astype(np.float64)
    keep = pv[:, 2] > 0.2
    if kind == "clamped":
        lim = 1.3 * np.array([tx, ty])
        assert (np.abs(pv[keep, :2] / pv[keep, 2:3]) > lim).any(axis=1).mean() > 0.35
    g2, gc, gd = _upstream(P, W, H, 7, depth)
    g2[~keep], gc[~keep] = 0.0, 0.0
    if gd is not None:
        gd[~keep] = 0.0
    sel = lambda a: None if a is None else a[keep]
    args = (means.numpy()[keep], scales.numpy()[keep], rots.numpy()[keep], 1.0, view, proj, tx, ty, H, W,
            g2[keep], gc[keep], sel(gd))
    terms = camera_terms(*args)
    got = terms.sum(0)
    gv, gp = project_camera_grads(*args)
    want = np.concatenate([gv, gp])
    S = np.abs(terms).sum(0)
    assert np.all(got[UNUSED] == 0.0) and np.all(want[UNUSED] == 0.0)
    assert np.all(np.abs(got - want) <= 1e-10 * S + 1e-14), np.abs(got - want) / np.maximum(S, 1e-30)
    assert S[2] > 0 and S[16] > 0 and S[16 + 15] > 0


def _dir_grads_via_mlp_inputs(monkeypatch):
    """Record dL/d(MLP input) of every head call (decode_oracle.mlp): its columns 32..35 are dir (3) and dist (1)."""
    seen = []
    orig = D.mlp

    def mlp(p, name, x, act):
        xi = x.view_as(x)                # one node per head call (opacity and cov share x)
        xi.retain_grad()
        seen.append(xi)
        return orig(p, name, xi, act)

    monkeypatch.setattr(D, "mlp", mlp)
    return seen


@pytest.mark.parametrize("tag", ["base", "variants"])
@pytest.mark.parametrize("level", [0, 2])
def test_decode_camera_gradient_is_minus_the_sum_of_the_direction_terms(tag, level, monkeypatch):
    d = np.load(os.path.join(GOLD, f"decode_{tag}.npz"))
    dd = torch.float64
    p = {k[len("param."):]: torch.from_numpy(d[k]).to(dd if d[k].dtype == np.float32 else None) for k in d.files
         if k.startswith("param.")}
    ins = {k: torch.from_numpy(d[f"in.{k}"]).to(dd) for k in ("_anchor", "_offset", "_anchor_feat", "_scaling")}
    cam = torch.from_numpy(d["cam_center"]).to(dd).requires_grad_()
    seen = _dir_grads_via_mlp_inputs(monkeypatch)
    vis = torch.from_numpy(d["vis"])
    dists = bool(d["dists"])
    outs = D.decode(p, ins["_anchor_feat"], ins["_anchor"], ins["_offset"], torch.exp(ins["_scaling"]), vis, cam, level,
                    int(d["K"]), appearance_dim=int(d["appearance_dim"]), uid=int(d["uid"]), dists=dists)
    loss = sum((t * torch.from_numpy(d[f"L{level}.w.{nm}"]).to(dd)).sum()
               for nm, t in zip(["xyz", "color", "opacity", "scaling", "rot"], outs[:5]))
    loss.backward()
    assert len(seen) == 3
    g = sum(x.grad[:, 32:35] for x in seen).numpy()
    gdist = sum(x.grad[:, 35] for x in seen).numpy() if dists else np.zeros(g.shape[0])
    anc = ins["_anchor"][vis].numpy()
    ob = anc - cam.detach().numpy()[None]
    dist = np.linalg.norm(ob, axis=1, keepdims=True)
    dr = ob / dist
    dot = (dr * g).sum(1, keepdims=True)
    dv = (g - dr * dot) / dist + gdist[:, None] * dr
    want = cam.grad.numpy()
    got = -dv.sum(0)
    assert np.abs(want).max() > 0
    assert np.abs(got - want).max() <= 1e-10 * np.abs(dv).sum(0).max()
