"""CPU tests of the depth / alpha references and of the new entry points' argument checks.

The C reference (tests/depth_alpha_oracle.c) is checked against an independent fp64 autograd composite, the way
tests/test_oracle_raster.py checks the colour oracle; the GPU kernels are then compared against the C reference
(tests/test_depth_alpha_gpu.py)."""
import numpy as np
import pytest
import torch

from oracle import composite_torch as CT
from oracle import raster as R
from splatco_b200 import _lib
from tests import depth_alpha_oracle as DA
from tests.util import rel_err, scene, tans

SCENES = [(7, 64, 48, 300, (1.0, 6.0)), (11, 40, 56, 200, (0.5, 3.0)), (13, 33, 17, 120, (2.0, 10.0))]


def _forward(cam, means, colors, opac, scales, rots, bg):
    tx, ty = tans(cam)
    return DA.rasterize_forward(means.numpy(), colors.numpy(), opac.numpy(), scales.numpy(), rots.numpy(), 1.0,
                                cam.world_view_transform.numpy(), cam.full_proj_transform.numpy(), tx, ty,
                                cam.image_height, cam.image_width, np.asarray(bg, np.float32))


@pytest.mark.parametrize("upstream", ["depth", "alpha", "all"])
@pytest.mark.parametrize("seed,W,H,M,sig", SCENES)
def test_depth_alpha_oracle_matches_fp64_autograd_composite(seed, W, H, M, sig, upstream):
    cam, means, colors, opac, scales, rots = scene(M, W, H, seed, sigma_px=sig)
    bg = torch.tensor([1.0, 0.5, 0.25])
    fw = _forward(cam, means, colors, opac, scales, rots, bg.numpy())
    pr = fw["pr"]
    # the colour walk is the colour oracle's, bit for bit
    img0, T0, n0, _ = R.blend_fwd(pr, fw["bn"], colors.numpy(), bg.numpy(), H, W)
    assert np.array_equal(img0, fw["image"]) and np.array_equal(T0, fw["final_T"]) and np.array_equal(n0, fw["n_contrib"])
    assert np.array_equal(fw["alpha"], (np.float32(1) - fw["final_T"]).astype(np.float32))

    tx, ty = tans(cam)
    d = torch.float64
    m, c, o, s, q = [t.to(d).requires_grad_() for t in (means, colors, opac, scales, rots)]
    xy, tz, conic, _ = CT.project(m, s, q, 1.0, cam.world_view_transform, cam.full_proj_transform, tx, ty, H, W)
    order = torch.tensor(sorted(range(M), key=lambda i: (int(np.float32(pr.depths[i]).view(np.uint32)), i)))
    img, dep, alp = DA.composite_depth_alpha(xy, tz, conic, o, c, bg, torch.tensor(pr.rect), order, H, W)
    frag = fw["fragile"]
    assert frag.mean() < 0.05
    zmax = float(np.abs(pr.depths[pr.radii > 0]).max())
    assert np.abs(alp.detach().numpy()[0] - fw["alpha"])[~frag].max() < 1e-5
    assert np.abs(dep.detach().numpy()[0] - fw["depth"])[~frag].max() < 1e-5 * zmax
    assert np.abs(img.detach().numpy() - fw["image"])[:, ~frag].max() < 1e-5

    g = torch.Generator().manual_seed(seed + 2)
    gD = torch.randn(1, H, W, generator=g, dtype=d) / (H * W) if upstream in ("depth", "all") else None
    gA = torch.randn(1, H, W, generator=g, dtype=d) / (H * W) if upstream in ("alpha", "all") else None
    gC = torch.randn(3, H, W, generator=g, dtype=d) / (H * W) if upstream == "all" else None
    outs, grads = zip(*[(t, gt) for t, gt in ((img, gC), (dep, gD), (alp, gA)) if gt is not None])
    torch.autograd.backward(outs, grads)
    f32 = lambda t: None if t is None else t.float().numpy()
    bw = DA.rasterize_backward(fw, means.numpy(), colors.numpy(), scales.numpy(), rots.numpy(), 1.0,
                               cam.world_view_transform.numpy(), cam.full_proj_transform.numpy(), tx, ty, H, W,
                               bg.numpy(), dL_dpix=f32(gC), dL_ddepth=f32(gD), dL_dalpha=f32(gA))
    tol = 5e-3        # fp32 per-pixel blend against fp64 autograd (the bar of tests/test_oracle_raster.py)
    assert rel_err(bw["means3D"], m.grad.numpy()) < tol
    assert rel_err(bw["opacities"], o.grad.numpy()) < tol
    assert rel_err(bw["scales"], s.grad.numpy()) < tol
    assert rel_err(bw["rotations"], q.grad.numpy()) < tol
    if upstream == "all":
        assert rel_err(bw["colors"], c.grad.numpy()) < tol
    else:
        assert not np.any(bw["colors"]) and (c.grad is None or not torch.any(c.grad))


@pytest.mark.parametrize("seed,W,H,M,sig", SCENES[:2])
def test_depth_alpha_oracle_equals_colour_oracle_without_map_gradients(seed, W, H, M, sig):
    """The depth / alpha reference repeats the colour oracle's walk; with no depth / alpha gradient its colour forward and
    its whole backward must be the colour oracle's.  Both run single-threaded so their fp64 sums add in the same order."""
    cam, means, colors, opac, scales, rots = scene(M, W, H, seed, sigma_px=sig)
    bg = np.array([1.0, 0.5, 0.25], np.float32)
    tx, ty = tans(cam)
    view, proj = cam.world_view_transform.numpy(), cam.full_proj_transform.numpy()
    args = (means.numpy(), colors.numpy(), scales.numpy(), rots.numpy(), 1.0, view, proj, tx, ty, H, W, bg)
    dL = (np.random.default_rng(seed).standard_normal((3, H, W)) / (3 * H * W)).astype(np.float32)
    R.lib().oracle_set_threads(1)
    DA.lib().da_set_threads(1)
    try:
        fw = _forward(cam, means, colors, opac, scales, rots, bg)
        fw0 = R.rasterize_forward(means.numpy(), colors.numpy(), opac.numpy(), scales.numpy(), rots.numpy(), 1.0, view,
                                  proj, tx, ty, H, W, bg)
        for k in ("image", "final_T", "n_contrib", "fragile"):
            assert np.array_equal(fw[k], fw0[k]), k
        got = DA.rasterize_backward(fw, *args, dL_dpix=dL)
        want = R.rasterize_backward(fw0, *args, dL)
    finally:
        R.lib().oracle_set_threads(0)
        DA.lib().da_set_threads(0)
    for k in ("means3D", "means2D", "colors", "opacities", "scales", "rotations", "conic"):
        assert np.array_equal(got[k], want[k]), k
    assert not np.any(got["depth"])


def test_depth_is_z_times_alpha_when_every_gaussian_shares_one_z():
    """With one z for every Gaussian, depth = z * sum(alpha T) = z * (1 - T_final) = z * alpha."""
    cam, means, colors, opac, scales, rots = scene(400, 48, 40, 17, sigma_px=(1.0, 6.0))
    tx, ty = tans(cam)
    H, W = 40, 48
    pr = R.preprocess(means.numpy(), scales.numpy(), rots.numpy(), opac.numpy(), 1.0, cam.world_view_transform.numpy(),
                      cam.full_proj_transform.numpy(), tx, ty, H, W)
    bn = R.binning(pr, H, W)
    z = np.float32(3.25)
    pr.depths[:] = z                           # after binning: the walk order is unchanged, only the z the blend reads
    img, T, n, depth, alpha, _ = DA.blend_fwd(pr, bn, colors.numpy(), np.ones(3, np.float32), H, W)
    assert (alpha > 0.5).mean() > 0.2
    # sum(alpha T) and 1 - T_final are the same quantity, rounded differently in fp32 over up to n_contrib steps
    tol = 4 * np.finfo(np.float32).eps * np.maximum(n, 1) * z
    assert np.all(np.abs(depth - z * alpha) <= tol)


def test_depth_alpha_entry_points_validate_arguments_without_gpu():
    L = _lib.lib()
    err = lambda: L.splatco_last_error().decode()
    nz = _lib.C.c_void_p(16)                 # never dereferenced: every call below is refused before device work
    # forward
    assert L.splatco_blend_fwd_depth_alpha(-1, 8, 8, nz, nz, nz, nz, nz, nz, nz, None) < 0 and "bad sizes" in err()
    assert L.splatco_blend_fwd_depth_alpha(0, 0, 8, nz, nz, nz, nz, nz, nz, nz, None) < 0 and "bad sizes" in err()
    assert L.splatco_blend_fwd_depth_alpha(0, 8, 8, nz, nz, nz, nz, nz, None, nz, None) < 0 and "null pointer" in err()
    assert L.splatco_blend_fwd_depth_alpha(0, 8, 8, nz, nz, nz, nz, nz, nz, None, None) < 0 and "null pointer" in err()
    assert L.splatco_blend_fwd_depth_alpha(5, 8, 8, nz, None, nz, nz, nz, nz, nz, None) < 0 and "null workspace" in err()
    assert L.splatco_blend_fwd_depth_alpha(5, 8, 8, nz, nz, None, nz, nz, nz, nz, None) < 0 and "null workspace" in err()
    # backward
    bwd = L.splatco_blend_bwd_depth_alpha
    g = [nz] * 5
    assert bwd(-1, 5, 8, 8, nz, nz, nz, nz, nz, nz, nz, *g, None) < 0 and "bad sizes" in err()
    assert bwd(4, 5, 8, -8, nz, nz, nz, nz, nz, nz, nz, *g, None) < 0 and "bad sizes" in err()
    assert bwd(4, 5, 8, 8, nz, nz, nz, nz, None, None, None, *g, None) < 0 and "all three" in err()
    assert bwd(0, 0, 8, 8, nz, nz, nz, nz, None, None, None, *g, None) < 0 and "all three" in err()
    assert bwd(4, 5, 8, 8, nz, None, nz, nz, nz, None, None, *g, None) < 0 and "null pointer" in err()
    assert bwd(4, 5, 8, 8, nz, nz, None, nz, None, nz, None, *g, None) < 0 and "null pointer" in err()
    assert bwd(4, 5, 8, 8, nz, nz, nz, nz, None, None, nz, nz, nz, nz, nz, None, None) < 0 and "null pointer" in err()
    assert bwd(0, 5, 8, 8, nz, nz, nz, nz, nz, None, None, *g, None) == 0           # nothing to do is not an error
    # preprocess backward with the depth term
    pre = L.splatco_preprocess_bwd_depth
    args = [nz, nz, 3, nz, 1.0, nz, nz, 1.0, 1.0, 8, 8, nz, nz, nz, nz, nz, nz]
    assert pre(-1, *args, nz, None) < 0 and "preprocess_bwd_depth: bad sizes" in err()
    assert pre(4, *args, None, None) < 0 and "preprocess_bwd_depth: null pointer" in err()
    a2 = list(args); a2[0] = None
    assert pre(4, *a2, nz, None) < 0 and "null pointer" in err()
    assert pre(0, *args, None, None) == 0
    # the colour-only entry point keeps its messages
    assert L.splatco_preprocess_bwd(-1, *args, None) < 0 and "preprocess_bwd: bad sizes" in err()
