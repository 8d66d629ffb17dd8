"""CPU tests of the antialiasing references (tests/antialiasing_oracle.py): the antialiased rasterizer reference against
fp64 autograd of oracle/composite_torch.project -> rho_torch -> composite, and its copy of the colour oracle's chains
pinned to oracle/raster.py (bitwise conic, byte-identical backward with antialiasing off).  Also the scale-consistency
property the feature exists for, on the fp64 composite, which fixes the margin tests/test_antialiasing_gpu.py asserts on
the GPU."""
import numpy as np
import pytest
import torch

from oracle import composite_torch as CT
from oracle import raster as R
from tests import antialiasing_oracle as AA
from tests.camera_grad_ref import clamp_scene
from tests.util import rel_err, scene, tans
from splatco_b200.synthetic import ring_cameras

RHO_MIN32 = np.sqrt(np.float32(2.5e-5))          # the fp32 clamp of the forward record
RHO_MIN64 = float(np.sqrt(2.5e-5))              # the fp64 clamp of the reference backward and AA.rho_torch


def sub_pixel_scene(M, W, H, seed, frac=0.7):
    """`frac` of the Gaussians with screen sigma 0.002-0.01 px (rho clamped) and opacity 0.9-0.99 (so that the clamped
    ones still pass the 1/255 cut near their centre pixel), the rest with sigma 0.5-4 px."""
    cam, means, colors, opac, scales, rots = scene(M, W, H, seed, sigma_px=(0.5, 4.0))
    _, _, _, tiny, _ = scene(M, W, H, seed, sigma_px=(0.002, 0.01))[1:]
    g = torch.Generator().manual_seed(seed + 100)
    pick = torch.rand(M, generator=g) < frac
    scales = torch.where(pick[:, None], tiny, scales).contiguous()
    opac = torch.where(pick[:, None], torch.empty(M, 1).uniform_(0.9, 0.99, generator=g), opac).contiguous()
    return cam, means, colors, opac, scales, rots


def make(kind, seed):
    if kind == "ordinary":
        return scene(300, 64, 48, seed, sigma_px=(0.2, 6.0))
    if kind == "ordinary_small":
        return scene(200, 40, 56, seed, sigma_px=(0.05, 1.5))
    if kind == "rho_clamp":
        return sub_pixel_scene(400, 48, 40, seed)
    cam = ring_cameras(3, 64, 48)[1]                          # "txy_clamp": half beyond the 1.3 tanfov clamp
    return (cam, *clamp_scene(cam, 300, seed, sigma_world=(0.002, 0.2)))


def fp64_reference(cam, means, colors, opac, scales, rots, bg, pr, antialiasing=True):
    """(image, leaf tensors, rho) of the fp64 autograd composite in the oracle's depth order."""
    tx, ty = tans(cam)
    H, W = int(cam.image_height), int(cam.image_width)
    d = torch.float64
    m, c, o, s, q = [t.to(d).requires_grad_() for t in (means, colors, opac, scales, rots)]
    xy, depth, conic, (a, b, cc) = CT.project(m, s, q, 1.0, cam.world_view_transform, cam.full_proj_transform,
                                              tx, ty, H, W)
    rho = AA.rho_torch(a, b, cc)
    op = o.reshape(-1) * rho if antialiasing else o.reshape(-1)
    M = means.shape[0]
    order = torch.tensor(sorted(range(M), key=lambda i: (int(np.float32(pr.depths[i]).view(np.uint32)), i)))
    img = CT.composite(xy, conic, op, c, torch.as_tensor(bg, dtype=d), torch.tensor(pr.rect), order, H, W)
    return img, (m, c, o, s, q), rho


def oracle_fw_bw(cam, means, colors, opac, scales, rots, bg, dL):
    tx, ty = tans(cam)
    H, W = int(cam.image_height), int(cam.image_width)
    V, Pm = cam.world_view_transform.numpy(), cam.full_proj_transform.numpy()
    fw = AA.rasterize_forward(means.numpy(), colors.numpy(), opac.numpy(), scales.numpy(), rots.numpy(), 1.0, V, Pm,
                              tx, ty, H, W, np.asarray(bg, np.float32))
    bw = None
    if dL is not None:
        bw = AA.rasterize_backward(fw, means.numpy(), colors.numpy(), opac.numpy(), scales.numpy(), rots.numpy(), 1.0, V,
                                   Pm, tx, ty, H, W, np.asarray(bg, np.float32), dL)
    return fw, bw


@pytest.mark.parametrize("kind,seed", [("ordinary", 7), ("ordinary_small", 11), ("rho_clamp", 13), ("txy_clamp", 17)])
def test_oracle_aa_backward_matches_fp64_autograd(kind, seed):
    cam, means, colors, opac, scales, rots = make(kind, seed)
    H, W = int(cam.image_height), int(cam.image_width)
    bg = [1.0, 0.5, 0.25]
    fw, _ = oracle_fw_bw(cam, means, colors, opac, scales, rots, bg, None)
    pr = fw["pr"]
    vis = pr.radii > 0
    img, (m, c, o, s, q), rho = fp64_reference(cam, means, colors, opac, scales, rots, bg, pr)
    # the compensated opacity of the record against fp64
    want_op = (o.detach().reshape(-1) * rho.detach()).numpy()
    assert np.abs(pr.conic_opacity[vis, 3] - want_op[vis]).max() < 1e-5
    clamped = vis & (rho.detach().numpy() <= RHO_MIN64 * (1 + 1e-12))
    if kind == "rho_clamp":
        assert clamped.sum() > 0.5 * vis.sum()
        # clamped: exactly opacity * sqrt(2.5e-5) in fp32
        want = opac.numpy().reshape(-1) * RHO_MIN32
        assert np.array_equal(pr.conic_opacity[clamped, 3].view(np.uint32), want[clamped].view(np.uint32))
    err = np.abs(img.detach().numpy() - fw["image"])
    assert err[:, ~fw["fragile"]].max() < 1e-5
    gt = torch.rand(3, H, W, generator=torch.Generator().manual_seed(seed + 1), dtype=torch.float64)
    dL = torch.sign(img.detach() - gt) / (3 * H * W)
    img.backward(dL)
    _, bw = oracle_fw_bw(cam, means, colors, opac, scales, rots, bg, dL.float().numpy())
    tol = 5e-3                       # the oracle's per-pixel blend is fp32 (see test_oracle_raster.py)
    for name, t in (("means3D", m), ("colors", c), ("opacities", o), ("scales", s), ("rotations", q)):
        assert np.abs(t.grad.numpy()).max() > 0, name
        assert rel_err(bw[name], t.grad.numpy()) < tol, (name, rel_err(bw[name], t.grad.numpy()))
    if kind == "rho_clamp":
        live = clamped & (np.abs(bw["opacities"][:, 0]) > 0)
        assert live.sum() > 0, "no clamped Gaussian contributes"


def test_oracle_aa_clamped_everywhere_is_a_constant_factor():
    """rho clamped for every Gaussian: dL/dopacity = rho dL/do' and no rho term reaches the geometry (the geometry
    gradients equal those of the plain backward on the same blend gradients)."""
    cam, means, colors, opac, scales, rots = sub_pixel_scene(300, 48, 40, 5, frac=1.0)
    H, W = int(cam.image_height), int(cam.image_width)
    tx, ty = tans(cam)
    V, Pm = cam.world_view_transform.numpy(), cam.full_proj_transform.numpy()
    pr = AA.preprocess(means.numpy(), scales.numpy(), rots.numpy(), opac.numpy(), 1.0, V, Pm, tx, ty, H, W)
    vis = pr.radii > 0
    assert vis.sum() > 100
    assert np.array_equal(pr.conic_opacity[vis, 3], opac.numpy()[vis, 0] * RHO_MIN32)
    rng = np.random.default_rng(3)
    P = means.shape[0]
    g2, gc, go = rng.normal(size=(P, 3)).astype(np.float32), rng.normal(size=(P, 3)).astype(np.float32), \
        rng.normal(size=(P, 1)).astype(np.float32)
    args = (means.numpy(), scales.numpy(), rots.numpy(), 1.0, V, Pm, tx, ty, H, W, pr.radii, g2, gc)
    plain = R.preprocess_bwd(*args)
    aa = AA.preprocess_bwd(*args, opac.numpy(), go)
    for x, y in zip(plain, aa[:3]):
        assert np.array_equal(x, y)
    assert np.array_equal(aa[3][vis], (go[vis].astype(np.float64) * RHO_MIN64).astype(np.float32))


def test_reference_chains_are_the_colour_oracles():
    """The reference's fp32 projection chain gives oracle.raster.preprocess's conic bit for bit, and its backward with
    antialiasing off gives oracle.raster.preprocess_bwd's outputs byte for byte; with it on, only the record opacity of
    the forward changes."""
    cam, means, colors, opac, scales, rots = sub_pixel_scene(2000, 96, 64, 21, frac=0.5)
    H, W = int(cam.image_height), int(cam.image_width)
    tx, ty = tans(cam)
    V, Pm = cam.world_view_transform.numpy(), cam.full_proj_transform.numpy()
    a = (means.numpy(), scales.numpy(), rots.numpy())
    plain = R.preprocess(*a, opac.numpy(), 1.0, V, Pm, tx, ty, H, W)
    vis = plain.radii > 0
    assert 0 < vis.sum() < vis.size
    rho, conic = AA.rho(*a, 1.0, V, tx, ty, H, W, plain.radii)
    assert conic.tobytes() == plain.conic_opacity[:, :3].tobytes()
    assert (rho[vis] > 0).all() and (rho[vis] < 1).all() and (rho[~vis] == 0).all()
    aa = AA.preprocess(*a, opac.numpy(), 1.0, V, Pm, tx, ty, H, W)
    for f in ("radii", "xy", "depths", "cov3d", "rect", "tiles_touched"):
        assert getattr(aa, f).tobytes() == getattr(plain, f).tobytes(), f
    assert aa.conic_opacity[:, :3].tobytes() == plain.conic_opacity[:, :3].tobytes()
    assert np.array_equal(aa.conic_opacity[vis, 3], opac.numpy()[vis, 0] * rho[vis])
    rng = np.random.default_rng(1)
    P = means.shape[0]
    g2, gc, go = [rng.normal(size=sh).astype(np.float32) for sh in ((P, 3), (P, 3), (P, 1))]
    args = (*a, 1.0, V, Pm, tx, ty, H, W, plain.radii, g2, gc)
    old = R.preprocess_bwd(*args)
    new = AA.preprocess_bwd(*args, opac.numpy(), go, antialiasing=False)
    for x, y in zip(old, new[:3]):
        assert x.tobytes() == y.tobytes()
    assert new[3].tobytes() == go.tobytes()


# ---- scale consistency: what antialiasing is for --------------------------------------------------------------------
def scale_scene(M, W, H, seed):
    """Gaussians of 0.4-2 px at W x H (0.1-0.5 px at a quarter of the resolution), moderate opacity."""
    cam, means, colors, opac, scales, rots = scene(M, W, H, seed, sigma_px=(0.4, 2.0))
    opac = torch.empty(M, 1).uniform_(0.1, 0.6, generator=torch.Generator().manual_seed(seed))
    return cam, means, colors, opac, scales, rots


def box4(img):
    c, h, w = img.shape
    return img.reshape(c, h // 4, 4, w // 4, 4).mean(axis=(2, 4))


def scale_errors_fp64(W=128, H=96, M=1500, seed=3):
    """Mean absolute error of the W/4 x H/4 render against the 4x4 box-downsampled W x H render, fp64 composite,
    for antialiasing off and on (each compared with the full-resolution render of the same setting)."""
    from splatco_b200.synthetic import ring_cameras as rc
    cam_hi, means, colors, opac, scales, rots = scale_scene(M, W, H, seed)
    cam_lo = rc(3, W // 4, H // 4)[1]
    bg = [0.0, 0.0, 0.0]
    out = {}
    for aa in (False, True):
        imgs = []
        for cam in (cam_hi, cam_lo):
            pr = R.preprocess(means.numpy(), scales.numpy(), rots.numpy(), opac.numpy(), 1.0,
                              cam.world_view_transform.numpy(), cam.full_proj_transform.numpy(), *tans(cam),
                              int(cam.image_height), int(cam.image_width))
            with torch.no_grad():
                img, _, _ = fp64_reference(cam, means, colors, opac, scales, rots, bg, pr, antialiasing=aa)
            imgs.append(img.numpy())
        out[aa] = float(np.abs(imgs[1] - box4(imgs[0])).mean())
    return out


def test_antialiasing_makes_the_quarter_resolution_render_consistent():
    e = scale_errors_fp64()
    # measured: off 0.222, on 0.019 (11x closer); tests/test_antialiasing_gpu.py holds the GPU to the same 0.5
    assert e[True] < 0.5 * e[False], e
