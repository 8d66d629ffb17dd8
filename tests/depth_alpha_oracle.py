"""References for the depth and alpha maps (test infrastructure only).

* `blend_fwd` / `blend_bwd` / `preprocess_bwd_depth`: the C oracle's blend (oracle/raster_oracle.c) with the depth
  channel and the alpha map added (tests/depth_alpha_oracle.c); fp32 per pixel, fp64 gradient sums.  The colour,
  final_T and n_contrib it returns are those of oracle.raster.blend_fwd.
* `composite_depth_alpha`: oracle/composite_torch.composite's walk returning (image, depth, alpha), with depth taken
  from project()'s differentiable view-space z, so fp64 autograd supplies reference gradients including the route
  through means3D.

These live next to the tests instead of extending oracle/: the colour oracle is the fixed reference of the colour
path, which this feature leaves unchanged.  tests/test_oracle_depth_alpha.py holds the copy to it: with the depth and
alpha gradients absent, forward and backward here equal oracle/raster.py's exactly.

The C library is compiled on first use into a temporary directory (the tree may be read-only)."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import torch

from oracle import raster as R

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "depth_alpha_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        tag = hashlib.sha256(src).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"splatco_depth_alpha_oracle_{os.getuid()}_{tag}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off",
                                   "-fno-fast-math", "-pthread", "-Wall", "-Wextra", "-o", tmp, _SRC, "-lm"])
            os.replace(tmp, so)
        _lib = C.CDLL(so)
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f32(a):
    return None if a is None else np.ascontiguousarray(np.asarray(a, dtype=np.float32))


def blend_fwd(pr, bn, colors, bg, H, W):
    """(image [3,H,W], final_T [H,W], n_contrib [H,W], depth [H,W], alpha [H,W], fragile [H,W])."""
    colors, bg = _f32(colors), _f32(bg)
    out = np.zeros((3, H, W), np.float32)
    final_T = np.zeros((H, W), np.float32)
    n_contrib = np.zeros((H, W), np.int32)
    depth = np.zeros((H, W), np.float32)
    alpha = np.zeros((H, W), np.float32)
    fragile = np.zeros((H, W), np.uint8)
    pl = bn.point_list if bn.R > 0 else np.zeros(1, np.uint32)
    rc = lib().da_blend_fwd(C.c_int(H), C.c_int(W), _p(bn.ranges), _p(pl), _p(pr.xy), _p(pr.conic_opacity), _p(colors),
                            _p(_f32(pr.depths)), _p(bg), _p(out), _p(final_T), _p(n_contrib), _p(depth), _p(alpha),
                            _p(fragile))
    assert rc == 0
    return out, final_T, n_contrib, depth, alpha, fragile.astype(bool)


def blend_bwd(pr, bn, colors, bg, final_T, n_contrib, dL_dpix, dL_ddepth, dL_dalpha, H, W):
    """Any of dL_dpix [3,H,W], dL_ddepth [H,W], dL_dalpha [H,W] may be None.
    Returns (dL_dmean2D, dL_dconic, dL_dopacity, dL_dcolor, dL_dz [P])."""
    P = pr.radii.shape[0]
    g_mean2D = np.zeros((P, 3), np.float32)
    g_conic = np.zeros((P, 3), np.float32)
    g_opac = np.zeros((P, 1), np.float32)
    g_color = np.zeros((P, 3), np.float32)
    g_z = np.zeros(P, np.float32)
    pl = bn.point_list if bn.R > 0 else np.zeros(1, np.uint32)
    maps = [_f32(dL_dpix), None if dL_ddepth is None else _f32(dL_ddepth).reshape(H, W),
            None if dL_dalpha is None else _f32(dL_dalpha).reshape(H, W)]
    rc = lib().da_blend_bwd(C.c_int(P), C.c_int(H), C.c_int(W), _p(bn.ranges), _p(pl), _p(pr.xy), _p(pr.conic_opacity),
                            _p(_f32(colors)), _p(_f32(pr.depths)), _p(_f32(bg)), _p(_f32(final_T)),
                            _p(np.ascontiguousarray(n_contrib, dtype=np.int32)), *[_p(m) for m in maps],
                            _p(g_mean2D), _p(g_conic), _p(g_opac), _p(g_color), _p(g_z))
    assert rc == 0
    return g_mean2D, g_conic, g_opac, g_color, g_z


def preprocess_bwd_depth(means3D, scales, rots, scale_mod, view, proj, tanfovx, tanfovy, H, W, radii, g_mean2D, g_conic,
                         g_z):
    """oracle.raster.preprocess_bwd plus dL/dz_view . (view[2], view[6], view[10]) on dL/dmeans3D (fp32)."""
    gm, gs, gq = R.preprocess_bwd(means3D, scales, rots, scale_mod, view, proj, tanfovx, tanfovy, H, W, radii,
                                  g_mean2D, g_conic)
    v = _f32(view).reshape(-1)
    dz_dmean = v[[2, 6, 10]]
    gz = np.where(np.asarray(radii) > 0, _f32(g_z), np.float32(0))
    gm = (gm + gz[:, None] * dz_dmean[None, :]).astype(np.float32)
    return gm, gs, gq


def rasterize_forward(means3D, colors, opacities, scales, rots, scale_mod, view, proj, tanfovx, tanfovy, H, W, bg):
    pr = R.preprocess(means3D, scales, rots, opacities, scale_mod, view, proj, tanfovx, tanfovy, H, W)
    bn = R.binning(pr, H, W)
    img, final_T, n_contrib, depth, alpha, fragile = blend_fwd(pr, bn, colors, bg, H, W)
    return dict(pr=pr, bn=bn, image=img, final_T=final_T, n_contrib=n_contrib, depth=depth, alpha=alpha,
                fragile=fragile)


def rasterize_backward(fw, means3D, colors, scales, rots, scale_mod, view, proj, tanfovx, tanfovy, H, W, bg,
                       dL_dpix=None, dL_ddepth=None, dL_dalpha=None):
    pr, bn = fw["pr"], fw["bn"]
    g_mean2D, g_conic, g_opac, g_color, g_z = blend_bwd(pr, bn, colors, bg, fw["final_T"], fw["n_contrib"], dL_dpix,
                                                        dL_ddepth, dL_dalpha, H, W)
    gm, gs, gq = preprocess_bwd_depth(means3D, scales, rots, scale_mod, view, proj, tanfovx, tanfovy, H, W, pr.radii,
                                      g_mean2D, g_conic, g_z)
    return dict(means3D=gm, means2D=g_mean2D, colors=g_color, opacities=g_opac, scales=gs, rotations=gq,
                conic=g_conic, depth=g_z)


def composite_depth_alpha(xy, tz, conic, opacities, colors, bg, rect, order, H, W):
    """oracle/composite_torch.composite's front-to-back walk, also returning depth = sum z alpha T (background 0) and
    alpha = 1 - T_final.  tz: project()'s view-space depth [P]."""
    dt = xy.dtype
    ys, xs = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    tx_, ty_ = xs // 16, ys // 16
    pxf, pyf = xs.to(dt), ys.to(dt)
    T = torch.ones(H, W, dtype=dt)
    Cc = torch.zeros(3, H, W, dtype=dt)
    D = torch.zeros(H, W, dtype=dt)
    done = torch.zeros(H, W, dtype=torch.bool)
    opac = opacities.reshape(-1)
    for g in order.tolist():
        r0x, r0y, r1x, r1y = rect[g].tolist()
        if (r1x - r0x) * (r1y - r0y) == 0:
            continue
        inside = (tx_ >= r0x) & (tx_ < r1x) & (ty_ >= r0y) & (ty_ < r1y) & ~done
        if not bool(inside.any()):
            continue
        dx, dy = xy[g, 0] - pxf, xy[g, 1] - pyf
        power = -0.5 * (conic[g, 0] * dx * dx + conic[g, 2] * dy * dy) - conic[g, 1] * dx * dy
        ea = opac[g] * torch.exp(power)
        alpha = ea + (torch.clamp(ea, max=0.99) - ea).detach()   # the gradient is kept through the clamp
        live = inside & (power <= 0) & (alpha >= 1.0 / 255.0)
        test_T = T * (1 - alpha)
        stop = live & (test_T < 0.0001)
        done = done | stop
        live = live & ~stop
        w = torch.where(live, alpha * T, torch.zeros_like(T))
        Cc = Cc + colors[g][:, None, None] * w[None]
        D = D + tz[g] * w
        T = torch.where(live, test_T, T)
    return Cc + T[None] * bg.to(dt)[:, None, None], D[None], (1 - T)[None]
