"""References for antialiasing (test infrastructure only).

* `preprocess` / `preprocess_bwd` / `rasterize_forward` / `rasterize_backward`: oracle/raster.py's rasterizer with the
  record opacity scaled by rho (tests/antialiasing_oracle.c: rho on the colour oracle's fp32 projection chain, and the
  fp64 preprocess backward with the rho term).  Binning and blend are oracle/raster.py's, unchanged: antialiasing only
  changes the opacity in the record.
* `rho_torch`: rho from the dilated (a, b, c) that oracle/composite_torch.project returns, so fp64 autograd through
  project -> rho_torch -> composite supplies reference gradients.

These live next to the tests instead of extending oracle/: the colour oracle is the fixed reference of the plain path,
which this feature leaves unchanged.  tests/test_oracle_antialiasing.py holds the copy to it: aa_rho's conic equals
oracle.raster.preprocess's bit for bit, and aa_preprocess_bwd with antialiasing off equals oracle.raster.preprocess_bwd
byte for byte.

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

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "antialiasing_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        tag = hashlib.sha256(src).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), f"splatco_antialiasing_oracle_{os.getuid()}_{tag}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}.tmp"
            subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off",
                                   "-fno-fast-math", "-Wall", "-Wextra", "-o", tmp, _SRC, "-lm"])
            os.replace(tmp, so)
        _lib = C.CDLL(so)
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _f32(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float32))


RHO_MIN = 2.5e-5                     # the clamp of det0 / det


def rho(means3D, scales, rots, scale_mod, view, tanfovx, tanfovy, H, W, radii):
    """(rho [P], conic [P,3]) in fp32 on the oracle's projection chain; 0 where radii == 0."""
    means3D, scales, rots, view = _f32(means3D), _f32(scales), _f32(rots), _f32(view).reshape(-1)
    radii = np.ascontiguousarray(radii, dtype=np.int32)
    P = means3D.shape[0]
    r, conic = np.zeros(P, np.float32), np.zeros((P, 3), np.float32)
    rc = lib().aa_rho(C.c_int(P), _p(means3D), _p(scales), C.c_int(3), _p(rots), C.c_float(scale_mod), _p(view),
                      C.c_float(tanfovx), C.c_float(tanfovy), C.c_int(H), C.c_int(W), _p(radii), _p(r), _p(conic))
    assert rc == 0
    return r, conic


def preprocess(means3D, scales, rots, opacities, scale_mod, view, proj, tanfovx, tanfovy, H, W) -> R.Projected:
    """oracle.raster.preprocess with the record opacity opacities * rho (one fp32 multiply, as the kernels)."""
    pr = R.preprocess(means3D, scales, rots, opacities, scale_mod, view, proj, tanfovx, tanfovy, H, W)
    r, _ = rho(means3D, scales, rots, scale_mod, view, tanfovx, tanfovy, H, W, pr.radii)
    vis = pr.radii > 0
    pr.conic_opacity[vis, 3] = _f32(opacities).reshape(-1)[vis] * r[vis]
    return pr


def preprocess_bwd(means3D, scales, rots, scale_mod, view, proj, tanfovx, tanfovy, H, W, radii, g_mean2D, g_conic,
                   opacities, g_opacity, antialiasing=True):
    """(dL/dmeans3D, dL/dscales, dL/drotations, dL/dopacities [P,1]) from the blend's gradients, g_opacity being the one
    with respect to the record opacity.  antialiasing=False: oracle.raster.preprocess_bwd's outputs and g_opacity."""
    means3D, scales, rots = _f32(means3D), _f32(scales), _f32(rots)
    view, proj = _f32(view).reshape(-1), _f32(proj).reshape(-1)
    P = means3D.shape[0]
    gm, gs, gq = np.zeros((P, 3), np.float32), np.zeros((P, 3), np.float32), np.zeros((P, 4), np.float32)
    go = np.zeros((P, 1), np.float32)
    radii, g_mean2D, g_conic = np.ascontiguousarray(radii, dtype=np.int32), _f32(g_mean2D), _f32(g_conic)
    opacities, g_opacity = _f32(opacities).reshape(-1), _f32(g_opacity).reshape(-1)
    rc = lib().aa_preprocess_bwd(C.c_int(P), _p(means3D), _p(scales), C.c_int(3), _p(rots), C.c_float(scale_mod),
                                 _p(view), _p(proj), C.c_float(tanfovx), C.c_float(tanfovy), C.c_int(H), C.c_int(W),
                                 _p(radii), _p(g_mean2D), _p(g_conic), _p(gm), _p(gs), _p(gq), _p(opacities),
                                 _p(g_opacity), _p(go), C.c_int(1 if antialiasing else 0))
    assert rc == 0
    return gm, gs, gq, go


def rasterize_forward(means3D, colors, opacities, scales, rots, scale_mod, view, proj, tanfovx, tanfovy, H, W, bg):
    """oracle.raster.rasterize_forward of the antialiased record."""
    pr = preprocess(means3D, scales, rots, opacities, scale_mod, view, proj, tanfovx, tanfovy, H, W)
    bn = R.binning(pr, H, W)
    img, final_T, n_contrib, fragile = R.blend_fwd(pr, bn, colors, bg, H, W)
    return dict(pr=pr, bn=bn, image=img, final_T=final_T, n_contrib=n_contrib, fragile=fragile)


def rasterize_backward(fw, means3D, colors, opacities, scales, rots, scale_mod, view, proj, tanfovx, tanfovy, H, W, bg,
                       dL_dpix):
    pr, bn = fw["pr"], fw["bn"]
    g_mean2D, g_conic, g_opac, g_color = R.blend_bwd(pr, bn, colors, bg, fw["final_T"], fw["n_contrib"], dL_dpix, H, W)
    gm, gs, gq, go = preprocess_bwd(means3D, scales, rots, scale_mod, view, proj, tanfovx, tanfovy, H, W, pr.radii,
                                    g_mean2D, g_conic, opacities, g_opac)
    return dict(means3D=gm, means2D=g_mean2D, colors=g_color, opacities=go, scales=gs, rotations=gq, conic=g_conic)


def rho_torch(a, b, c):
    """rho from oracle/composite_torch.project's dilated 2D covariance (a, b, c): sqrt(max(2.5e-5, det0 / det)) with
    det0 of (a - 0.3, b, c - 0.3).  Constant (zero gradient) where the clamp is active."""
    a0, c0 = a - 0.3, c - 0.3
    return torch.sqrt(torch.clamp((a0 * c0 - b * b) / (a * c - b * b), min=RHO_MIN))
