"""fp64 references of the camera gradients (dL/dviewmatrix, dL/dprojmatrix) of the rasterizer's preprocess.

* `camera_terms`: the closed form of include/splatco_b200.h's splatco_preprocess_bwd_camera, per Gaussian, in numpy fp64,
  from per-Gaussian upstream gradients (dL/dmean2D in the kernels' NDC scaling, dL/dconic, dL/dz).  Row g, column e is
  Gaussian g's contribution to entry e of [view (16) | proj (16)]; the sum over rows is the gradient, the sum of the
  absolute values the scale S_e that bounds fp32 rounding in a sum of that many terms.
* `project_camera_grads`: torch.autograd through oracle/composite_torch.project in fp64 with the same upstream gradients
  (dL_dconic in the kernels' convention, see there).
* `clamp_scene`: Gaussians of which half sit beyond the 1.3 tanfov clamp of the EWA Jacobian, large enough to reach
  into the image."""
from __future__ import annotations

import numpy as np
import torch

from oracle import composite_torch as CT


def quat_rot(q):
    r, x, y, z = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    return np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y),
                     2 * (x * y + r * z), 1 - 2 * (x * x + z * z), 2 * (y * z - r * x),
                     2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], axis=1).reshape(-1, 3, 3)


def camera_terms(means, scales, rots, mod, view, proj, tanfovx, tanfovy, H, W, g2, gconic, gdepth=None):
    """[P, 32] fp64 per-Gaussian contributions.  g2: [P,>=2] dL/dndc (the kernels' dL_dmean2D), gconic [P,3], gdepth [P]
    or None.  Rows with zero upstream gradients contribute zero; the caller zeroes culled Gaussians' rows."""
    f = lambda a: np.asarray(a, np.float64)
    p, s, q = f(means), f(scales)[:, :3] * mod, f(rots)
    V, Pm = f(view).reshape(16), f(proj).reshape(16)
    P = p.shape[0]
    ph = np.concatenate([p, np.ones((P, 1))], axis=1)
    Vm, Pmm = V.reshape(4, 4), Pm.reshape(4, 4)
    pv, hom = ph @ Vm, ph @ Pmm
    M = quat_rot(q) * s[:, None, :]
    S = M @ M.transpose(0, 2, 1)
    fx, fy = W / (2.0 * tanfovx), H / (2.0 * tanfovy)
    limx, limy = 1.3 * tanfovx, 1.3 * tanfovy
    vz = pv[:, 2]
    txtz, tytz = pv[:, 0] / vz, pv[:, 1] / vz
    clx, cly = np.abs(txtz) > limx, np.abs(tytz) > limy
    tx, ty = np.clip(txtz, -limx, limx) * vz, np.clip(tytz, -limy, limy) * vz
    J00, J02, J11, J12 = fx / vz, -fx * tx / vz ** 2, fy / vz, -fy * ty / vz ** 2
    Rot = Vm[:3, :3].T                                   # Rot[r][k] = V[4k + r]
    A = np.zeros((P, 2, 3))
    A[:, 0] = J00[:, None] * Rot[0][None] + J02[:, None] * Rot[2][None]
    A[:, 1] = J11[:, None] * Rot[1][None] + J12[:, None] * Rot[2][None]
    B = A @ S
    cov = B @ A.transpose(0, 2, 1)
    a, b, c = cov[:, 0, 0] + 0.3, cov[:, 0, 1], cov[:, 1, 1] + 0.3
    den = a * c - b * b
    gc = f(gconic)
    # conic = (c, -b, a) / den
    da = (-c * c * gc[:, 0] + 2 * b * c * gc[:, 1] + (den - a * c) * gc[:, 2]) / den ** 2
    dc = (-a * a * gc[:, 2] + 2 * a * b * gc[:, 1] + (den - a * c) * gc[:, 0]) / den ** 2
    db = 2 * (b * c * gc[:, 0] - (den + 2 * b * b) * gc[:, 1] + a * b * gc[:, 2]) / den ** 2
    G2 = np.stack([da, 0.5 * db, 0.5 * db, dc], axis=1).reshape(P, 2, 2)
    dA = 2 * G2 @ B                                      # dL/dA
    dJ00 = (dA[:, 0] * Rot[0][None]).sum(1)
    dJ02 = (dA[:, 0] * Rot[2][None]).sum(1)
    dJ11 = (dA[:, 1] * Rot[1][None]).sum(1)
    dJ12 = (dA[:, 1] * Rot[2][None]).sum(1)
    dtx = np.where(clx, 0.0, -fx / vz ** 2 * dJ02)
    dty = np.where(cly, 0.0, -fy / vz ** 2 * dJ12)
    dtz = -fx / vz ** 2 * dJ00 - fy / vz ** 2 * dJ11 + 2 * fx * tx / vz ** 3 * dJ02 + 2 * fy * ty / vz ** 3 * dJ12
    if gdepth is not None:
        dtz = dtz + f(gdepth).reshape(P)
    g = np.stack([dtx, dty, dtz], axis=1)
    out = np.zeros((P, 32))
    for k in range(4):
        out[:, 4 * k:4 * k + 3] = g * ph[:, k:k + 1]
    for k in range(3):
        out[:, 4 * k] += dA[:, 0, k] * J00
        out[:, 4 * k + 1] += dA[:, 1, k] * J11
        out[:, 4 * k + 2] += dA[:, 0, k] * J02 + dA[:, 1, k] * J12
    mw = 1.0 / (hom[:, 3] + 1e-7)
    g2 = f(g2)
    e = np.stack([g2[:, 0] * mw, g2[:, 1] * mw, -(g2[:, 0] * hom[:, 0] + g2[:, 1] * hom[:, 1]) * mw * mw], axis=1)
    for k in range(4):
        out[:, 16 + 4 * k] = e[:, 0] * ph[:, k]
        out[:, 16 + 4 * k + 1] = e[:, 1] * ph[:, k]
        out[:, 16 + 4 * k + 3] = e[:, 2] * ph[:, k]
    return out


def project_camera_grads(means, scales, rots, mod, view, proj, tanfovx, tanfovy, H, W, g2, gconic, gdepth=None):
    """(dL/dview [16], dL/dproj [16]) in fp64 by autograd through oracle/composite_torch.project, for the same upstream
    gradients as `camera_terms` (g2 in NDC scaling, converted here to the pixel coordinates project() returns)."""
    d = torch.float64
    t = lambda a: torch.as_tensor(np.asarray(a, np.float64), dtype=d)
    v = t(view).reshape(4, 4).requires_grad_()
    pm = t(proj).reshape(4, 4).requires_grad_()
    xy, tz, conic, _ = CT.project(t(means), t(scales)[:, :3], t(rots), mod, v, pm, tanfovx, tanfovy, H, W)
    g_xy = t(g2)[:, :2] / torch.tensor([0.5 * W, 0.5 * H], dtype=d)
    # the blend kernels' dL_dconic[1] is half of dL/dconic[1] (the reference rasterizer's convention, undone by the
    # factor 2 in the preprocess backward's dL_db)
    g_conic = t(gconic) * torch.tensor([1.0, 2.0, 1.0], dtype=d)
    outs, grads = [xy, conic], [g_xy, g_conic]
    if gdepth is not None:
        outs.append(tz)
        grads.append(t(gdepth).reshape(-1))
    gv, gp = torch.autograd.grad(outs, [v, pm], grads, allow_unused=True)
    z = lambda g: np.zeros(16) if g is None else g.reshape(16).numpy()
    return z(gv), z(gp)


def clamp_scene(cam, P, seed, frac=0.5, k=(1.35, 1.8), z=(2.0, 5.0), sigma_world=(0.15, 0.4)):
    """World-space Gaussians for `cam` (a splatco_b200.synthetic camera): a fraction `frac` at |x/z| or |y/z| between
    k[0] and k[1] times tanfov (the clamp of the EWA Jacobian is active), the rest inside the frustum."""
    import math
    rng = np.random.default_rng(seed)
    tx, ty = math.tan(cam.FoVx * 0.5), math.tan(cam.FoVy * 0.5)
    zz = rng.uniform(*z, P)
    u, v = rng.uniform(-0.9, 0.9, P), rng.uniform(-0.9, 0.9, P)
    out = rng.random(P) < frac
    side = rng.choice([-1.0, 1.0], P)
    kk = rng.uniform(*k, P)
    on_x = rng.random(P) < 0.5
    u = np.where(out & on_x, side * kk, u)
    v = np.where(out & ~on_x, side * kk, v)
    pv = np.stack([u * tx * zz, v * ty * zz, zz, np.ones(P)], axis=1)
    Vm = cam.world_view_transform.numpy().astype(np.float64)
    world = pv @ np.linalg.inv(Vm)
    means = world[:, :3].astype(np.float32)
    scales = np.exp(rng.uniform(np.log(sigma_world[0]), np.log(sigma_world[1]), (P, 3))).astype(np.float32)
    q = rng.normal(size=(P, 4))
    rots = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)
    colors = rng.uniform(0, 1, (P, 3)).astype(np.float32)
    opac = rng.uniform(0.2, 0.9, (P, 1)).astype(np.float32)
    return [torch.from_numpy(a) for a in (means, colors, opac, scales, rots)]


def se3_exp(delta):
    """4x4 exp of the twist delta = (omega [3], t [3]) (torch, differentiable, any dtype)."""
    w, t = delta[:3], delta[3:]
    z = delta.new_zeros(())
    X = torch.stack([torch.stack([z, -w[2], w[1], t[0]]), torch.stack([w[2], z, -w[0], t[1]]),
                     torch.stack([-w[1], w[0], z, t[2]]), torch.stack([z, z, z, z])])
    return torch.linalg.matrix_exp(X)


def posed_matrices(wv0, full0, delta):
    """(world_view_transform, full_proj_transform, camera_center) of the camera whose world->camera transform is
    exp(delta) applied after the one of (wv0, full0) -- the row-vector convention of the reference's Camera:
    wv = wv0 @ exp(delta)^T, full = wv @ proj, centre = wv^-1[3, :3]."""
    proj = torch.linalg.solve(wv0, full0)
    wv = wv0 @ se3_exp(delta).transpose(0, 1)
    return wv, wv @ proj, torch.linalg.inv(wv)[3, :3]
