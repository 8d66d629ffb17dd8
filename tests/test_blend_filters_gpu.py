"""The blend kernels' cull filters against the kernels' own per-pixel alpha test.

Every blend kernel decides per (pixel, splat) pair with the same fp32 test (`eval_p2` in csrc/blend.cu):
    p2 = fma(c2 dy, dy, fma(a2, dx, b2 dy) dx) <= 0   and   e = p2 + log2(op) >= log2(1/255)
and in front of it sits a filter that must only remove pairs this test rejects: the per-row spans of
`splat_patch_words` (blend_fwd2) and the bounding-box patch masks of `splat_setup` (blend_fwd, both backwards).
The filters solve the conic's quadratic from det = a2 c2 - b2^2 / 4, which cancels for needle-shaped splats,
so they are checked here against an independent reference: the pair test recomputed bit for bit in numpy
from the fp32 records the kernels consumed (read back from the geometry workspace), the front-to-back walk
and the upstream per-pixel gradient formulas (the ones oracle/raster_oracle.c implements) in fp64.

Pixels where a pair sits so close to a cut that the kernels' approximate log2 / ex2 may legitimately decide
it either way are `undecided`: excluded from the image comparison, given dL/dpixel = 0 in the backward, and
held to a small share of the image.
"""
import math

import numpy as np
import pytest
import torch

from splatco_b200.synthetic import ring_cameras
from tests.util import chunk, layout, oracle_backward, oracle_forward, rel_err, scene, settings_for, tans

f32 = np.float32
LOG2E = f32(1.4426950408889634)
CUT = f32(-7.994353436858858)                 # log2(1/255) as the kernels hold it
T_STOP = 1e-4
FP32_STEP = 2.0 ** -22                        # two fp32 roundings per blended splat


def _fma(a, b, c):
    """fp32 fma, correctly rounded: the product is exact in fp64; the fp64 sum is exact up to its TwoSum error, which
    decides the one case where rounding the fp64 sum to fp32 differs from rounding the exact value (a tie)."""
    p = a.astype(np.float64) * b.astype(np.float64)
    c = np.broadcast_to(c, p.shape).astype(np.float64)
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)
    f = s.astype(f32)
    lo = np.where(f.astype(np.float64) <= s, f, np.nextafter(f, f32(-np.inf)))
    hi = np.nextafter(lo, f32(np.inf))
    tie = (s == 0.5 * (lo.astype(np.float64) + hi.astype(np.float64))) & (err != 0)
    return np.where(tie, np.where(err > 0, hi, lo), f)


def _tile_pairs(xy, con, lo, ids, tx, ty):
    """p2, e, dx, dy [n, 256] of the splats `ids` on the pixels of tile (tx, ty), evaluated like eval_p2
    (pixel p = ly * 16 + lx; tile-centred coordinates as pixel_of_thread forms them)."""
    lx = np.tile(np.arange(16), 16)
    ly = np.repeat(np.arange(16), 16)
    u = (lx.astype(f32) - f32(7.5))[None, :]
    v = (ly.astype(f32) - f32(7.5))[None, :]
    cx, cy = f32(tx * 16) + f32(7.5), f32(ty * 16) + f32(7.5)
    sx = (xy[ids, 0] - cx)[:, None]
    sy = (xy[ids, 1] - cy)[:, None]
    a2 = (f32(-0.5) * LOG2E * con[ids, 0])[:, None]
    b2 = (-LOG2E * con[ids, 1])[:, None]
    c2 = (f32(-0.5) * LOG2E * con[ids, 2])[:, None]
    dx = sx - u
    dy = sy - v
    t = _fma(np.broadcast_to(a2, dx.shape), dx, b2 * dy)
    p2 = _fma(c2 * dy, dy, t * dx)
    e = p2 + lo[ids][:, None]
    return p2, e, dx, dy


def reference_blend(xy, con, op, colors, ranges, point_list, H, W, bg, dL=None):
    """The kernels' decisions, evaluated independently (see the module docstring).  Returns image [3,H,W],
    final_T, n_contrib, undecided [H,W] and, with dL [3,H,W], the blend gradients (mean2D [P,2] including the
    0.5 W / 0.5 H NDC factors, conic [P,3], opacity [P], colour [P,3]) in fp64."""
    xy, con, colors = np.asarray(xy, f32), np.asarray(con, f32), np.asarray(colors, np.float64)
    op = np.asarray(op, f32).reshape(-1)
    P = op.shape[0]
    with np.errstate(divide="ignore"):
        lo = np.where(op > 0, np.log2(op.astype(np.float64)), -1e30).astype(f32)
    bg = np.asarray(bg, np.float64)
    gx, gy = (W + 15) // 16, (H + 15) // 16
    img = np.zeros((3, H, W))
    final_T = np.ones((H, W))
    n_contrib = np.zeros((H, W), np.int64)
    undecided = np.zeros((H, W), bool)
    grads = None
    if dL is not None:
        dL = np.asarray(dL, np.float64)
        grads = dict(mean2D=np.zeros((P, 2)), conic=np.zeros((P, 3)), opacity=np.zeros(P), color=np.zeros((P, 3)))
        grads_abs = {k: np.zeros_like(v) for k, v in grads.items()}          # the same sums over |terms|
    lx = np.tile(np.arange(16), 16)
    ly = np.repeat(np.arange(16), 16)
    for tile in range(gx * gy):
        tx, ty = tile % gx, tile // gx
        px, py = tx * 16 + lx, ty * 16 + ly
        inside = (px < W) & (py < H)
        pxi, pyi = px[inside], py[inside]
        beg, end = int(ranges[tile, 0]), int(ranges[tile, 1])
        bgc = np.broadcast_to(bg[:, None], (3, inside.sum()))
        if end <= beg:
            img[:, pyi, pxi] = bgc
            continue
        ids = np.asarray(point_list[beg:end], np.int64)
        n = ids.shape[0]
        p2, e, dx, dy = _tile_pairs(xy, con, lo, ids, tx, ty)
        acc = (p2 <= 0) & (e >= CUT)
        alpha = np.where(acc, np.minimum(0.99, np.exp2(e.astype(np.float64))), 0.0)
        T_after = np.cumprod(1.0 - alpha, axis=0)
        stops = acc & (T_after < T_STOP)
        stop = np.where(stops.any(axis=0), stops.argmax(axis=0), n)          # first pair that would end the walk
        pos = np.arange(n)[:, None]
        valid = acc & (pos < stop[None, :])
        av = np.where(valid, alpha, 0.0)
        T_before = np.cumprod(np.vstack([np.ones((1, 256)), 1.0 - av[:-1]]), axis=0)
        Tf = T_before[-1] * (1.0 - av[-1])
        w = av * T_before
        col = colors[ids]                                                     # [n, 3]
        C = w.T @ col                                                         # [256, 3]
        last = np.where(valid.any(axis=0), n - np.argmax(valid[::-1], axis=0), 0)
        # undecided: some evaluated pair within the approximate log2 / ex2 error of a cut
        seen = pos <= stop[None, :]
        tol_e = 1e-6 * np.maximum(1.0, np.abs(lo[ids].astype(np.float64)))[:, None]
        und = seen & (np.abs(e.astype(np.float64) - float(CUT)) <= tol_e)
        und |= seen & (np.abs(p2) < 4 * np.finfo(f32).tiny)                 # the kernels flush denormals to zero
        und |= seen & acc & (np.abs(T_after - T_STOP) <= 1e-5 * T_STOP)
        und = und.any(axis=0)
        img[:, pyi, pxi] = (C + Tf[:, None] * bg[None, :]).T[:, inside]
        final_T[pyi, pxi] = Tf[inside]
        n_contrib[pyi, pxi] = last[inside]
        undecided[pyi, pxi] = und[inside]
        if grads is None:
            continue
        dp = np.zeros((256, 3))
        dp[inside] = dL[:, pyi, pxi].T
        bgdot = dp @ bg                                                       # [256]
        # S_i = sum_{j > i} c_j alpha_j T_j  (per channel), dL/dalpha_i = dp . (c_i T_i - S_i / (1 - alpha_i)) - T_f bg.dp / (1 - alpha_i)
        wc = w[:, :, None] * col[:, None, :]                                  # [n, 256, 3]
        S = np.cumsum(wc[::-1], axis=0)[::-1] - wc
        inv1m = 1.0 / (1.0 - av)
        dLda = ((col[:, None, :] * T_before[:, :, None] - S * inv1m[:, :, None]) * dp[None]).sum(-1) - Tf * bgdot * inv1m
        D = np.where(valid, dLda * np.exp2(e.astype(np.float64)), 0.0)       # dL/dG * G  (op * G = 2^e, unclamped)
        dxd, dyd = dx.astype(np.float64), dy.astype(np.float64)
        A, B, Cc = [con[ids, k].astype(np.float64)[:, None] for k in range(3)]
        gm = np.stack([(-0.5 * W) * (D * (A * dxd + B * dyd)).sum(1), (-0.5 * H) * (D * (Cc * dyd + B * dxd)).sum(1)], 1)
        gc = -0.5 * np.stack([(D * dxd * dxd).sum(1), (D * dxd * dyd).sum(1), (D * dyd * dyd).sum(1)], 1)
        opi = op[ids].astype(np.float64)
        go = np.where(opi > 0, D.sum(1) / np.where(opi > 0, opi, 1.0), 0.0)
        gcol = w @ dp                                                         # [n, 3]
        np.add.at(grads["mean2D"], ids, gm)
        np.add.at(grads["conic"], ids, gc)
        np.add.at(grads["opacity"], ids, go)
        np.add.at(grads["color"], ids, gcol)
        adp = np.abs(dp)
        Da = np.where(valid, (((col[:, None, :] * T_before[:, :, None] + S * inv1m[:, :, None]) * adp[None]).sum(-1)
                              + Tf * np.abs(bgdot) * inv1m) * np.exp2(e.astype(np.float64)), 0.0)
        adx, ady = np.abs(dxd), np.abs(dyd)
        np.add.at(grads_abs["mean2D"], ids, np.stack([0.5 * W * (Da * (np.abs(A) * adx + np.abs(B) * ady)).sum(1),
                                                      0.5 * H * (Da * (np.abs(Cc) * ady + np.abs(B) * adx)).sum(1)], 1))
        np.add.at(grads_abs["conic"], ids, 0.5 * np.stack([(Da * adx * adx).sum(1), (Da * adx * ady).sum(1), (Da * ady * ady).sum(1)], 1))
        np.add.at(grads_abs["opacity"], ids, np.where(opi > 0, Da.sum(1) / np.where(opi > 0, opi, 1.0), 0.0))
        np.add.at(grads_abs["color"], ids, w @ adp)
    if grads is not None:
        grads["abs"] = grads_abs
    return dict(image=img, final_T=final_T, n_contrib=n_contrib, undecided=undecided, grads=grads)


# ---- pin the reference to the C oracle on a benign scene (CPU only) ------------------------------------
def test_reference_agrees_with_oracle_on_benign_scene():
    W, H = 250, 130
    cam, means, colors, opac, scales, rots = scene(5000, W, H, 2, sigma_px=(0.5, 4.0))
    bg = [0.1, 0.2, 0.3]
    fw = oracle_forward(cam, means, colors, opac, scales, rots, bg)
    pr, bn = fw["pr"], fw["bn"]
    ref = reference_blend(pr.xy, pr.conic_opacity[:, :3], pr.conic_opacity[:, 3], colors.numpy(), bn.ranges,
                          bn.point_list, H, W, bg)
    frag = fw["fragile"] | ref["undecided"]
    assert frag.mean() < 0.02
    assert np.abs(ref["image"] - fw["image"])[:, ~frag].max() <= 1e-4
    assert np.array_equal(ref["n_contrib"][~frag], fw["n_contrib"][~frag])
    assert np.abs(ref["final_T"] - fw["final_T"])[~frag].max() <= 1e-5
    dL = np.random.default_rng(3).standard_normal((3, H, W)) / (3 * H * W)
    dL[:, frag] = 0.0
    dL = dL.astype(f32)
    bw = oracle_backward(fw, cam, means, colors, scales, rots, bg, dL)
    ref = reference_blend(pr.xy, pr.conic_opacity[:, :3], pr.conic_opacity[:, 3], colors.numpy(), bn.ranges,
                          bn.point_list, H, W, bg, dL=dL)
    g = ref["grads"]
    assert rel_err(g["mean2D"], bw["means2D"][:, :2]) < 1e-3
    assert rel_err(g["conic"], bw["conic"]) < 1e-3
    assert rel_err(g["opacity"], bw["opacities"][:, 0]) < 1e-3
    assert rel_err(g["color"], bw["colors"]) < 1e-3


# ---- scenes ---------------------------------------------------------------------------------------------
def _camera(W, H):
    return ring_cameras(3, W, H)[1]


def _world_at(cam, px, py, z):
    """World points that project to pixel coordinates (px, py) at view depth z."""
    W, H = cam.image_width, cam.image_height
    tx, ty = tans(cam)
    px, py, z = [np.broadcast_to(np.asarray(a, np.float64), np.broadcast(px, py, z).shape) for a in (px, py, z)]
    ndc_x, ndc_y = (2.0 * px + 1.0) / W - 1.0, (2.0 * py + 1.0) / H - 1.0
    pv = np.stack([ndc_x * tx * z, ndc_y * ty * z, z, np.ones_like(z)], axis=1)
    return (pv @ np.linalg.inv(cam.world_view_transform.double().numpy()))[:, :3]


def _quat_of(Rm):
    """Unit quaternion (r, x, y, z) of the rotation matrix Rm."""
    tr = np.trace(Rm)
    if tr > 0:
        s = 2.0 * math.sqrt(1.0 + tr)
        q = [0.25 * s, (Rm[2, 1] - Rm[1, 2]) / s, (Rm[0, 2] - Rm[2, 0]) / s, (Rm[1, 0] - Rm[0, 1]) / s]
    else:
        i = int(np.argmax(np.diag(Rm)))
        j, k = (i + 1) % 3, (i + 2) % 3
        s = 2.0 * math.sqrt(1.0 + Rm[i, i] - Rm[j, j] - Rm[k, k])
        q = [0.0] * 4
        q[0] = (Rm[k, j] - Rm[j, k]) / s
        q[1 + i] = 0.25 * s
        q[1 + j] = (Rm[j, i] + Rm[i, j]) / s
        q[1 + k] = (Rm[k, i] + Rm[i, k]) / s
    return np.asarray(q) / np.linalg.norm(q)


def _in_plane_rotation(cam, angle):
    """Rotation whose local x axis lies in the image plane at `angle` from the image's x axis."""
    right, down, fwd = cam.R[:, 0], cam.R[:, 1], cam.R[:, 2]
    d = math.cos(angle) * right + math.sin(angle) * down
    d2 = -math.sin(angle) * right + math.cos(angle) * down
    return _quat_of(np.stack([d, d2, np.cross(d, d2)], axis=1))


class _Scene:
    def __init__(self, W, H, bg):
        self.cam = _camera(W, H)
        self.W, self.H, self.bg = W, H, bg
        self.focal = W / (2.0 * tans(self.cam)[0])
        self.parts = []
        self.rng = np.random.default_rng(W * 1000 + H)

    def add(self, px, py, z, sig_px, op, angle=0.0, aniso=(1.0, 1.0, 1.0), color=None):
        """Splats centred on pixel coordinates (px, py) at depth z, screen sigma ~ sig_px along `angle`."""
        px, py, z, sig_px, op = np.broadcast_arrays(*[np.atleast_1d(np.asarray(a, np.float64)) for a in (px, py, z, sig_px, op)])
        n = px.shape[0]
        means = _world_at(self.cam, px, py, z)
        s = sig_px * z / self.focal
        scales = np.stack([s * aniso[0], s * aniso[1], s * aniso[2]], axis=1)
        rots = np.tile(_in_plane_rotation(self.cam, angle), (n, 1))
        cols = self.rng.random((n, 3)) if color is None else np.tile(color, (n, 1))
        self.parts.append((means, cols, op[:, None], scales, rots))

    def add_random(self, n, sigma_px, depth=(2.0, 6.0), op=(0.05, 0.9)):
        r = self.rng
        z = r.uniform(*depth, n)
        lo, hi = math.log(sigma_px[0]), math.log(sigma_px[1])
        sig = np.exp(r.uniform(lo, hi, (n, 3)))
        means = _world_at(self.cam, r.uniform(-20, self.W + 20, n), r.uniform(-20, self.H + 20, n), z)
        q = r.standard_normal((n, 4))
        self.parts.append((means, r.random((n, 3)), r.uniform(*op, (n, 1)), sig * z[:, None] / self.focal,
                           q / np.linalg.norm(q, axis=1, keepdims=True)))

    def tensors(self):
        cat = lambda k: torch.from_numpy(np.concatenate([p[k] for p in self.parts]).astype(np.float32)).contiguous()
        return [cat(k) for k in range(5)]


def needle_scene(sig_major, op):
    sc = _Scene(160, 112, [0.2, 0.5, 0.8])
    sc.add_random(300, (0.5, 6.0))
    for k, ang in enumerate((0.0, 0.3, math.pi / 4, math.pi / 2 - 0.01)):
        # screen sigma_major ~ sig_major, sigma_minor^2 ~ (1e-4 sig_major)^2 + 0.3 (the low-pass dilation)
        sc.add(40.3 + 27.1 * k, 30.7 + 17.9 * k, 2.5 + 0.7 * k, sig_major, op, angle=ang, aniso=(1.0, 1e-4, 1e-4))
        # the same needle centred far outside, so that the image sees its flank near the alpha cut, where the
        # tile-relative offsets -- and with them the filters' rounding error -- are largest
        d = 0.8 * sig_major * math.sqrt(2.0 * math.log(255.0 * op))
        sc.add(80.2 - d * math.cos(ang), 56.6 - d * math.sin(ang), 3.1 + 0.5 * k, sig_major, op, angle=ang, aniso=(1.0, 1e-4, 1e-4))
    return sc


def straddle_scene():
    """Opacities 1 %-5 % above and below 1/255 on broad splats (op * G crosses the cut on many pixels), the 0.99
    alpha clamp and opacity 0."""
    sc = _Scene(128, 96, [1.0, 1.0, 1.0])
    sc.add_random(200, (0.5, 5.0))
    r = sc.rng
    n = 160
    delta = r.uniform(0.01, 0.05, n) * np.where(np.arange(n) % 2 == 0, 1.0, -1.0)
    sc.add(r.uniform(0, 128, n), r.uniform(0, 96, n), r.uniform(2.0, 6.0, n), r.uniform(6.0, 25.0, n), (1.0 + delta) / 255.0)
    sc.add(r.uniform(0, 128, 40), r.uniform(0, 96, 40), r.uniform(2.0, 6.0, 40), r.uniform(2.0, 12.0, 40), 0.995)
    sc.add(r.uniform(0, 128, 40), r.uniform(0, 96, 40), r.uniform(2.0, 6.0, 40), r.uniform(2.0, 12.0, 40), 0.0)
    return sc


def _crossing_opacity(k):
    """alpha with (1 - alpha)^(k - 1/2) = 1e-4: a pixel at the splats' centre ends its walk at list position k."""
    return 1.0 - math.exp(math.log(T_STOP) / (k - 0.5))


def batch_scene():
    """Stacks of co-located splats, each inside one tile: lists of 511, 512, 513, 1024 and 1025 instances (the
    512-splat staging batch), walks that end at positions 511, 512 and 513, and a stack whose neighbouring pixels of
    one 8x4 patch end at positions 31, 32 and 33 (the backward's skip mask at a 32-splat word boundary)."""
    sc = _Scene(128, 64, [0.3, 0.3, 0.3])
    tc = lambda t: 16 * t + 8.0                          # a pixel centre near the tile centre
    for i, n in enumerate((511, 512, 513, 1024, 1025)):
        sc.add(np.full(n, tc(i)), tc(0), 3.0, 1.5, 0.004)
    for i, k in enumerate((511, 512, 513)):
        sc.add(np.full(1025, tc(i)), tc(2), 3.0, 1.5, _crossing_opacity(k))
    sc.add(np.full(40, tc(7)), tc(3), 3.0, 6.0, _crossing_opacity(32))
    return sc


def geometry_scene(W, H):
    """Image sizes that are not multiples of the tile, centres on tile / patch borders and half pixels, centres
    thousands of pixels outside the image, a screen-filling splat."""
    sc = _Scene(W, H, [0.0, 0.4, 1.0])
    sc.add_random(60 if W * H < 1000 else 400, (0.5, 10.0))
    xs = [x for x in (-0.5, 7.5, 15.5, 16.0, 23.5, 31.5, 0.5, 3.5) if x < W + 8]
    ys = [y for y in (-0.5, 3.5, 7.5, 11.5, 15.5, 16.0, 19.5, 0.5) if y < H + 8]
    gx, gy = np.meshgrid(xs, ys)
    n = gx.size
    sc.add(gx.ravel(), gy.ravel(), np.linspace(2.0, 5.0, n), np.linspace(0.6, 6.0, n), np.linspace(0.1, 0.95, n),
           angle=0.4, aniso=(1.0, 0.3, 0.3))
    sc.add([-3000.0, W + 2500.0, W / 2], [H / 2, -4000.0, H + 6000.0], [4.0, 4.5, 5.0], [1500.0, 2000.0, 2500.0], 0.6)
    sc.add([-5000.0], [H / 3], [4.2], [4000.0], 0.7, angle=0.05, aniso=(1.0, 2e-3, 2e-3))     # far needle aimed at the image
    sc.add([W / 2], [H / 2], [5.5], [4.0 * max(W, H)], 0.5)                                   # screen-filling
    return sc


SCENES = {f"needle_s{s}_op{op}": (lambda s=s, op=op: needle_scene(s, op)) for s in (30, 300, 1000, 3000) for op in (0.9, 0.02)}
SCENES["straddle"] = straddle_scene
SCENES["batch_edges"] = batch_scene
SCENES.update({f"geometry_{W}x{H}": (lambda W=W, H=H: geometry_scene(W, H)) for W, H in ((1, 17), (15, 15), (17, 1), (250, 131))})
IMPLS = [("fwd", 1), ("fwd", 2), ("bwd", 1), ("bwd", 2), ("bwd", 3)]

_cache = {}


def _prepared(name):
    """The scene rasterized on the GPU, the records the kernels consumed, the reference forward and backward."""
    if name in _cache:
        return _cache[name]
    from splatco_b200 import _lib
    from splatco_b200.diff_gaussian_rasterization import rasterize_forward_state
    from tests.test_raster_gpu import unpack_state
    sc = SCENES[name]()
    means, colors, opac, scales, rots = sc.tensors()
    st = settings_for(sc.cam, sc.bg)
    _, _, state = rasterize_forward_state(*[t.cuda() for t in (means, colors, opac, scales, rots)], st)
    torch.cuda.synchronize()
    assert state.R > 0
    g = unpack_state(state)
    P = state.P
    rec = chunk(state.geom, layout("geom", P)[0], torch.float32, 12 * P).view(P, 12).cpu().numpy()
    H, W = sc.H, sc.W
    xy, con, op, col = rec[:, 0:2], rec[:, 2:5], rec[:, 5], rec[:, [6, 7, 8]]
    ref = reference_blend(xy, con, op, col, g["ranges"], g["point_list"], H, W, sc.bg)
    und = ref["undecided"]
    dL = np.random.default_rng(11).standard_normal((3, H, W)) / (3 * H * W)
    dL[:, und] = 0.0
    dL = dL.astype(f32)
    ref["grads"] = reference_blend(xy, con, op, col, g["ranges"], g["point_list"], H, W, sc.bg, dL=dL)["grads"]
    out = dict(state=state, ref=ref, dL=dL, bg=sc.bg, counts=g["ranges"][:, 1] - g["ranges"][:, 0], L=_lib.lib())
    _cache[name] = out
    return out


def _scene_exercises(name, p):
    """The scene really contains the edge it is named for."""
    ref, counts = p["ref"], p["counts"]
    if name == "batch_edges":
        for n in (511, 512, 513, 1024, 1025):
            assert (counts == n).any(), f"no tile lists {n} instances"
        nc = ref["n_contrib"]
        for k in (510, 511, 512):                       # walk ended AT position k + 1: last contributor k
            assert (nc == k).any(), f"no walk ends at list position {k + 1}"
        patch = nc[56:60, 120:128]                      # rows 56..59, columns 120..127: one warp's 8x4 patch
        assert {31, 32, 33} <= set(np.unique(patch).tolist()), np.unique(patch)
    if name.startswith("needle"):
        assert counts.max() > 0 and (ref["n_contrib"] > 0).mean() > 0.3


@pytest.mark.gpu
@pytest.mark.parametrize("impl", IMPLS, ids=[f"{k}{i}" for k, i in IMPLS])
@pytest.mark.parametrize("name", list(SCENES))
def test_blend_kernels_match_reference(name, impl):
    from splatco_b200._lib import check, ptr
    p = _prepared(name)
    state, ref, L = p["state"], p["ref"], p["L"]
    _scene_exercises(name, p)
    und = ref["undecided"]
    assert und.mean() < 0.02, f"{und.mean():.3%} of the pixels undecided"
    H, W, P, R = state.H, state.W, state.P, state.RL
    stream = torch.cuda.current_stream().cuda_stream
    bg = torch.tensor(p["bg"], dtype=torch.float32, device="cuda")
    io = layout("image", H, W)
    fT = chunk(state.image, io[1], torch.float32, H * W).view(H, W)
    nc = chunk(state.image, io[2], torch.int32, H * W).view(H, W)
    kind, k = impl
    try:
        if kind == "fwd":
            check(L.splatco_blend_set_impl(k, 0), "set_impl")
            img = torch.empty(3, H, W, device="cuda")
            check(L.splatco_blend_fwd(R, H, W, ptr(bg), ptr(state.geom), ptr(state.binning), ptr(state.image), ptr(img), stream), "blend_fwd")
            torch.cuda.synchronize()
            img, got_T, got_n = img.cpu().numpy(), fT.cpu().numpy(), nc.cpu().numpy()
            bad = (got_n != ref["n_contrib"]) & ~und
            if bad.any():
                y, x = np.argwhere(bad)[0]
                pytest.fail(f"{kind}{k}: n_contrib differs on {bad.sum()} decided pixels, first ({x}, {y}): "
                            f"kernel {got_n[y, x]}, reference {ref['n_contrib'][y, x]} (list position of the last contributor "
                            f"in tile {(y // 16) * ((W + 15) // 16) + x // 16})")
            # the kernels carry T in fp32: every contributor rounds 1 - alpha and the product (FP32_STEP), so a walk
            # of n contributors may drift by n FP32_STEP relative on top of the fixed bars
            drift = FP32_STEP * ref["n_contrib"]
            errT = (np.abs(got_T - ref["final_T"]) - drift * ref["final_T"])[~und]
            assert errT.max() <= 1e-6, f"{kind}{k}: final_T err {errT.max()} beyond the fp32 walk drift"
            erri = (np.abs(img - ref["image"]) - drift)[:, ~und]
            assert erri.max() <= 1e-5, f"{kind}{k}: image err {erri.max()} beyond the fp32 walk drift"
        else:
            # the backward replays from the REFERENCE walk's final_T / n_contrib, so it is checked on its own
            fT.copy_(torch.from_numpy(ref["final_T"].astype(np.float32)))
            nc.copy_(torch.from_numpy(ref["n_contrib"].astype(np.int32)))
            check(L.splatco_blend_set_impl(0, k), "set_impl")
            gs = [torch.zeros(P, c, device="cuda") for c in (3, 3, 1, 3)]
            dL = torch.from_numpy(p["dL"]).cuda()
            check(L.splatco_blend_bwd(P, R, H, W, ptr(bg), ptr(state.geom), ptr(state.binning), ptr(state.image), ptr(dL),
                                      *[ptr(t) for t in gs], stream), "blend_bwd")
            torch.cuda.synchronize()
            got = [t.double().cpu().numpy() for t in gs]
            want = ref["grads"]
            # T is reconstructed in fp32 by dividing final_T by 1 - alpha per contributor: on top of rel_err's 1e-3
            # every per-pixel term may drift by FP32_STEP per contributor of the pixel's walk
            drift = FP32_STEP * ref["n_contrib"].max()
            for nm, a, b in (("mean2D", got[0][:, :2], want["mean2D"]), ("conic", got[1], want["conic"]),
                             ("opacity", got[2][:, 0], want["opacity"]), ("color", got[3], want["color"])):
                floor = 1e-3 * np.abs(b).max()
                err = (np.abs(a - b) - drift * want["abs"][nm]) / np.maximum(np.abs(b), max(floor, 1e-30))
                i = int(err.argmax())
                assert err.flat[i] < 1e-3, (f"{kind}{k}: d{nm} rel err {err.flat[i]:.3g} at splat {i // (a.size // P)}: "
                                            f"kernel {a.flat[i]}, reference {b.flat[i]} (max {np.abs(b).max()})")
            assert not got[0][:, 2].any()
    finally:
        check(L.splatco_blend_set_impl(2, 2), "set_impl")
