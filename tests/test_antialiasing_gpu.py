"""GPU tests of antialiasing (GaussianRasterizationSettings(..., antialiasing=True)): the forward against the C reference
(tests/antialiasing_oracle.py, the colour oracle with the compensated opacity) bit for bit, the backward against that
reference and against fp64 autograd (including the rho clamp), with depth / alpha maps
and camera gradients, through render(), and with antialiasing off exactly as before."""
import math
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import composite_torch as CT
from oracle import raster as R
from splatco_b200 import _lib
from tests import antialiasing_oracle as AA
from tests import depth_alpha_oracle as DA
from tests.test_oracle_antialiasing import RHO_MIN32, box4, make, scale_scene, sub_pixel_scene
from tests.test_raster_gpu import assert_forward_parity, unpack_state
from tests.util import full_path_grad_errors, rel_err, scene, settings_for, tans

pytestmark = pytest.mark.gpu
ptr = _lib.ptr
UNUSED = [3, 7, 11, 15, 16 + 2, 16 + 6, 16 + 10, 16 + 14]


def aa_settings(cam, bg, **kw):
    return settings_for(cam, bg, **kw)._replace(antialiasing=True)


def oracle_fw(cam, means, colors, opac, scales, rots, bg):
    tx, ty = tans(cam)
    return AA.rasterize_forward(means.numpy(), colors.numpy(), opac.numpy(), scales.numpy(), rots.numpy(), 1.0,
                                cam.world_view_transform.numpy(), cam.full_proj_transform.numpy(), tx, ty,
                                int(cam.image_height), int(cam.image_width), np.asarray(bg, np.float32))


def oracle_bw(fw, cam, means, colors, opac, scales, rots, bg, dL):
    tx, ty = tans(cam)
    return AA.rasterize_backward(fw, means.numpy(), colors.numpy(), opac.numpy(), scales.numpy(), rots.numpy(), 1.0,
                                 cam.world_view_transform.numpy(), cam.full_proj_transform.numpy(), tx, ty,
                                 int(cam.image_height), int(cam.image_width), np.asarray(bg, np.float32), dL)


def gpu_fw(settings, means, colors, opac, scales, rots):
    from splatco_b200.diff_gaussian_rasterization import rasterize_forward_state
    d = "cuda"
    color, radii, st = rasterize_forward_state(means.to(d), colors.to(d), opac.to(d), scales.to(d), rots.to(d), settings)
    torch.cuda.synchronize()
    return color, radii, st


def rasterize(settings, ins, depth_alpha=False):
    from splatco_b200.diff_gaussian_rasterization import GaussianRasterizer
    m, c, o, s, q = ins
    return GaussianRasterizer(settings)(means3D=m, means2D=torch.zeros_like(m, requires_grad=True), shs=None,
                                        colors_precomp=c, opacities=o, scales=s, rotations=q, cov3D_precomp=None,
                                        depth_alpha=depth_alpha)


# ---- forward ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed,W,H,M,sig", [
    (1, 64, 48, 300, (1.0, 6.0)), (2, 250, 130, 5000, (0.5, 4.0)), (3, 256, 256, 100000, (0.5, 4.0)),
    (4, 980, 545, 60000, (0.5, 8.0)), (5, 97, 33, 2000, (4.0, 40.0))])
def test_forward_parity_aa(seed, W, H, M, sig):
    cam, means, colors, opac, scales, rots = scene(M, W, H, seed, sigma_px=sig)
    bg = [1.0, 1.0, 1.0] if seed % 2 else [0.1, 0.2, 0.3]
    fw = oracle_fw(cam, means, colors, opac, scales, rots, bg)
    color, radii, st = gpu_fw(aa_settings(cam, bg), means, colors, opac, scales, rots)
    g = assert_forward_parity(fw, color, radii, st)          # conic_opacity bits include the compensated opacity
    vis = fw["pr"].radii > 0
    assert (fw["pr"].conic_opacity[vis, 3] <= opac.numpy()[vis, 0]).all()
    # the integer path and the conic are those of the plain call
    color0, radii0, st0 = gpu_fw(settings_for(cam, bg), means, colors, opac, scales, rots)
    g0 = unpack_state(st0)
    assert torch.equal(radii, radii0) and st.R == st0.R
    for k in ("tiles", "depths", "xy", "keys", "point_list", "ranges"):
        if k in g0:
            assert np.array_equal(g[k], g0[k]), k
    assert np.array_equal(g["conic_opacity"][:, :3], g0["conic_opacity"][:, :3])


# ---- backward against the C oracle -------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed,W,H,M,sig", [
    (41, 64, 48, 300, (1.0, 6.0)), (42, 250, 130, 5000, (0.5, 4.0)), (43, 97, 33, 2000, (4.0, 40.0)),
    (44, 256, 256, 100000, (0.5, 4.0)), (45, 980, 545, 1_000_000, (0.5, 4.0))])
def test_backward_parity_aa(seed, W, H, M, sig):
    cam, means, colors, opac, scales, rots = scene(M, W, H, seed, sigma_px=sig)
    bg = [1.0, 1.0, 1.0]
    fw = oracle_fw(cam, means, colors, opac, scales, rots, bg)
    ins = [t.cuda().requires_grad_() for t in (means, colors, opac, scales, rots)]
    img, radii = rasterize(aa_settings(cam, bg), ins)
    gt = torch.rand(3, H, W, generator=torch.Generator().manual_seed(seed))
    dL = (torch.sign(torch.from_numpy(fw["image"]) - gt) / (3 * H * W)).float()
    # no upstream gradient on the pixels the oracle flags fragile: there a 1-ulp difference may legitimately end the walk
    # at another contributor (test_raster_gpu's forward rule), which at 1 M Gaussians moves single gradient entries by
    # more than the 1e-3 bar, with antialiasing off as well as on
    dL[:, torch.from_numpy(fw["fragile"])] = 0.0
    img.backward(dL.cuda())
    bw = oracle_bw(fw, cam, means, colors, opac, scales, rots, bg, dL.numpy())
    for name, t in zip(("means3D", "colors", "opacities", "scales", "rotations"), ins):
        assert rel_err(t.grad.cpu().numpy(), bw[name]) < 1e-3, name


# ---- backward against fp64 autograd, depth / alpha maps and camera gradients --------------------------------------------
def fp64_maps(cam, means, colors, opac, scales, rots, bg, pr):
    """fp64 autograd composite (image, depth, alpha) with the compensated opacity; leaves include the two matrices."""
    tx, ty = tans(cam)
    H, W = int(cam.image_height), int(cam.image_width)
    d = torch.float64
    leaves = [t.to(d).requires_grad_() for t in (means, colors, opac, scales, rots)]
    m, c, o, s, q = leaves
    v64 = cam.world_view_transform.to(d).requires_grad_()
    p64 = cam.full_proj_transform.to(d).requires_grad_()
    xy, tz, conic, (a, b, cc) = CT.project(m, s, q, 1.0, v64, p64, tx, ty, H, W)
    op = o.reshape(-1) * AA.rho_torch(a, b, cc)
    order = torch.tensor(sorted(range(means.shape[0]), key=lambda i: (int(np.float32(pr.depths[i]).view(np.uint32)), i)))
    maps = DA.composite_depth_alpha(xy, tz, conic, op, c, torch.as_tensor(bg, dtype=d), torch.tensor(pr.rect), order,
                                    H, W)
    return maps, leaves, (v64, p64)


@pytest.mark.parametrize("loss", ["colour", "depth", "alpha"])
@pytest.mark.parametrize("kind,seed", [("ordinary", 7), ("ordinary_small", 11), ("rho_clamp", 13), ("txy_clamp", 17)])
def test_aa_gradients_vs_fp64_autograd_with_maps_and_camera(kind, seed, loss):
    cam, means, colors, opac, scales, rots = make(kind, seed)
    H, W = int(cam.image_height), int(cam.image_width)
    bg = [1.0, 0.5, 0.25]
    fw = oracle_fw(cam, means, colors, opac, scales, rots, bg)
    g = torch.Generator().manual_seed(seed + 3)
    ups = {"colour": torch.randn(3, H, W, generator=g, dtype=torch.float64) / (H * W),
           "depth": torch.randn(1, H, W, generator=g, dtype=torch.float64) / (H * W),
           "alpha": torch.randn(1, H, W, generator=g, dtype=torch.float64) / (H * W)}
    k = ["colour", "depth", "alpha"].index(loss)
    (maps, leaves, mats) = fp64_maps(cam, means, colors, opac, scales, rots, bg, fw["pr"])
    want = torch.autograd.grad(maps[k], leaves + list(mats), ups[loss], allow_unused=True)
    ins = [t.cuda().requires_grad_() for t in (means, colors, opac, scales, rots)]
    vm = cam.world_view_transform.cuda().requires_grad_()
    pm = cam.full_proj_transform.cuda().requires_grad_()
    st = aa_settings(cam, bg)._replace(viewmatrix=vm, projmatrix=pm)
    outs = rasterize(st, ins, depth_alpha=True)
    (outs[0], outs[2], outs[3])[k].backward(ups[loss].float().cuda())
    got = [t.grad.cpu().numpy() for t in ins] + [vm.grad.reshape(-1).cpu().numpy(), pm.grad.reshape(-1).cpu().numpy()]
    names = ("means3D", "colors", "opacities", "scales", "rotations", "viewmatrix", "projmatrix")
    for name, x, w in zip(names, got, want):
        if w is None:                                       # the colours of a depth or alpha loss
            assert name == "colors" and np.abs(x).max() == 0
            continue
        w = w.reshape(x.shape).numpy()
        assert np.abs(w).max() > 0, name
        assert rel_err(x, w) < 5e-3, (name, rel_err(x, w))   # the fp32-blend bar of tests/test_oracle_raster.py
    assert np.all(np.concatenate(got[5:])[UNUSED] == 0.0)


def test_rho_clamped_everywhere_scales_the_opacity_gradient_only():
    """Every Gaussian in the rho clamp: splatco_preprocess_bwd_aa rewrites dL/dopacity to exactly rho * dL/do' and adds
    no rho term, so its geometry gradients are those of splatco_preprocess_bwd on the same inputs."""
    cam, means, colors, opac, scales, rots = sub_pixel_scene(20000, 250, 130, 5, frac=1.0)
    bg = [0.0, 0.0, 0.0]
    _, radii, st = gpu_fw(aa_settings(cam, bg), means, colors, opac, scales, rots)
    rec = unpack_state(st)
    vis = radii.cpu().numpy() > 0
    assert vis.sum() > 10000
    assert np.array_equal(rec["conic_opacity"][vis, 3], opac.numpy()[vis, 0] * RHO_MIN32)
    P, H, W = st.P, st.H, st.W
    tx, ty = tans(cam)
    gen = torch.Generator().manual_seed(2)
    g2, gc, go = [torch.randn(P, n, generator=gen).cuda() for n in (3, 3, 1)]
    d = [t.cuda() for t in (means, scales, rots, opac)]
    view, proj = cam.world_view_transform.cuda(), cam.full_proj_transform.cuda()
    L = _lib.lib()
    s = torch.cuda.current_stream().cuda_stream

    def outs():
        return torch.empty(P, 3, device="cuda"), torch.empty(P, 3, device="cuda"), torch.empty(P, 4, device="cuda")
    a, b = outs(), outs()
    common = (P, ptr(d[0]), ptr(d[1]), 3, ptr(d[2]), 1.0, ptr(view), ptr(proj), tx, ty, H, W, ptr(radii), ptr(g2),
              ptr(gc))
    _lib.check(L.splatco_preprocess_bwd(*common, *[ptr(t) for t in a], s), "splatco_preprocess_bwd")
    go_aa = go.clone()
    _lib.check(L.splatco_preprocess_bwd_aa(*common, *[ptr(t) for t in b], ptr(d[3]), ptr(go_aa), None, None, None, None,
                                           s), "splatco_preprocess_bwd_aa")
    torch.cuda.synchronize()
    for x, y in zip(a, b):
        x, y = x.cpu().numpy(), y.cpu().numpy()
        assert np.abs(x - y).max() <= 1e-6 * np.abs(x).max()
    want = go.cpu().numpy()[:, 0] * RHO_MIN32
    assert np.array_equal(go_aa.cpu().numpy()[vis, 0], want[vis])
    assert np.array_equal(go_aa.cpu().numpy()[~vis, 0], go.cpu().numpy()[~vis, 0])


@pytest.mark.parametrize("depth", [False, True])
def test_aa_camera_call_is_reproducible_and_keeps_the_per_gaussian_outputs(depth):
    """splatco_preprocess_bwd_aa with camera outputs: two calls on the same inputs are bitwise equal, and the per-Gaussian
    outputs (dL_dopacity's rewrite included) are bitwise those of the call without camera outputs."""
    cam, means, colors, opac, scales, rots = sub_pixel_scene(100000, 980, 545, 8, frac=0.5)
    _, radii, st = gpu_fw(aa_settings(cam, [0, 0, 0]), means, colors, opac, scales, rots)
    P, H, W = st.P, st.H, st.W
    tx, ty = tans(cam)
    gen = torch.Generator().manual_seed(4)
    g2, gc, go, gd = [torch.randn(P, n, generator=gen).cuda() * 1e-2 for n in (3, 3, 1, 1)]
    d = [t.cuda() for t in (means, scales, rots, opac)]
    view, proj = cam.world_view_transform.cuda(), cam.full_proj_transform.cuda()
    L = _lib.lib()
    s = torch.cuda.current_stream().cuda_stream
    ws = torch.empty(L.splatco_camera_grad_ws_bytes(P), dtype=torch.uint8, device="cuda")

    def call(camera):
        o = [torch.empty(P, n, device="cuda") for n in (3, 3, 4)] + [go.clone()]
        cg = torch.empty(32, device="cuda")
        cam_args = (ptr(ws), ptr(cg[:16]), ptr(cg[16:])) if camera else (None, None, None)
        _lib.check(L.splatco_preprocess_bwd_aa(P, ptr(d[0]), ptr(d[1]), 3, ptr(d[2]), 1.0, ptr(view), ptr(proj), tx, ty,
                                               H, W, ptr(radii), ptr(g2), ptr(gc), *[ptr(t) for t in o[:3]], ptr(d[3]),
                                               ptr(o[3]), ptr(gd) if depth else None, *cam_args, s),
                   "splatco_preprocess_bwd_aa")
        torch.cuda.synchronize()
        return [t.cpu().numpy() for t in o], cg.cpu().numpy()
    (a, ca), (b, cb), (c, _) = call(True), call(True), call(False)
    assert ca.tobytes() == cb.tobytes() and np.abs(ca).max() > 0 and np.all(ca[UNUSED] == 0.0)
    for x, y, z in zip(a, b, c):
        assert x.tobytes() == y.tobytes() == z.tobytes()


# ---- AA off is untouched ----------------------------------------------------------------------------------------------
def test_antialiasing_off_is_the_twelve_field_call():
    cam, means, colors, opac, scales, rots = scene(20000, 250, 130, 9, sigma_px=(0.1, 4.0))
    bg = [0.2, 0.3, 0.4]
    L = _lib.lib()
    twelve = settings_for(cam, bg)
    assert len(twelve) == 13 and twelve.antialiasing is False
    st12 = type(twelve)(*tuple(twelve)[:12])                     # positional, upstream's 12 fields
    results = []
    for st in (st12, twelve._replace(antialiasing=False)):
        ins = [t.cuda().requires_grad_() for t in (means, colors, opac, scales, rots)]
        n0 = L.splatco_launch_count()
        img, radii = rasterize(st, ins)
        img.square().sum().backward()
        torch.cuda.synchronize()
        results.append((L.splatco_launch_count() - n0, img.detach().cpu().numpy(), radii.cpu().numpy(),
                        [t.grad.cpu().numpy() for t in ins]))
    (n0, i0, r0, g0), (n1, i1, r1, g1) = results
    assert n0 == n1 and i0.tobytes() == i1.tobytes() and r0.tobytes() == r1.tobytes()
    for x, y in zip(g0, g1):                          # (the blend backward's float atomics reorder sums)
        assert np.abs(x - y).max() <= 1e-5 * np.abs(x).max()
    ins = [t.cuda().requires_grad_() for t in (means, colors, opac, scales, rots)]
    img_aa, _ = rasterize(twelve._replace(antialiasing=True), ins)
    assert not torch.equal(img_aa.detach().cpu(), torch.from_numpy(i0))


def test_edge_cases_empty_all_culled_and_zero_opacity():
    cam, means, colors, opac, scales, rots = scene(64, 50, 34, 5)
    bg = [0.2, 0.4, 0.6]
    bgi = torch.tensor(bg, device="cuda")[:, None, None].expand(3, 34, 50)
    z = lambda *s: torch.zeros(*s, device="cuda", requires_grad=True)
    vm = cam.world_view_transform.cuda().requires_grad_()
    st = aa_settings(cam, bg)._replace(viewmatrix=vm)
    img, radii, dep, alp = rasterize(st, [z(0, 3), z(0, 3), z(0, 1), z(0, 3), z(0, 4)], depth_alpha=True)
    assert radii.numel() == 0 and torch.allclose(img, bgi)
    (img.sum() + dep.sum()).backward()
    assert torch.count_nonzero(vm.grad) == 0
    behind = (cam.camera_center * 3.0)[None].repeat(64, 1)
    ins = [t.cuda().requires_grad_() for t in (behind, colors, opac, scales, rots)]
    img, radii = rasterize(aa_settings(cam, bg), ins)
    assert (radii == 0).all() and torch.allclose(img, bgi)
    img.sum().backward()
    assert all(torch.count_nonzero(t.grad) == 0 for t in ins)
    ins = [t.cuda().requires_grad_() for t in (means, colors, torch.zeros_like(opac), scales, rots)]
    img, radii = rasterize(aa_settings(cam, bg), ins)
    assert (radii > 0).any() and torch.allclose(img, bgi)
    img.sum().backward()
    assert torch.isfinite(ins[2].grad).all() and torch.count_nonzero(ins[0].grad) == 0


# ---- render() ---------------------------------------------------------------------------------------------------------
PIPE_AA = SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False, antialiasing=True)


def test_render_with_pipe_antialiasing():
    from splatco_b200.diff_gaussian_rasterization import GaussianRasterizer
    from splatco_b200.gaussian_renderer import _settings, generate_neural_gaussians, prefilter_voxel, render
    from tests.test_render_gpu import PIPE, _cams, _model
    pc = _model(N=3000, seed=5)
    cams = list(_cams(160, 112))
    bg = torch.ones(3, device="cuda")
    assert _settings(cams[0], PIPE_AA, bg, 1.0).antialiasing and not _settings(cams[0], PIPE, bg, 1.0).antialiasing
    # the speculative fast path equals the plain two calls bit for bit, forward and gradients
    out = []
    for fast in (True, False):
        vm = prefilter_voxel(cams[1], pc, PIPE_AA, bg)
        if fast:
            img = render(cams[1], pc, PIPE_AA, bg, visible_mask=vm)["render"]
        else:
            xyz, color, opacity, scaling, rot, _, _ = generate_neural_gaussians(cams[1], pc, vm, is_training=True)
            img, _ = GaussianRasterizer(_settings(cams[1], PIPE_AA, bg, 1.0))(
                means3D=xyz, means2D=torch.zeros_like(xyz), shs=None, colors_precomp=color, opacities=opacity,
                scales=scaling, rotations=rot, cov3D_precomp=None)
        out.append((img.detach().clone(), torch.autograd.grad(img.square().mean(), [pc._anchor_feat, pc._offset])))
    assert torch.equal(out[0][0], out[1][0])
    for a, b in zip(out[0][1], out[1][1]):                # (the blend backward's float atomics reorder sums)
        assert a.abs().max() > 0 and (a - b).abs().max() <= 1e-5 * a.abs().max()

    # one backward over two views equals the sum of separate backwards
    def loss_of(i, pipe=PIPE_AA):
        vm = prefilter_voxel(cams[i], pc, pipe, bg)
        pkg = render(cams[i], pc, pipe, bg, visible_mask=vm, depth_alpha=True)
        return pkg["render"].square().mean() + 0.1 * pkg["depth"].mean() + pkg["alpha"].mean()
    leaves = [pc._anchor_feat, pc._offset, pc._scaling]
    both = torch.autograd.grad(loss_of(0) + loss_of(1), leaves)
    sep = [a + b for a, b in zip(torch.autograd.grad(loss_of(0), leaves), torch.autograd.grad(loss_of(1), leaves))]
    for a, b in zip(both, sep):
        assert a.abs().max() > 0 and (a - b).abs().max() <= 1e-4 * a.abs().max()
    # antialiasing changes the image; a pipe without the attribute renders as before
    with torch.no_grad():
        i_aa = render(cams[0], pc, PIPE_AA, bg, visible_mask=prefilter_voxel(cams[0], pc, PIPE_AA, bg))["render"]
        i_0 = render(cams[0], pc, PIPE, bg, visible_mask=prefilter_voxel(cams[0], pc, PIPE, bg))["render"]
        assert not torch.equal(i_aa, i_0)
    # eval mode
    pc.eval()
    try:
        with torch.no_grad():
            pkg = render(cams[0], pc, PIPE_AA, bg, visible_mask=prefilter_voxel(cams[0], pc, PIPE_AA, bg))
        assert torch.isfinite(pkg["render"]).all() and (pkg["radii"] > 0).any()
    finally:
        pc.train()


def test_render_pipe_without_the_attribute_keeps_launches_and_outputs():
    from splatco_b200.gaussian_renderer import prefilter_voxel, render
    from tests.test_render_gpu import PIPE, _cams, _model
    pc = _model(N=3000, seed=5)
    cam = _cams(160, 112)[1]
    bg = torch.ones(3, device="cuda")
    L = _lib.lib()
    pipe_off = SimpleNamespace(**vars(PIPE), antialiasing=False)

    def run(pipe):
        n0 = L.splatco_launch_count()
        pkg = render(cam, pc, pipe, bg, visible_mask=prefilter_voxel(cam, pc, pipe, bg))
        grads = torch.autograd.grad(pkg["render"].square().mean(), [pc._anchor_feat, pc._offset])
        torch.cuda.synchronize()
        return L.splatco_launch_count() - n0, pkg["render"].detach().clone(), grads
    run(PIPE)
    a, b = run(PIPE), run(pipe_off)
    assert a[0] == b[0] and torch.equal(a[1], b[1])
    for x, y in zip(a[2], b[2]):                      # (the blend backward's float atomics reorder sums)
        assert (x - y).abs().max() <= 1e-5 * x.abs().max()


def test_full_path_c1_aa_vs_oracle_chain():
    """prefilter_voxel -> render() with antialiasing on the bench's C1 model; the leaf gradients against the oracle
    decode followed by the antialiased C oracle rasterizer."""
    import bench
    from oracle import decode_oracle as D
    from splatco_b200.gaussian_renderer import prefilter_voxel, render
    cfg = dict(bench.WORKLOADS["c1"])
    bench.LEVEL = 2
    dev = torch.device("cuda")
    pc = bench.build_model(cfg, dev)
    pc.feat_planes.Q0 = 0.0
    cams, _ = bench.build_views(cfg)
    cam = cams[1 % len(cams)]
    H, W, K = cfg["H"], cfg["W"], cfg["K"]
    bg = torch.ones(3, device=dev)
    pipe = SimpleNamespace(**vars(bench.PIPE), antialiasing=True)
    cam_d = cam.to(dev)
    vm = prefilter_voxel(cam_d, pc, pipe, bg)
    pkg = render(cam_d, pc, pipe, bg, visible_mask=vm)
    dC = torch.randn(3, H, W, generator=torch.Generator().manual_seed(21)) / (3 * H * W)
    pkg["render"].backward(dC.to(dev))
    leaves = {"_anchor": pc._anchor, "_offset": pc._offset, "_anchor_feat": pc._anchor_feat, "_scaling": pc._scaling}
    for name in ("mlp_opacity", "mlp_cov", "mlp_color"):
        for k, v in getattr(pc, name).named_parameters():
            leaves[f"{name}.{k}"] = v
    for k, v in pc.feat_planes._feat.named_parameters():
        leaves[f"feat.{k}"] = v
    cpu = bench.build_model(cfg, "cpu")
    cpu.feat_planes.Q0 = 0.0
    p = {"feat." + k: v for k, v in cpu.feat_planes._feat.state_dict().items()}
    for name in ("mlp_opacity", "mlp_cov", "mlp_color"):
        p.update({f"{name}.{k}": v for k, v in getattr(cpu, name).state_dict().items()})
    for k, v in p.items():
        if v.dtype.is_floating_point and "running" not in k and "xyz_m" not in k:
            v.requires_grad_(True)
    tx, ty = math.tan(cam.FoVx * 0.5), math.tan(cam.FoVy * 0.5)
    view, proj = cam.world_view_transform.numpy(), cam.full_proj_transform.numpy()
    scaling = torch.exp(cpu._scaling)
    radii_a = R.visible_filter(cpu._anchor.detach().numpy(), scaling.detach().numpy()[:, :3],
                               torch.nn.functional.normalize(cpu._rotation).numpy(), 1.0, view, proj, tx, ty, H, W)
    vis = torch.from_numpy(radii_a > 0)
    assert np.array_equal(vm.cpu().numpy(), vis.numpy())
    xyz, color, opacity, scl, rot, _, mask = D.decode(p, cpu._anchor_feat, cpu._anchor, cpu._offset, scaling, vis,
                                                      cam.camera_center, 2, K)
    assert np.array_equal(pkg["selection_mask"].cpu().numpy(), mask.numpy())
    a = [t.detach().numpy() for t in (xyz, color, opacity, scl, rot)]
    bgn = np.ones(3, np.float32)
    fw = AA.rasterize_forward(a[0], a[1], a[2], a[3], a[4], 1.0, view, proj, tx, ty, H, W, bgn)
    frag = fw["fragile"]
    assert np.abs(pkg["render"].detach().cpu().numpy() - fw["image"])[:, ~frag].max() <= 1e-3
    g = AA.rasterize_backward(fw, a[0], a[1], a[2], a[3], a[4], 1.0, view, proj, tx, ty, H, W, bgn, dC.numpy())
    torch.autograd.backward([xyz, color, opacity, scl, rot],
                            [torch.from_numpy(g[k]) for k in ("means3D", "colors", "opacities", "scales", "rotations")])
    want = {"_anchor": cpu._anchor.grad, "_offset": cpu._offset.grad, "_anchor_feat": cpu._anchor_feat.grad,
            "_scaling": cpu._scaling.grad}
    want.update({k: v.grad for k, v in p.items() if v.requires_grad})
    worst = {}
    for k, w_ in want.items():
        if w_ is None:
            continue
        got = leaves[k].grad
        assert got is not None, k
        wn = w_.numpy()
        if float(np.abs(wn).max()) == 0.0:
            assert float(got.abs().max()) == 0.0, k
            continue
        e = full_path_grad_errors(got.cpu().numpy(), wn)
        worst[k] = (e["l2"] / (3e-3 if ".TA." in k else 1e-3), e["amax"])
    assert "_anchor" in worst and "_offset" in worst
    ranked = sorted(worst.items(), key=lambda kv: -kv[1][0])
    assert ranked[0][1][0] < 1.0, ranked[:8]


# ---- it does its job ---------------------------------------------------------------------------------------------------
def test_quarter_resolution_render_is_closer_to_the_downsampled_full_render():
    """The scene and metric of tests/test_oracle_antialiasing.py's fp64 check, at 4x the size: the W/4 x H/4 render
    against the 4x4 box average of the W x H render, each with the same antialiasing setting."""
    from splatco_b200.synthetic import ring_cameras
    W, H, M = 512, 384, 24000
    cam_hi, means, colors, opac, scales, rots = scale_scene(M, W, H, 3)
    cam_lo = ring_cameras(3, W // 4, H // 4)[1]
    bg = [0.0, 0.0, 0.0]
    err = {}
    for aa in (False, True):
        imgs = []
        for cam in (cam_hi, cam_lo):
            st = settings_for(cam, bg)._replace(antialiasing=aa)
            with torch.no_grad():
                img, _ = rasterize(st, [t.cuda() for t in (means, colors, opac, scales, rots)])
            imgs.append(img.cpu().numpy())
        err[aa] = float(np.abs(imgs[1] - box4(imgs[0])).mean())
    assert err[True] < 0.5 * err[False], err
