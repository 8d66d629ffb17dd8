"""GPU tests of the camera gradients: splatco_preprocess_bwd_camera against fp64 autograd of the projection, the
rasterizer's view / projection gradients against the fp64 autograd composite, the decode's camera-centre gradient against
the fp64 decode oracle, the whole render() path with a learnable pose, and the autograd plumbing."""
import math
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import composite_torch as CT
from splatco_b200 import _lib
from splatco_b200.synthetic import ring_cameras
from tests import depth_alpha_oracle as DA
from tests.camera_grad_ref import camera_terms, clamp_scene, posed_matrices, project_camera_grads
from tests.util import full_path_grad_errors, rel_err, scene, settings_for, tans

pytestmark = pytest.mark.gpu
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
UNUSED = [3, 7, 11, 15, 16 + 2, 16 + 6, 16 + 10, 16 + 14]
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ptr = _lib.ptr


# ---- preprocess backward, C level ------------------------------------------------------------------------------------
def _scene(name):
    if name == "small":
        return scene(3000, 250, 130, 42, sigma_px=(0.5, 8.0))
    if name == "c2_1M":
        return scene(1_000_000, 980, 545, 77, sigma_px=(0.5, 4.0))
    cam = ring_cameras(3, 250, 130)[1]
    if name == "clamped":
        return (cam, *clamp_scene(cam, 20000, 3))
    # just beyond the 0.2 near cull
    return (cam, *clamp_scene(cam, 5000, 4, frac=0.0, z=(0.2005, 0.26), sigma_world=(0.003, 0.02)))


def _blend_upstream(cam, means, colors, opac, scales, rots, seed):
    """The kernels' own per-Gaussian upstream gradients of a depth / alpha / colour loss."""
    from splatco_b200.diff_gaussian_rasterization import rasterize_backward_state, rasterize_forward_state
    st = settings_for(cam, [1.0, 1.0, 1.0])
    ins = [t.cuda().contiguous() for t in (means, colors, opac, scales, rots)]
    H, W = cam.image_height, cam.image_width
    _, radii, state = rasterize_forward_state(*ins, st, depth_alpha=True)
    g = torch.Generator().manual_seed(seed)
    dC = (torch.randn(3, H, W, generator=g) / (H * W)).cuda()
    dD = (torch.randn(1, H, W, generator=g) / (H * W)).cuda()
    out = rasterize_backward_state(state, dC, ins[0], ins[3], ins[4], st, grad_depth=dD)
    return ins, st, radii, out["means2D"].contiguous(), out["conic"].contiguous(), out["depth"].contiguous()


def _preprocess(ins, st, radii, g2, gc, gd, camera):
    L = _lib.lib()
    P = int(ins[0].shape[0])
    m, s, q = ins[0], ins[3], ins[4]
    gm = torch.empty(P, 3, device="cuda")
    gs = torch.empty(P, 3, device="cuda")
    gq = torch.empty(P, 4, device="cuda")
    view, proj = st.viewmatrix.contiguous(), st.projmatrix.contiguous()
    args = (P, ptr(m), ptr(s), 3, ptr(q), 1.0, ptr(view), ptr(proj), float(st.tanfovx), float(st.tanfovy),
            int(st.image_height), int(st.image_width), ptr(radii), ptr(g2), ptr(gc), ptr(gm), ptr(gs), ptr(gq))
    stream = _lib.raw_stream(m.device)
    cam = None
    if camera:
        cam = torch.full((32,), float("nan"), device="cuda")
        ws = torch.full((L.splatco_camera_grad_ws_bytes(P),), 255, dtype=torch.uint8, device="cuda")
        _lib.check(L.splatco_preprocess_bwd_camera(*args, ptr(gd), ptr(ws), ptr(cam[:16]), ptr(cam[16:]), stream), "cam")
    elif gd is not None:
        _lib.check(L.splatco_preprocess_bwd_depth(*args, ptr(gd), stream), "depth")
    else:
        _lib.check(L.splatco_preprocess_bwd(*args, stream), "plain")
    torch.cuda.synchronize()
    return [t.cpu().numpy() for t in (gm, gs, gq)], None if cam is None else cam.cpu().numpy().astype(np.float64)


@pytest.mark.parametrize("depth", [False, True])
@pytest.mark.parametrize("name", ["small", "c2_1M", "clamped", "near_cull"])
def test_preprocess_bwd_camera_vs_fp64_autograd(name, depth):
    cam, means, colors, opac, scales, rots = _scene(name)
    ins, st, radii, g2, gc, gd = _blend_upstream(cam, means, colors, opac, scales, rots, 5)
    gd = gd if depth else None
    per0, _ = _preprocess(ins, st, radii, g2, gc, gd, camera=False)
    per1, cg = _preprocess(ins, st, radii, g2, gc, gd, camera=True)
    _, cg2 = _preprocess(ins, st, radii, g2, gc, gd, camera=True)
    for a, b in zip(per0, per1):
        assert a.tobytes() == b.tobytes()
    assert cg.tobytes() == cg2.tobytes()
    assert np.all(cg[UNUSED] == 0.0)
    vis = radii.cpu().numpy() > 0
    assert vis.sum() > 100
    tx, ty = tans(cam)
    H, W = cam.image_height, cam.image_width
    n = lambda t: None if t is None else t.cpu().numpy()[vis].astype(np.float64)
    args = (means.numpy()[vis], scales.numpy()[vis], rots.numpy()[vis], 1.0, cam.world_view_transform.numpy(),
            cam.full_proj_transform.numpy(), tx, ty, H, W, n(g2), n(gc), n(gd))
    gv, gp = project_camera_grads(*args)
    ref = np.concatenate([gv, gp])
    S = np.abs(camera_terms(*args)).sum(0)
    bound = 1e-3 * np.abs(ref) + 2.0 ** -18 * S
    assert np.all(np.abs(cg - ref) <= bound), (np.abs(cg - ref) / np.maximum(bound, 1e-30)).max()
    if name == "clamped":
        pv = np.concatenate([means.numpy()[vis], np.ones((vis.sum(), 1))], 1) @ cam.world_view_transform.numpy()
        assert (np.abs(pv[:, :2] / pv[:, 2:3]) > 1.3 * np.array([tx, ty])).any(1).mean() > 0.2


# ---- rasterizer vs the fp64 autograd composite -----------------------------------------------------------------------
@pytest.mark.parametrize("loss", ["colour", "depth", "alpha"])
@pytest.mark.parametrize("seed,W,H,M,sig", [(7, 64, 48, 300, (1.0, 6.0)), (13, 33, 17, 120, (2.0, 10.0))])
def test_rasterizer_camera_gradients_vs_fp64_composite(seed, W, H, M, sig, loss):
    from splatco_b200.diff_gaussian_rasterization import GaussianRasterizer
    cam, means, colors, opac, scales, rots = scene(M, W, H, seed, sigma_px=sig)
    bg = torch.tensor([1.0, 0.5, 0.25])
    tx, ty = tans(cam)
    g = torch.Generator().manual_seed(seed + 3)
    gC = torch.randn(3, H, W, generator=g, dtype=torch.float64) / (H * W)
    gD = torch.randn(1, H, W, generator=g, dtype=torch.float64) / (H * W)
    gA = torch.randn(1, H, W, generator=g, dtype=torch.float64) / (H * W)
    # GPU: the view matrix as the reference hands it over (a transposed view), the projection in fp64
    vt = cam.world_view_transform.t().contiguous().cuda().requires_grad_()
    pm = cam.full_proj_transform.double().cuda().requires_grad_()
    st = settings_for(cam, bg.tolist())._replace(viewmatrix=vt.t(), projmatrix=pm)
    img, radii, dep, alp = GaussianRasterizer(st)(
        means3D=means.cuda(), means2D=torch.zeros(M, 3, device="cuda"), shs=None, colors_precomp=colors.cuda(),
        opacities=opac.cuda(), scales=scales.cuda(), rotations=rots.cuda(), cov3D_precomp=None, depth_alpha=True)
    out, up = {"colour": (img, gC), "depth": (dep, gD), "alpha": (alp, gA)}[loss]
    out.backward(up.float().cuda())
    # fp64 reference on the C oracle's rectangles and depth order
    fw = DA.rasterize_forward(means.numpy(), colors.numpy(), opac.numpy(), scales.numpy(), rots.numpy(), 1.0,
                              cam.world_view_transform.numpy(), cam.full_proj_transform.numpy(), tx, ty, H, W,
                              bg.numpy())
    pr = fw["pr"]
    assert np.array_equal(radii.cpu().numpy(), pr.radii)
    d = torch.float64
    v64 = cam.world_view_transform.to(d).requires_grad_()
    p64 = cam.full_proj_transform.to(d).requires_grad_()
    xy, tz, conic, _ = CT.project(means.to(d), scales.to(d), rots.to(d), 1.0, v64, p64, tx, ty, H, W)
    order = torch.tensor(sorted(range(M), key=lambda i: (int(np.float32(pr.depths[i]).view(np.uint32)), i)))
    rimg, rdep, ralp = DA.composite_depth_alpha(xy, tz, conic, opac.to(d), colors.to(d), bg, torch.tensor(pr.rect),
                                                order, H, W)
    rout = {"colour": rimg, "depth": rdep, "alpha": ralp}[loss]
    gv, gp = torch.autograd.grad(rout, [v64, p64], up)
    got = np.concatenate([vt.grad.t().reshape(16).cpu().numpy(), pm.grad.reshape(16).cpu().numpy()])
    want = np.concatenate([gv.reshape(16).numpy(), gp.reshape(16).numpy()])
    assert pm.grad.dtype == torch.float64 and vt.grad.dtype == torch.float32
    assert np.all(got[UNUSED] == 0.0)
    assert rel_err(got, want) < 5e-3, (got, want)      # the fp32-blend bar of tests/test_oracle_depth_alpha.py


# ---- decode --------------------------------------------------------------------------------------------------------
class _Cam:
    def __init__(self, center, uid):
        self.camera_center = center
        self.uid = uid


def _decode_ref_cam_grad(d, level):
    from oracle import decode_oracle as D
    dd = torch.float64
    p = {k[len("param."):]: torch.from_numpy(d[k]).to(dd if d[k].dtype == np.float32 else None) for k in d.files
         if k.startswith("param.")}
    ins = {k: torch.from_numpy(d[f"in.{k}"]).to(dd) for k in ("_anchor", "_offset", "_anchor_feat", "_scaling")}
    cam = torch.from_numpy(d["cam_center"]).to(dd).requires_grad_()
    outs = D.decode(p, ins["_anchor_feat"], ins["_anchor"], ins["_offset"], torch.exp(ins["_scaling"]),
                    torch.from_numpy(d["vis"]), cam, level, int(d["K"]), appearance_dim=int(d["appearance_dim"]),
                    uid=int(d["uid"]), dists=bool(d["dists"]))
    loss = sum((t * torch.from_numpy(d[f"L{level}.w.{nm}"]).to(dd)).sum()
               for nm, t in zip(["xyz", "color", "opacity", "scaling", "rot"], outs[:5]))
    loss.backward()
    return cam.grad.numpy()


def _gpu_decode_grads(d, level, cam_grad):
    from splatco_b200.gaussian_renderer import generate_neural_gaussians
    from tests.test_decode_gpu import NAMES, named_leaves, pc_from_fixture
    pc = pc_from_fixture(d)
    pc.feat_planes._feat.activate_level = level
    cam = torch.from_numpy(d["cam_center"]).cuda().requires_grad_(cam_grad)
    outs = generate_neural_gaussians(_Cam(cam, int(d["uid"])), pc, torch.from_numpy(d["vis"]).cuda(), is_training=True)
    loss = sum((t * torch.from_numpy(d[f"L{level}.w.{nm}"]).cuda()).sum() for nm, t in zip(NAMES, outs[:5]))
    loss.backward()
    leaves = {k: v.grad.detach().clone() for k, v in named_leaves(pc).items() if v.grad is not None}
    return (cam.grad.cpu().numpy() if cam_grad else None), leaves


@pytest.mark.parametrize("packed", [False, True], ids=["planar", "channel_last"])
@pytest.mark.parametrize("impl", [1, 2])
@pytest.mark.parametrize("level", [0, 2])
@pytest.mark.parametrize("tag", ["base", "variants"])
def test_decode_camera_gradient_vs_fp64_oracle(tag, level, impl, packed):
    from splatco_b200 import decode
    L = _lib.lib()
    d = np.load(os.path.join(GOLD, f"decode_{tag}.npz"))
    prev_impl, prev_pack = L.splatco_decode_get_impl(), decode.PACK_PLANES
    try:
        L.splatco_decode_set_impl(impl)
        decode.PACK_PLANES = packed
        _, off = _gpu_decode_grads(d, level, False)
        _, off2 = _gpu_decode_grads(d, level, False)
        got, on = _gpu_decode_grads(d, level, True)
    finally:
        L.splatco_decode_set_impl(prev_impl)
        decode.PACK_PLANES = prev_pack
    want = _decode_ref_cam_grad(d, level)
    assert rel_err(got, want, floor_frac=3e-3) < 1e-3, (got, want)
    assert set(off) == set(on)
    # the per-anchor rows are bitwise those of the camera-off call wherever the camera-off backward itself is bitwise
    # reproducible (impl 1 reduces its weight gradients with atomics, which feeds run-to-run rounding into these rows)
    for k in off:
        a, b = off[k].cpu().numpy(), on[k].cpu().numpy()
        if k in ("_anchor", "_offset", "_anchor_feat", "_scaling") and a.tobytes() == off2[k].cpu().numpy().tobytes():
            assert a.tobytes() == b.tobytes(), k
        else:
            assert rel_err(b, a) < 1e-3, k


def test_decode_variants_cover_distances_and_appearance():
    flags = {t: np.load(os.path.join(GOLD, f"decode_{t}.npz")) for t in ("base", "variants")}
    assert {bool(v["dists"]) for v in flags.values()} == {False, True}
    assert max(int(v["appearance_dim"]) for v in flags.values()) > 0


# ---- render() end to end with a learnable pose -------------------------------------------------------------------------
def _posed_cam(cam, delta):
    wv, full, centre = posed_matrices(cam.world_view_transform.to(delta), cam.full_proj_transform.to(delta), delta)
    return SimpleNamespace(uid=cam.uid, image_width=cam.image_width, image_height=cam.image_height, FoVx=cam.FoVx,
                           FoVy=cam.FoVy, world_view_transform=wv.float(), full_proj_transform=full.float(),
                           camera_center=centre.float())


def test_full_path_c1_pose_gradient_vs_fp64_chain():
    """render() on the bench's C1 model with a camera built from a learnable se(3) delta; the delta's gradient against
    the chain oracle decode -> depth / alpha C reference -> fp64 projection autograd."""
    import bench
    from oracle import decode_oracle as D
    from oracle import raster as R
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
    delta0 = torch.tensor([0.002, -0.003, 0.001, 0.01, -0.02, 0.015], dtype=torch.float64)
    delta = delta0.clone().to(dev).requires_grad_()
    cam_d = _posed_cam(cam, delta)
    vm = prefilter_voxel(cam_d, pc, bench.PIPE, bg)
    pkg = render(cam_d, pc, bench.PIPE, bg, visible_mask=vm, depth_alpha=True)
    g = torch.Generator().manual_seed(21)
    dC = torch.randn(3, H, W, generator=g) / (3 * H * W)
    dD = torch.randn(1, H, W, generator=g) / (H * W)
    dA = torch.randn(1, H, W, generator=g) / (H * W)
    torch.autograd.backward([pkg["render"], pkg["depth"], pkg["alpha"]], [dC.to(dev), dD.to(dev), dA.to(dev)])
    got = delta.grad.cpu().numpy()
    # reference chain on the CPU
    cam_c = _posed_cam(cam, delta0.clone())
    view = cam_c.world_view_transform.detach().numpy()
    proj = cam_c.full_proj_transform.detach().numpy()
    cpu = bench.build_model(cfg, "cpu")
    cpu.feat_planes.Q0 = 0.0
    p = {"feat." + k: v for k, v in cpu.feat_planes._feat.state_dict().items()}
    for name in ("mlp_opacity", "mlp_cov", "mlp_color"):
        p.update({f"{name}.{k}": v for k, v in getattr(cpu, name).state_dict().items()})
    tx, ty = math.tan(cam.FoVx * 0.5), math.tan(cam.FoVy * 0.5)
    scaling = torch.exp(cpu._scaling).detach()
    radii_a = R.visible_filter(cpu._anchor.detach().numpy(), scaling.numpy()[:, :3],
                               torch.nn.functional.normalize(cpu._rotation).detach().numpy(), 1.0, view, proj, tx, ty, H, W)
    vis = torch.from_numpy(radii_a > 0)
    assert np.array_equal(vm.cpu().numpy(), vis.numpy())
    centre = cam_c.camera_center.detach().clone().requires_grad_()
    xyz, color, opacity, scl, rot, _, mask = D.decode(p, cpu._anchor_feat.detach(), cpu._anchor.detach(),
                                                      cpu._offset.detach(), scaling, vis, centre, 2, K)
    assert np.array_equal(pkg["selection_mask"].cpu().numpy(), mask.numpy())
    a = [t.detach().numpy() for t in (xyz, color, opacity, scl, rot)]
    fw = DA.rasterize_forward(a[0], a[1], a[2], a[3], a[4], 1.0, view, proj, tx, ty, H, W, np.ones(3, np.float32))
    bw = DA.rasterize_backward(fw, a[0], a[1], a[3], a[4], 1.0, view, proj, tx, ty, H, W, np.ones(3, np.float32),
                               dC.numpy(), dD.numpy(), dA.numpy())
    torch.autograd.backward([xyz, color, opacity, scl, rot],
                            [torch.from_numpy(bw[k]) for k in ("means3D", "colors", "opacities", "scales", "rotations")])
    keep = fw["pr"].radii > 0
    gv, gp = project_camera_grads(a[0][keep], a[3][keep], a[4][keep], 1.0, view, proj, tx, ty, H, W,
                                  bw["means2D"][keep], bw["conic"][keep], bw["depth"][keep])
    d64 = delta0.clone().requires_grad_()
    wv, full, c = posed_matrices(cam.world_view_transform.double(), cam.full_proj_transform.double(), d64)
    torch.autograd.backward([wv, full, c], [torch.from_numpy(gv).reshape(4, 4), torch.from_numpy(gp).reshape(4, 4),
                                            centre.grad.double()])
    want = d64.grad.numpy()
    e = full_path_grad_errors(got, want)
    assert e["l2"] < 5e-3, (got, want, e)


# ---- plumbing ---------------------------------------------------------------------------------------------------------
def _render_setup(N=3000, seed=5, W=160, H=112):
    from tests.test_render_gpu import _cams, _model
    return _model(N=N, seed=seed), list(_cams(W, H))


def test_camera_tensors_without_grad_keep_launches_and_outputs():
    """A camera whose tensors require grad changes nothing in the forward: under no_grad, and in grad mode up to the
    backward, the launches and the image are those of a plain camera."""
    from splatco_b200.gaussian_renderer import prefilter_voxel, render
    from tests.test_render_gpu import PIPE
    pc, cams = _render_setup()
    bg = torch.ones(3, device="cuda")
    L = _lib.lib()

    def run(cam, grad):
        n0 = L.splatco_launch_count()
        with torch.set_grad_enabled(grad):
            pkg = render(cam, pc, PIPE, bg, visible_mask=prefilter_voxel(cam, pc, PIPE, bg))
        torch.cuda.synchronize()
        return L.splatco_launch_count() - n0, pkg["render"].detach().clone(), pkg["render"]

    zero = lambda rg: torch.zeros(6, dtype=torch.float64, device="cuda", requires_grad=rg)
    plain, learn = _posed_cam(cams[0], zero(False)), _posed_cam(cams[0], zero(True))
    assert learn.world_view_transform.requires_grad and learn.camera_center.requires_grad
    assert not plain.world_view_transform.requires_grad
    for grad in (False, True):
        run(plain, grad)                                 # warms the per-iteration caches of this grad mode
        n_plain, img_plain, _ = run(plain, grad)
        n_learn, img_learn, out = run(learn, grad)
        assert n_plain == n_learn and torch.equal(img_plain, img_learn), (grad, n_plain, n_learn)
        assert out.requires_grad == grad


def test_two_views_one_backward_equals_separate_and_eval_mode():
    from splatco_b200.gaussian_renderer import prefilter_voxel, render
    from tests.test_render_gpu import PIPE
    pc, cams = _render_setup()
    bg = torch.ones(3, device="cuda")
    deltas = [torch.tensor(v, dtype=torch.float64, device="cuda", requires_grad=True)
              for v in ([0.001, 0.002, -0.001, 0.01, 0.0, -0.01], [-0.002, 0.0, 0.001, 0.0, 0.02, 0.005])]

    def loss_of(i):
        c = _posed_cam(cams[i], deltas[i])
        pkg = render(c, pc, PIPE, bg, visible_mask=prefilter_voxel(c, pc, PIPE, bg), depth_alpha=True)
        return pkg["render"].square().mean() + 0.1 * pkg["depth"].mean() + pkg["alpha"].mean()

    (loss_of(0) + loss_of(1)).backward()
    both = [dl.grad.clone() for dl in deltas]
    for dl in deltas:
        dl.grad = None
    loss_of(0).backward()
    loss_of(1).backward()
    for a, dl in zip(both, deltas):
        assert a.abs().max() > 0
        assert (a - dl.grad).abs().max() <= 1e-4 * a.abs().max()
    pc.eval()
    try:
        for dl in deltas:
            dl.grad = None
        loss_of(0).backward()
        assert torch.isfinite(deltas[0].grad).all() and deltas[0].grad.abs().max() > 0
    finally:
        pc.train()


def test_speculative_path_equals_direct_rasterizer_call():
    from splatco_b200.diff_gaussian_rasterization import GaussianRasterizer
    from splatco_b200.gaussian_renderer import _settings, generate_neural_gaussians, prefilter_voxel, render
    from tests.test_render_gpu import PIPE
    pc, cams = _render_setup()
    bg = torch.ones(3, device="cuda")
    base = cams[1]
    out = []
    for fast in (True, False):
        wv = base.world_view_transform.cuda().clone().requires_grad_()
        full = base.full_proj_transform.cuda().clone().requires_grad_()
        c = SimpleNamespace(uid=0, image_width=base.image_width, image_height=base.image_height, FoVx=base.FoVx,
                            FoVy=base.FoVy, world_view_transform=wv, full_proj_transform=full,
                            camera_center=base.camera_center.cuda())
        vm = prefilter_voxel(c, pc, PIPE, bg)
        if fast:
            img = render(c, pc, PIPE, bg, visible_mask=vm)["render"]
        else:
            xyz, color, opacity, scaling, rot, _, _ = generate_neural_gaussians(c, pc, vm, is_training=True)
            img, _ = GaussianRasterizer(_settings(c, PIPE, bg, 1.0))(
                means3D=xyz, means2D=torch.zeros_like(xyz), shs=None, colors_precomp=color, opacities=opacity,
                scales=scaling, rotations=rot, cov3D_precomp=None)
        out.append((img.detach().clone(), *torch.autograd.grad(img.square().mean(), [wv, full])))
    assert torch.equal(out[0][0], out[1][0])
    for a, b in zip(out[0][1:], out[1][1:]):
        assert a.abs().max() > 0 and (a - b).abs().max() <= 1e-5 * a.abs().max()


def test_empty_all_culled_and_zero_view_give_zero_camera_gradients():
    from splatco_b200.diff_gaussian_rasterization import GaussianRasterizer
    cam, means, colors, opac, scales, rots = scene(64, 50, 34, 5)
    z = lambda *s: torch.zeros(*s, device="cuda")

    def grads(vm, pm, m):
        vm = vm.cuda().clone().requires_grad_()
        pm = pm.cuda().clone().requires_grad_()
        st = settings_for(cam, [0.2, 0.4, 0.6])._replace(viewmatrix=vm, projmatrix=pm)
        n = m.shape[0]
        img, radii, dep, alp = GaussianRasterizer(st)(
            means3D=m.cuda(), means2D=z(n, 3), shs=None, colors_precomp=colors[:n].cuda(), opacities=opac[:n].cuda(),
            scales=scales[:n].cuda(), rotations=rots[:n].cuda(), cov3D_precomp=None, depth_alpha=True)
        (img.sum() + dep.sum() + alp.sum()).backward()
        return vm.grad, pm.grad
    for vm, pm, m in ((cam.world_view_transform, cam.full_proj_transform, torch.zeros(0, 3)),         # P = 0
                      (cam.world_view_transform, cam.full_proj_transform, (cam.camera_center * 3.0)[None].repeat(64, 1)),
                      (torch.zeros(4, 4), cam.full_proj_transform, means)):                         # V = 0: all culled
        gv, gp = grads(vm, pm, m)
        assert gv is not None and gp is not None
        assert torch.count_nonzero(gv) == 0 and torch.count_nonzero(gp) == 0
    # the decode with no visible anchor
    from tests.test_decode_gpu import pc_from_fixture
    from splatco_b200.gaussian_renderer import generate_neural_gaussians
    d = np.load(os.path.join(GOLD, "decode_base.npz"))
    pc = pc_from_fixture(d)
    centre = torch.from_numpy(d["cam_center"]).cuda().requires_grad_()
    outs = generate_neural_gaussians(_Cam(centre, 0), pc, torch.zeros(int(d["N"]), dtype=torch.bool, device="cuda"),
                                     is_training=True)
    (outs[0].sum() + outs[1].sum() + centre.sum() * 0).backward()
    assert centre.grad is not None and torch.count_nonzero(centre.grad) == 0
