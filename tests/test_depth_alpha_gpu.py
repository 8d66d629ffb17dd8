"""GPU tests of the depth and alpha maps: the kernels against the C reference (tests/depth_alpha_oracle.py), the
colour path left as it was, the autograd / render() plumbing and the whole decode + rasterizer path."""
import math

import numpy as np
import pytest
import torch

from tests import depth_alpha_oracle as DA
from tests.util import full_path_grad_errors, rel_err, scene, settings_for, tans

pytestmark = pytest.mark.gpu

FWD_SCENES = [
    (1, 64, 48, 300, (1.0, 6.0)), (2, 250, 130, 5000, (0.5, 4.0)), (3, 256, 256, 100000, (0.5, 4.0)),
    (4, 980, 545, 60000, (0.5, 8.0)), (5, 97, 33, 2000, (4.0, 40.0)),          # tests/test_raster_gpu.py's scenes
    (6, 1, 17, 200, (0.5, 6.0)), (7, 17, 1, 200, (0.5, 6.0)), (8, 15, 15, 300, (0.5, 6.0)), (9, 250, 131, 5000, (0.5, 6.0)),
]


def _to(d, *ts):
    return [t.to(d) for t in ts]


def _da_oracle_forward(cam, means, colors, opac, scales, rots, bg, scale_mod=1.0):
    tx, ty = tans(cam)
    return DA.rasterize_forward(means.numpy(), colors.numpy(), opac.numpy(), scales.numpy(), rots.numpy(), scale_mod,
                                cam.world_view_transform.numpy(), cam.full_proj_transform.numpy(), tx, ty,
                                cam.image_height, cam.image_width, np.asarray(bg, np.float32))


def _da_oracle_backward(fw, cam, means, colors, scales, rots, bg, dC, dD, dA):
    tx, ty = tans(cam)
    return DA.rasterize_backward(fw, means.numpy(), colors.numpy(), scales.numpy(), rots.numpy(), 1.0,
                                 cam.world_view_transform.numpy(), cam.full_proj_transform.numpy(), tx, ty,
                                 cam.image_height, cam.image_width, np.asarray(bg, np.float32), dC, dD, dA)


def _image_ws(state):
    from tests.test_raster_gpu import unpack_state
    g = unpack_state(state)
    return g["final_T"], g["n_contrib"]


def _both_forwards(means, colors, opac, scales, rots, st):
    """The colour-only and the depth/alpha forward on the same inputs: (color, final_T, n_contrib) of each, the maps."""
    from splatco_b200.diff_gaussian_rasterization import rasterize_forward_state
    ins = [t.cuda() for t in (means, colors, opac, scales, rots)]
    c0, r0, s0 = rasterize_forward_state(*ins, st)
    c1, r1, s1 = rasterize_forward_state(*ins, st, depth_alpha=True)
    torch.cuda.synchronize()
    assert torch.equal(r0, r1)
    return (c0, *_image_ws(s0)), (c1, *_image_ws(s1)), s1.depth, s1.alpha, s1


def _assert_colour_identical(a, b):
    for x, y in zip(a, b):
        x = x.cpu().numpy() if torch.is_tensor(x) else x
        y = y.cpu().numpy() if torch.is_tensor(y) else y
        assert x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes()


@pytest.mark.parametrize("seed,W,H,M,sig", FWD_SCENES)
def test_forward_colour_bit_identical_and_maps_match_oracle(seed, W, H, M, sig):
    cam, means, colors, opac, scales, rots = scene(M, W, H, seed, sigma_px=sig)
    bg = [1.0, 1.0, 1.0] if seed % 2 else [0.1, 0.2, 0.3]
    plain, da, depth, alpha, st = _both_forwards(means, colors, opac, scales, rots, settings_for(cam, bg))
    _assert_colour_identical(plain, da)
    assert depth.shape == (1, H, W) and alpha.shape == (1, H, W)
    fw = _da_oracle_forward(cam, means, colors, opac, scales, rots, bg)
    frag = fw["fragile"]
    assert frag.mean() < 0.02
    vis = fw["pr"].radii > 0
    zmax = float(np.abs(fw["pr"].depths[vis]).max()) if vis.any() else 1.0
    d, a = depth.cpu().numpy()[0], alpha.cpu().numpy()[0]
    assert np.abs(a - fw["alpha"])[~frag].max() <= 1e-4
    assert np.abs(d - fw["depth"])[~frag].max() <= 1e-4 * zmax
    # alpha is 1 - final_T of the same walk
    assert np.array_equal(a, (np.float32(1) - da[1]).astype(np.float32))


@pytest.mark.parametrize("name", ["needle_s1000_op0.9", "needle_s3000_op0.02", "straddle", "batch_edges",
                                  "geometry_1x17", "geometry_250x131"])
def test_depth_alpha_forward_inherits_the_cull_filters(name):
    """Needles, opacities at the 1/255 cut, 512-splat batch edges and odd image sizes (tests/test_blend_filters_gpu.py's
    scenes): the depth / alpha kernel makes exactly the colour kernel's decisions."""
    from tests.test_blend_filters_gpu import SCENES
    sc = SCENES[name]()
    means, colors, opac, scales, rots = sc.tensors()
    plain, da, depth, alpha, st = _both_forwards(means, colors, opac, scales, rots, settings_for(sc.cam, sc.bg))
    assert st.R > 0
    _assert_colour_identical(plain, da)
    assert torch.isfinite(depth).all() and torch.equal(alpha[0], 1.0 - da[0].new_tensor(da[1]))


def _rast(cam, bg):
    from splatco_b200.diff_gaussian_rasterization import GaussianRasterizer
    return GaussianRasterizer(settings_for(cam, bg))


def _upstream(H, W, seed, which):
    g = torch.Generator().manual_seed(seed)
    dC = torch.randn(3, H, W, generator=g) / (3 * H * W) if which in ("all",) else None
    dD = torch.randn(1, H, W, generator=g) / (H * W) if which in ("depth", "all") else None
    dA = torch.randn(1, H, W, generator=g) / (H * W) if which in ("alpha", "all") else None
    return dC, dD, dA


def _gpu_backward(cam, bg, means, colors, opac, scales, rots, dC, dD, dA):
    m, c, o, s, q = [t.cuda().requires_grad_() for t in (means, colors, opac, scales, rots)]
    m2d = torch.zeros_like(m, requires_grad=True)
    img, radii, depth, alpha = _rast(cam, bg)(means3D=m, means2D=m2d, shs=None, colors_precomp=c, opacities=o, scales=s,
                                             rotations=q, cov3D_precomp=None, depth_alpha=True)
    outs, grads = zip(*[(t, gt.cuda()) for t, gt in ((img, dC), (depth, dD), (alpha, dA)) if gt is not None])
    torch.autograd.backward(outs, grads)
    z = lambda t, like: t if t is not None else torch.zeros_like(like)
    return dict(means3D=m.grad, colors=z(c.grad, c), opacities=o.grad, scales=s.grad, rotations=q.grad, means2D=m2d.grad)


def _check_backward(cam, bg, means, colors, opac, scales, rots, dC, dD, dA, tol=1e-3):
    fw = _da_oracle_forward(cam, means, colors, opac, scales, rots, bg)
    got = _gpu_backward(cam, bg, means, colors, opac, scales, rots, dC, dD, dA)
    n = lambda t: None if t is None else t.numpy()
    bw = _da_oracle_backward(fw, cam, means, colors, scales, rots, bg, n(dC), n(dD), n(dA))
    errs = {}
    for k in ("means3D", "colors", "opacities", "scales", "rotations", "means2D"):
        g, w = got[k].cpu().numpy(), bw[k]
        if k == "means2D":
            g, w = g[:, :2], w[:, :2]
        errs[k] = rel_err(g, w)
    assert max(errs.values()) < tol, errs


@pytest.mark.parametrize("which", ["depth", "alpha", "all"])
@pytest.mark.parametrize("seed,W,H,M,sig", [(41, 64, 48, 300, (1.0, 6.0)), (42, 250, 130, 5000, (0.5, 4.0)),
                                           (43, 97, 33, 2000, (4.0, 40.0))])
def test_backward_vs_oracle(seed, W, H, M, sig, which):
    cam, means, colors, opac, scales, rots = scene(M, W, H, seed, sigma_px=sig)
    _check_backward(cam, [1.0, 1.0, 1.0], means, colors, opac, scales, rots, *_upstream(H, W, seed, which))


def test_backward_c2_size_vs_oracle():
    W, H, M = 980, 545, 1_000_000
    cam, means, colors, opac, scales, rots = scene(M, W, H, 77, sigma_px=(0.5, 4.0))
    _check_backward(cam, [1.0, 1.0, 1.0], means, colors, opac, scales, rots, *_upstream(H, W, 5, "all"))


def test_zero_map_gradients_equal_colour_only_and_none_is_the_colour_path():
    W, H, M = 250, 130, 5000
    cam, means, colors, opac, scales, rots = scene(M, W, H, 42, sigma_px=(0.5, 4.0))
    bg = [1.0, 1.0, 1.0]
    dC = _upstream(H, W, 3, "all")[0]
    m, c, o, s, q = [t.cuda().requires_grad_() for t in (means, colors, opac, scales, rots)]
    m2d = torch.zeros_like(m, requires_grad=True)
    ins = dict(means3D=m, means2D=m2d, shs=None, colors_precomp=c, opacities=o, scales=s, rotations=q, cov3D_precomp=None)

    def grads():
        out = [t.grad.clone() for t in (m, c, o, s, q, m2d)]
        for t in (m, c, o, s, q, m2d):
            t.grad = None
        return out

    img, _ = _rast(cam, bg)(**ins)
    img.backward(dC.cuda())
    ref = grads()
    img, _, depth, alpha = _rast(cam, bg)(**ins, depth_alpha=True)
    torch.autograd.backward([img, depth, alpha], [dC.cuda(), torch.zeros_like(depth), torch.zeros_like(alpha)])
    zero = grads()
    img, _, depth, alpha = _rast(cam, bg)(**ins, depth_alpha=True)
    img.backward(dC.cuda())                              # depth and alpha receive no gradient: None
    none = grads()
    # Bit identity with the colour-only backward is NOT asserted: the blend backward sums per-Gaussian gradients with
    # fp32 atomics, so even two runs of the colour-only backward on the same inputs agree only to rounding.  What is
    # asserted instead: explicit zero maps agree to 1e-6 of max|g|, and with None maps the depth/alpha Function runs
    # exactly the colour-only entry points (splatco_blend_bwd + splatco_preprocess_bwd), checked by counting calls.
    for a, b, n in zip(ref, zero, none):
        assert (a - b).abs().max().item() <= 1e-6 * max(a.abs().max().item(), 1e-30)
        assert (a - n).abs().max().item() <= 1e-6 * max(a.abs().max().item(), 1e-30)
    from splatco_b200 import _lib
    L = _lib.lib()
    names = ("splatco_blend_bwd", "splatco_preprocess_bwd", "splatco_blend_bwd_depth_alpha", "splatco_preprocess_bwd_depth")
    orig = {k: getattr(L, k) for k in names}
    calls = []

    def spy(k):
        return lambda *args: calls.append(k) or orig[k](*args)

    try:
        for k in names:
            setattr(L, k, spy(k))
        img, _, depth, alpha = _rast(cam, bg)(**ins, depth_alpha=True)
        img.backward(dC.cuda())
        grads()
        assert calls == ["splatco_blend_bwd", "splatco_preprocess_bwd"], calls
        calls.clear()
        img, _, depth, alpha = _rast(cam, bg)(**ins, depth_alpha=True)
        depth.sum().backward()
        grads()
        assert calls == ["splatco_blend_bwd_depth_alpha", "splatco_preprocess_bwd_depth"], calls
    finally:
        for k in names:
            setattr(L, k, orig[k])


def test_edge_cases_empty_all_culled_and_colour_gradient_none():
    cam, means, colors, opac, scales, rots = scene(64, 50, 34, 5)
    bg = [0.2, 0.4, 0.6]
    rast = _rast(cam, bg)
    bgt = torch.tensor(bg, device="cuda")[:, None, None].expand(3, 34, 50)
    z = lambda *s: torch.zeros(*s, device="cuda")
    img, radii, depth, alpha = rast(means3D=z(0, 3), means2D=z(0, 3), shs=None, colors_precomp=z(0, 3),
                                    opacities=z(0, 1), scales=z(0, 3), rotations=z(0, 4), cov3D_precomp=None,
                                    depth_alpha=True)
    assert radii.numel() == 0 and torch.allclose(img, bgt)
    assert depth.shape == (1, 34, 50) and not depth.any() and not alpha.any()
    behind = (cam.camera_center * 3.0)[None].repeat(64, 1)
    m = behind.cuda().requires_grad_()
    img, radii, depth, alpha = rast(means3D=m, means2D=torch.zeros_like(m), shs=None, colors_precomp=colors.cuda(),
                                    opacities=opac.cuda(), scales=scales.cuda(), rotations=rots.cuda(),
                                    cov3D_precomp=None, depth_alpha=True)
    assert (radii == 0).all() and torch.allclose(img, bgt) and not depth.any() and not alpha.any()
    (depth.sum() + alpha.sum()).backward()
    assert torch.count_nonzero(m.grad) == 0
    # only the colour gradient None: depth and alpha losses alone
    cam, means, colors, opac, scales, rots = scene(2000, 97, 33, 43, sigma_px=(1.0, 8.0))
    m = means.cuda().requires_grad_()
    o = opac.cuda().requires_grad_()
    img, radii, depth, alpha = _rast(cam, bg)(means3D=m, means2D=torch.zeros_like(m), shs=None,
                                              colors_precomp=colors.cuda(), opacities=o, scales=scales.cuda(),
                                              rotations=rots.cuda(), cov3D_precomp=None, depth_alpha=True)
    (depth.mean() - alpha.mean()).backward()
    assert torch.isfinite(m.grad).all() and m.grad.abs().max() > 0 and o.grad.abs().max() > 0


# ---- render() -----------------------------------------------------------------------------------------------
def test_render_fast_path_equals_plain_calls():
    from splatco_b200 import diff_gaussian_rasterization as dgr
    from splatco_b200.gaussian_renderer import _settings, generate_neural_gaussians, prefilter_voxel, render
    from tests.test_render_gpu import PIPE, _cams, _model
    W, H = 200, 144
    pc = _model()
    far, near = _cams(W, H)
    bg = torch.ones(3, device="cuda")
    dgr._r_guess.clear()
    Rs = []
    for cam in (far, near, far, near):          # no guess -> guess too small -> too large -> about right
        vm = prefilter_voxel(cam, pc, PIPE, bg)
        with torch.no_grad():
            pkg = render(cam, pc, PIPE, bg, visible_mask=vm, depth_alpha=True)
            xyz, color, opacity, scaling, rot, nopac, mask = generate_neural_gaussians(cam, pc, vm, is_training=True)
            st = _settings(cam, PIPE, bg, 1.0)
            img, radii, state = dgr.rasterize_forward_state(xyz, color, opacity, scaling, rot, st, depth_alpha=True)
        Rs.append(state.R)
        assert torch.equal(pkg["radii"], radii)
        assert torch.equal(pkg["render"], img)
        assert torch.equal(pkg["depth"], state.depth) and torch.equal(pkg["alpha"], state.alpha)
    assert Rs[1] > 1.5 * Rs[0], f"cameras do not exercise the overflow path: {Rs}"
    # depth_alpha=False: today's keys and image; a speculation queued for the other flag is not taken
    vm = prefilter_voxel(near, pc, PIPE, bg)
    with torch.no_grad():
        pkg = render(near, pc, PIPE, bg, visible_mask=vm)
        pkg_da = render(near, pc, PIPE, bg, visible_mask=prefilter_voxel(near, pc, PIPE, bg), depth_alpha=True)
        xyz, color, opacity, scaling, rot, _, _ = generate_neural_gaussians(near, pc, vm, is_training=True, _raster_settings=st,
                                                                            _depth_alpha=True)
        img, _, state = dgr.rasterize_forward_state(xyz, color, opacity, scaling, rot, st)     # flag differs
    assert set(pkg) == {"render", "viewspace_points", "visibility_filter", "radii", "selection_mask", "neural_opacity",
                        "scaling"}
    assert set(pkg_da) == set(pkg) | {"depth", "alpha"}
    assert torch.equal(pkg["render"], pkg_da["render"]) and state.depth is None and torch.equal(img, pkg["render"])


def test_eval_mode_render_with_depth_alpha():
    from splatco_b200.gaussian_renderer import prefilter_voxel, render
    from tests.test_render_gpu import PIPE, _cams, _model
    pc = _model(N=3000, seed=6)
    cam = _cams(160, 112)[1]
    bg = torch.zeros(3, device="cuda")
    img_train = render(cam, pc, PIPE, bg, visible_mask=prefilter_voxel(cam, pc, PIPE, bg))["render"].detach().clone()
    pc.eval()
    with torch.no_grad():
        pkg = render(cam, pc, PIPE, bg, visible_mask=prefilter_voxel(cam, pc, PIPE, bg), depth_alpha=True)
    pc.train()
    assert set(pkg) == {"render", "viewspace_points", "visibility_filter", "radii", "depth", "alpha"}
    assert torch.equal(pkg["render"], img_train)
    a = pkg["alpha"]
    assert a.min() >= 0 and a.max() <= 1 and a.max() > 0.5 and (pkg["depth"] >= 0).all()


def test_full_path_c1_depth_alpha_vs_oracle():
    """prefilter_voxel -> render(depth_alpha=True) on the bench's C1 model with a loss on image, depth and alpha; the
    leaf gradients against the oracle decode followed by the depth / alpha C reference."""
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
    cam_d = cam.to(dev)
    vm = prefilter_voxel(cam_d, pc, bench.PIPE, bg)
    pkg = render(cam_d, pc, bench.PIPE, bg, visible_mask=vm, retain_grad=True, depth_alpha=True)
    dC, dD, dA = _upstream(H, W, 21, "all")
    torch.autograd.backward([pkg["render"], pkg["depth"], pkg["alpha"]], [dC.to(dev), dD.to(dev), dA.to(dev)])
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
    xyz, color, opacity, scl, rot, nopac, mask = D.decode(p, cpu._anchor_feat, cpu._anchor, cpu._offset, scaling, vis,
                                                          cam.camera_center, 2, K)
    assert np.array_equal(pkg["selection_mask"].cpu().numpy(), mask.numpy()), "the two decodes keep different Gaussians"
    a = [t.detach().numpy() for t in (xyz, color, opacity, scl, rot)]
    bgn = np.ones(3, np.float32)
    fw = DA.rasterize_forward(a[0], a[1], a[2], a[3], a[4], 1.0, view, proj, tx, ty, H, W, bgn)
    frag = fw["fragile"]
    assert np.abs(pkg["alpha"].detach().cpu().numpy()[0] - fw["alpha"])[~frag].max() <= 1e-3
    g = DA.rasterize_backward(fw, a[0], a[1], a[3], a[4], 1.0, view, proj, tx, ty, H, W, bgn, dC.numpy(), dD.numpy(),
                              dA.numpy())
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
    assert max(v[1] for v in worst.values()) < 5e-3, sorted(worst.items(), key=lambda kv: -kv[1][1])[:8]


def test_two_views_depth_alpha_losses_one_backward_equals_sum_of_separate():
    from splatco_b200.gaussian_renderer import prefilter_voxel, render
    from tests.test_render_gpu import PIPE, _cams, _model
    W, H = 160, 112
    pc = _model(N=3000, seed=5)
    cams = list(_cams(W, H))
    bg = torch.ones(3, device="cuda")
    params = [p for p in pc.parameters() if p.requires_grad]

    def loss_of(i):
        pkg = render(cams[i], pc, PIPE, bg, visible_mask=prefilter_voxel(cams[i], pc, PIPE, bg), depth_alpha=True)
        return pkg["render"].mean() + 0.1 * pkg["depth"].square().mean() + (1.0 - pkg["alpha"]).abs().mean()

    for p in params:
        p.grad = None
    (loss_of(0) + loss_of(1)).backward()
    g_sum = [p.grad.clone() if p.grad is not None else None for p in params]
    for p in params:
        p.grad = None
    for i in range(2):
        loss_of(i).backward()
    n = 0
    for p, a in zip(params, g_sum):
        b = p.grad
        assert (a is None) == (b is None)
        if a is None:
            continue
        n += 1
        assert (a - b).abs().max().item() <= 1e-4 * max(b.abs().max().item(), 1e-12) + 1e-9, tuple(p.shape)
    assert n > 10
