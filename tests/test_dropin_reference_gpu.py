"""The drop-in behind the REFERENCE's real model classes (INTEGRATION.md options A and B).

Needs the reference's own Python sources, staged by `python oracle/build_ref.py` under the git-ignored oracle/_ref/
(they travel to the GPU box with gpurun); skipped when they are absent.  With splatco_shims standing in for the
import-time-only packages, the test

  * constructs the reference's real `GaussianModel` (scene/gaussian_model.py:226: its `GaussianLearner` :183 with the
    integer-list bbox, `FeaturePlanes` :97 whose `k0s` has four entries, the three MLP heads :316-337) on the GPU,
    with per-anchor Parameters set the way `create_from_pcd` sets them (:470-508);
  * option A: the reference's own `gaussian_renderer.prefilter_voxel` / `render` (its PyTorch decode,
    gaussian_renderer/__init__.py:18-188) on top of `splatco_b200.diff_gaussian_rasterization`;
  * option B: `splatco_b200.gaussian_renderer.prefilter_voxel` / `render` on the same model object;
and requires the two to agree: prefilter mask and opacity mask identical, image <= 1e-4 on 99.99 % of the pixels, every
trained leaf's gradient within 1e-3 in norm (TriPlaneAttention's conv weights 3e-3; tests/util.full_path_grad_errors),
BatchNorm running statistics updated identically.
"""
import os
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from tests.util import full_path_grad_errors

pytestmark = pytest.mark.gpu
# the reference's decode runs through torch / cuDNN here: keep its convolutions and matmuls in true fp32
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")


def _reference_modules():
    if not os.path.exists(os.path.join(REF, "scene", "gaussian_model.py")):
        pytest.skip("needs the original SplatCo Python sources staged under oracle/_ref by oracle/build_ref.py; the "
                    "repository does not include them (its decode is pinned by tests/golden/decode_*.npz)")
    import splatco_shims
    splatco_shims.install(hot_path="rasterizer")          # option A aliasing; the reference's gaussian_renderer stays its own
    if REF not in sys.path:
        sys.path.insert(0, REF)
    for name in [m for m in sys.modules if m == "gaussian_renderer" or m.startswith("gaussian_renderer.")]:
        if "splatco_b200" in (getattr(sys.modules[name], "__file__", None) or ""):
            del sys.modules[name]
    import gaussian_renderer as ref_gr
    from scene import gaussian_model as gm
    assert REF in os.path.abspath(ref_gr.__file__) and REF in os.path.abspath(gm.__file__)
    return ref_gr, gm


def _real_model(gm, N=20000, K=10, plane_size=512, seed=3):
    mp = SimpleNamespace(plane_size=plane_size, num_channels=15, mlp_dim=168, subplane_multiplier=1, bbox_scale=1.0,
                         scene_center=[0.0, 0.0, 0.0], scene_length=[4.0, 4.0, 4.0], contractor=True)
    torch.manual_seed(seed)
    pc = gm.GaussianModel(feat_dim=32, n_offsets=K, voxel_size=0.01, update_depth=3, update_init_factor=16,
                          update_hierachy_factor=4, use_feat_bank=False, appearance_dim=0, ratio=1,
                          add_opacity_dist=False, add_cov_dist=False, add_color_dist=False, model_params=mp)
    g = torch.Generator().manual_seed(seed + 1)
    anchor = (torch.rand(N, 3, generator=g) * 2 - 1) * 1.2
    anchor[: N // 10] *= 2.2                                   # a shell outside the planes' [-2,2]^3 box
    s0 = 1.0 / N ** (1 / 3)
    dev = "cuda"
    P = lambda t, rg=True: torch.nn.Parameter(t.to(dev).requires_grad_(rg))
    pc._anchor = P(anchor)
    pc._offset = P(torch.randn(N, K, 3, generator=g) * 0.5)
    pc._anchor_feat = P(torch.randn(N, 32, generator=g) * 0.3)
    pc._scaling = P(torch.log(s0 * torch.exp(torch.randn(N, 6, generator=g) * 0.3)))
    rots = torch.zeros(N, 4); rots[:, 0] = 1
    pc._rotation = P(rots, False)
    pc._opacity = P(torch.zeros(N, 1), False)
    with torch.no_grad():
        pc.mlp_opacity[2].bias += 0.3
        for mod in pc.feat_planes.modules():
            if isinstance(mod, torch.nn.BatchNorm1d):
                mod.weight.uniform_(0.5, 1.5)
                mod.bias.uniform_(-0.2, 0.2)
    pc.feat_planes.Q0 = 0.0
    pc.feat_planes._feat.activate_level = 2
    pc.train()
    return pc


def _leaves(pc):
    named = {"_anchor": pc._anchor, "_offset": pc._offset, "_anchor_feat": pc._anchor_feat, "_scaling": pc._scaling}
    for name in ("mlp_opacity", "mlp_cov", "mlp_color"):
        for k, v in getattr(pc, name).named_parameters():
            named[f"{name}.{k}"] = v
    for k, v in pc.feat_planes._feat.named_parameters():
        named[f"feat.{k}"] = v
    return named


def test_real_reference_model_renders_through_the_dropin():
    ref_gr, gm = _reference_modules()
    import splatco_b200.gaussian_renderer as our_gr
    from splatco_b200.synthetic import ring_cameras
    pc = _real_model(gm)
    feat = pc.feat_planes._feat
    assert len(feat.k0s) == 4 and len(feat.models) >= 3        # the quirk of scene/gaussian_model.py:112-118
    W, H = 320, 200
    cam = ring_cameras(3, W, H)[1].to("cuda")
    bg = torch.ones(3, device="cuda")
    pipe = SimpleNamespace(debug=False, compute_cov3D_python=False, convert_SHs_python=False)
    gt = torch.rand(3, H, W, generator=torch.Generator().manual_seed(5)).cuda()
    leaves = _leaves(pc)
    bn_keys = [k for k in feat.state_dict() if "running" in k or "num_batches" in k]

    def run(gr):
        sd0 = {k: v.clone() for k, v in feat.state_dict().items() if k in bn_keys}
        for p in leaves.values():
            p.grad = None
        vm = gr.prefilter_voxel(cam, pc, pipe, bg)
        pkg = gr.render(cam, pc, pipe, bg, visible_mask=vm, retain_grad=True)
        loss = (pkg["render"] - gt).abs().mean() + 0.01 * pkg["scaling"].prod(dim=1).mean()
        loss.backward()
        out = dict(vm=vm.cpu().numpy(), img=pkg["render"].detach().cpu().numpy(), mask=pkg["selection_mask"].cpu().numpy(),
                   radii=pkg["radii"].cpu().numpy(), nopac=pkg["neural_opacity"].detach().cpu().numpy(),
                   grads={k: (None if p.grad is None else p.grad.detach().cpu().numpy().copy()) for k, p in leaves.items()},
                   vsp=pkg["viewspace_points"].grad.detach().cpu().numpy().copy(),
                   bn={k: v.clone() for k, v in feat.state_dict().items() if k in bn_keys})
        feat.load_state_dict({**feat.state_dict(), **sd0})     # both runs start from the same running statistics
        return out

    a = run(ref_gr)         # option A: the reference's own decode on our rasterizer
    b = run(our_gr)         # option B: the whole hot path
    assert a["vm"].sum() > 1000 and np.array_equal(a["vm"], b["vm"])
    decided = np.abs(a["nopac"][:, 0]) > 1e-5
    assert np.array_equal(a["mask"][decided], b["mask"][decided]) and (a["mask"] != b["mask"]).sum() <= 2
    assert np.abs(a["nopac"] - b["nopac"]).max() < 2e-5
    same = np.array_equal(a["mask"], b["mask"])
    if same:
        assert (a["radii"] != b["radii"]).sum() <= max(2, int(2e-5 * a["radii"].size))
    err = np.abs(a["img"] - b["img"])
    # (both sides blend with the same kernels; the decodes agree to ~1e-6, so does the image except where a Gaussian
    #  crosses one of the rasterizer's integer decisions)
    assert np.quantile(err, 0.9999) <= 1e-4 and err.max() <= 1e-2, (float(np.quantile(err, 0.9999)), float(err.max()))
    if same:
        checked = 0
        for k, ga in a["grads"].items():
            gb = b["grads"][k]
            assert (ga is None) == (gb is None), k
            if ga is None or float(np.abs(ga).max()) == 0.0:
                continue
            e = full_path_grad_errors(gb, ga)
            assert e["l2"] < (3e-3 if ".TA." in k else 1e-3) and e["amax"] < 5e-3, (k, e)
            checked += 1
        assert checked >= 30
        e = full_path_grad_errors(b["vsp"][:, :2], a["vsp"][:, :2])
        assert e["l2"] < 1e-3 and e["amax"] < 5e-3, e
    for k in bn_keys:
        assert torch.allclose(a["bn"][k].float(), b["bn"][k].float(), rtol=1e-4, atol=1e-6), k
