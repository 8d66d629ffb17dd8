"""Drop-in for the reference's `gaussian_renderer` package (gaussian_renderer/__init__.py:1-244).

Same public names, signatures, return dicts and error behaviour:
    generate_neural_gaussians(viewpoint_camera, pc, visible_mask=None, is_training=False)   (:18-116)
    render(viewpoint_camera, pc, pipe, bg_color, scaling_modifier=1.0, visible_mask=None, retain_grad=False)  (:118-188)
    prefilter_voxel(viewpoint_camera, pc, pipe, bg_color, scaling_modifier=1.0, override_color=None)          (:191-244)
plus the `GaussianModel` re-export render.py relies on (:16, render.py:34) when the reference's
`scene` package is importable.  Everything below these functions runs in libsplatco_b200.so.
"""
from __future__ import annotations

import math
import weakref

import torch

from ..decode import generate_neural_gaussians
from ..diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer, visible_mask_compact

try:  # re-export, as the reference module does
    from scene.gaussian_model import GaussianModel  # type: ignore  # noqa: F401
except Exception:  # the reference tree is not on sys.path (tests, bench)
    GaussianModel = None

try:
    from . import network_gui  # type: ignore  # noqa: F401   (train.py:18 imports it from here)
except Exception:
    network_gui = None


def _settings(viewpoint_camera, pipe, bg_color, scaling_modifier):
    tanfovx = math.tan(viewpoint_camera.FoVx * 0.5)
    tanfovy = math.tan(viewpoint_camera.FoVy * 0.5)
    return GaussianRasterizationSettings(
        image_height=int(viewpoint_camera.image_height),
        image_width=int(viewpoint_camera.image_width),
        tanfovx=tanfovx,
        tanfovy=tanfovy,
        bg=bg_color,
        scale_modifier=scaling_modifier,
        viewmatrix=viewpoint_camera.world_view_transform,
        projmatrix=viewpoint_camera.full_proj_transform,
        sh_degree=1,
        campos=viewpoint_camera.camera_center,
        prefiltered=False,
        debug=pipe.debug,
        antialiasing=bool(getattr(pipe, "antialiasing", False)),   # upstream PipelineParams' flag; off when absent
    )


# prefilter_voxel and render() both read pc.get_scaling (= 1.0 * exp(pc._scaling), two launches plus two more in the
# backward); when render() follows the prefilter of the same model state it reuses that tensor -- same values, same
# autograd node -- instead of evaluating the accessor a second time.
_scaling_stash = {"pc": None, "src": None, "version": -1, "grad": None, "value": None}


def _get_scaling(pc, remember):
    src = getattr(pc, "_scaling", None)
    st = _scaling_stash
    if (not remember and src is not None and st["value"] is not None and st["pc"] is not None and st["pc"]() is pc
            and st["src"] is src and st["version"] == src._version and st["grad"] == torch.is_grad_enabled()):
        value = st["value"]
        st["value"] = None                      # single use: the next view's prefilter computes a fresh one
        return value
    value = pc.get_scaling
    if remember and src is not None:
        st.update(pc=weakref.ref(pc), src=src, version=src._version, grad=torch.is_grad_enabled(), value=value)
    return value


# pc.get_rotation = normalize(pc._rotation) is four launches per prefilter call on a tensor nothing in the render path
# ever updates (anchor rotations receive no gradient); the normalised copy is kept for as long as the same tensor object
# has the same version counter (any in-place update, e.g. an optimizer step, bumps it; densification replaces the object).
_rotation_stash = {"src": None, "version": -1, "fn": None, "value": None}


def _get_rotation(pc):
    src = getattr(pc, "_rotation", None)
    if src is None or not isinstance(src, torch.Tensor):
        return pc.get_rotation              # (the prefilter is not differentiable: a detached copy serves it in any grad mode)
    st = _rotation_stash
    fn = getattr(pc, "rotation_activation", None)
    held = st["src"]() if st["src"] is not None else None
    if held is src and st["version"] == src._version and st["fn"] is fn and st["value"] is not None:
        return st["value"]
    value = pc.get_rotation
    st.update(src=weakref.ref(src), version=src._version, fn=fn, value=value.detach())
    return st["value"]


def render(viewpoint_camera, pc, pipe, bg_color: torch.Tensor, scaling_modifier=1.0, visible_mask=None,
           retain_grad=False, *, depth_alpha=False):
    """Render the scene.  Background tensor (bg_color) must be on GPU!

    depth_alpha=True also returns, under "depth" and "alpha", the differentiable maps [1,H,W]
    depth = sum_i z_i alpha_i T_i (accumulated view-space depth, background 0) and alpha = 1 - T_final, from the
    same front-to-back walk as the image.  The expected depth is depth / alpha where alpha > 0; the caller forms it."""
    is_training = pc.get_color_mlp.training
    settings = _settings(viewpoint_camera, pipe, bg_color, scaling_modifier)
    if is_training:
        xyz, color, opacity, scaling, rot, neural_opacity, mask = generate_neural_gaussians(
            viewpoint_camera, pc, visible_mask, is_training=is_training, _raster_settings=settings,
            _scaling=_get_scaling(pc, remember=False), _depth_alpha=depth_alpha)
    else:
        xyz, color, opacity, scaling, rot = generate_neural_gaussians(
            viewpoint_camera, pc, visible_mask, is_training=is_training, _raster_settings=settings,
            _scaling=_get_scaling(pc, remember=False), _depth_alpha=depth_alpha)

    # zero tensor whose .grad receives the 2D (screen-space) mean gradients (reference :133-138)
    # (the reference adds `+ 0` to make it a non-leaf and calls retain_grad(); a leaf holds the same .grad after backward
    # without the extra add kernel in the forward and the gradient copy in the backward)
    screenspace_points = torch.zeros_like(xyz, dtype=pc.get_anchor.dtype, requires_grad=True, device="cuda")

    rasterizer = GaussianRasterizer(raster_settings=settings)
    if depth_alpha:
        rendered_image, radii, depth, alpha = rasterizer(
            means3D=xyz, means2D=screenspace_points, shs=None, colors_precomp=color, opacities=opacity, scales=scaling,
            rotations=rot, cov3D_precomp=None, depth_alpha=True)
    else:
        rendered_image, radii = rasterizer(
            means3D=xyz,
            means2D=screenspace_points,
            shs=None,
            colors_precomp=color,
            opacities=opacity,
            scales=scaling,
            rotations=rot,
            cov3D_precomp=None)

    out = {"render": rendered_image,
           "viewspace_points": screenspace_points,
           "visibility_filter": radii > 0,
           "radii": radii}
    if depth_alpha:
        out.update({"depth": depth, "alpha": alpha})
    if is_training:
        out.update({"selection_mask": mask, "neural_opacity": neural_opacity, "scaling": scaling})
    return out


def prefilter_voxel(viewpoint_camera, pc, pipe, bg_color: torch.Tensor, scaling_modifier=1.0, override_color=None):
    """Anchor-level frustum/size prefilter: bool[N] (reference :191-244)."""
    rasterizer = GaussianRasterizer(raster_settings=_settings(viewpoint_camera, pipe, bg_color, scaling_modifier))
    means3D = pc.get_anchor
    scales = None
    rotations = None
    cov3D_precomp = None
    if pipe.compute_cov3D_python:
        # the reference's branch is broken here (scales stays None and is then sliced, :233-240)
        cov3D_precomp = pc.get_covariance(scaling_modifier)
    else:
        scales = _get_scaling(pc, remember=True)
        rotations = _get_rotation(pc)
    if cov3D_precomp is not None:
        radii_pure = rasterizer.visible_filter(means3D=means3D, scales=scales, rotations=rotations,
                                               cov3D_precomp=cov3D_precomp)          # raises (unsupported, see above)
        return radii_pure > 0
    # radii_pure > 0, plus the index list of the visible anchors kept aside for the render() call that follows
    return visible_mask_compact(means3D, scales[:, :3], rotations, rasterizer.raster_settings)
