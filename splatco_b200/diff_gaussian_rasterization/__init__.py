"""Drop-in for the `diff_gaussian_rasterization` package SplatCo imports
(reference gaussian_renderer/__init__.py:15; call sites :145-171 and :208-242).

Same public names and call signatures as the package in the reference's submodules.zip
(Inria diff-gaussian-rasterization with the Scaffold-GS `visible_filter` addition, SURVEY.md
Appendix A.1): `GaussianRasterizationSettings`, `GaussianRasterizer`, `rasterize_gaussians`.
Underneath, everything runs in libsplatco_b200.so (hand-written sm_100a CUDA, C ABI in
include/splatco_b200.h).  No CPU / PyTorch fallback exists: without the library, calls raise.

Supported argument combinations are the ones the reference uses: `colors_precomp` (not `shs`) and
`scales` + `rotations` (not `cov3D_precomp`).  The other upstream combinations raise
NotImplementedError instead of silently doing something else.
"""
from __future__ import annotations

import threading
from typing import NamedTuple

import torch
import torch.nn as nn

from .. import _lib
from ..profiling import stage
from .._lib import check, ptr


class GaussianRasterizationSettings(NamedTuple):
    # field order = the keyword order used at gaussian_renderer/__init__.py:145-158
    image_height: int
    image_width: int
    tanfovx: float
    tanfovy: float
    bg: torch.Tensor
    scale_modifier: float
    viewmatrix: torch.Tensor
    projmatrix: torch.Tensor
    sh_degree: int
    campos: torch.Tensor
    prefiltered: bool
    debug: bool
    # screen-space mip filter with opacity compensation (upstream's `antialiasing`): each Gaussian's opacity is scaled
    # by rho = sqrt(max(2.5e-5, det(cov2D) / det(cov2D + 0.3 I))), so sub-pixel Gaussians keep their integrated weight
    antialiasing: bool = False


_tls = threading.local()


def _pinned_counter(device: torch.device, slot: int = 0) -> torch.Tensor:
    """One pinned int32 per (thread, device, slot) for the num_rendered read-back."""
    cache = getattr(_tls, "counters", None)
    if cache is None:
        cache = _tls.counters = {}
    key = (device.index if device.index is not None else torch.cuda.current_device(), slot)
    buf = cache.get(key)
    if buf is None:
        buf = cache[key] = torch.zeros(1, dtype=torch.int32).pin_memory()
    return buf


def _stream_ptr(device) -> int:
    return _lib.raw_stream(device)


def _f32c(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


def _rows_f32(t: torch.Tensor, cols: int):
    """Return (tensor, row_stride_in_floats) for a [N,cols] fp32 tensor whose rows may be strided
    (the reference passes get_scaling[:, :3], a view of an [N,6] tensor)."""
    if t.dtype != torch.float32:
        t = t.float()
    if t.dim() == 2 and t.shape[1] == cols and t.stride(1) == 1 and t.stride(0) >= cols and t.shape[0] > 0:
        return t, int(t.stride(0))
    return t.contiguous(), cols


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("splatco_b200 rasterizer needs CUDA tensors (no CPU fallback)")


def _debug_sync(settings, what):
    if settings.debug:
        torch.cuda.synchronize()


class RasterState:
    """What forward leaves behind for backward and for the stage-wise parity tests."""
    __slots__ = ("P", "PL", "R", "RL", "H", "W", "geom", "binning", "image", "radii", "radii_full", "depth_alpha",
                 "depth", "alpha")
    # P / R: Gaussians and instances of this view; PL / RL: the row counts the geometry / binning
    # workspaces were laid out for (>= P, R when the forward was queued before the counts were known)
    # depth_alpha: the forward also produced the depth and alpha maps [1,H,W] (`depth`, `alpha`)


class _Speculated:
    """preprocess_fwd launched by the decode on its own outputs before their row count M was known on
    the host (splatco_preprocess_fwd_counted), so that M and R come back in ONE sync."""
    __slots__ = ("tensors", "versions", "settings", "M", "PL", "R", "RL", "geom", "radii_full", "counter", "binning",
                 "image", "color", "event", "depth_alpha", "depth", "alpha")


_spec_slot = threading.local()


def preprocess_speculative(xyz_b, color_b, opacity_b, scaling_b, rot_b, count_ptr, settings, depth_alpha=False):
    """Called by the decode forward with its VK-row output buffers (row count still on the device at
    `count_ptr`).  Launches the counted preprocess and returns the pending record; the caller syncs,
    then `publish_speculated` makes it available to the next rasterizer forward on these tensors.
    `depth_alpha`: the rasterizer call will ask for the depth and alpha maps, so the queued blend produces them."""
    L = _lib.lib()
    dev = xyz_b.device
    H, W = int(settings.image_height), int(settings.image_width)
    PL = int(xyz_b.shape[0])
    sp = _Speculated()
    sp.settings, sp.PL, sp.depth_alpha = settings, PL, bool(depth_alpha)
    sp.radii_full = _lib.empty_rows(PL, None, torch.int32, dev)
    sp.geom = _lib.empty_u8(L.splatco_geom_bytes(PL), dev)
    sp.counter = _pinned_counter(dev, 1)
    view, proj = _f32c(settings.viewmatrix), _f32c(settings.projmatrix)
    name = "splatco_preprocess_fwd_aa_counted" if settings.antialiasing else "splatco_preprocess_fwd_counted"
    with stage("preprocess_fwd"):
        check(getattr(L, name)(PL, count_ptr, ptr(xyz_b), ptr(scaling_b), 3, ptr(rot_b), ptr(opacity_b), ptr(color_b),
                               float(settings.scale_modifier), ptr(view), ptr(proj), float(settings.tanfovx),
                               float(settings.tanfovy), H, W, ptr(sp.radii_full), ptr(sp.geom), sp.counter.data_ptr(),
                               _stream_ptr(dev)), name)
    # M and R are complete once this event has passed; the caller waits for IT, not for the stream
    sp.event = torch.cuda.Event()
    sp.event.record(torch.cuda.current_stream(dev))
    # binning + blend are queued too, on buffers sized from the last view of this resolution: when the
    # host learns M and R the GPU is already working on them instead of idling through the host-side
    # bookkeeping that follows the sync.  A wrong guess (R larger than the buffers) is detected after the
    # sync and the two stages are simply re-run (publish_speculated).
    sp.binning = sp.image = sp.color = sp.depth = sp.alpha = None
    sp.RL = 0
    guess = _r_guess.get((H, W))
    if guess:
        RL = int(guess * 1.25) + 4096
        # only the tile-segmented binning path clamps to a capacity; its radix fallback (sparse views: few instances per
        # row of the V*K-row buffers) needs the exact count, so nothing is queued ahead of the sync then
        if L.splatco_binning_accepts_capacity(PL, RL, H, W):
            sp.RL = RL
            _queue_binning_blend(sp, dev, H, W)
    return sp


_r_guess = {}


def _queue_binning_blend(sp, dev, H, W):
    L = _lib.lib()
    settings = sp.settings
    stream = _stream_ptr(dev)
    sp.binning = _lib.empty_u8(L.splatco_binning_bytes(sp.RL), dev)
    sp.image = torch.empty(L.splatco_image_bytes(H, W), dtype=torch.uint8, device=dev)
    sp.color = torch.empty((3, H, W), dtype=torch.float32, device=dev)
    with stage("binning"):
        check(L.splatco_binning(sp.PL, sp.RL, H, W, ptr(sp.radii_full), ptr(sp.geom), ptr(sp.binning), ptr(sp.image),
                                stream), "splatco_binning")
    with stage("blend_fwd"):
        if sp.depth_alpha:
            sp.depth = torch.empty((1, H, W), dtype=torch.float32, device=dev)
            sp.alpha = torch.empty((1, H, W), dtype=torch.float32, device=dev)
            check(L.splatco_blend_fwd_depth_alpha(sp.RL, H, W, ptr(_f32c(settings.bg)), ptr(sp.geom), ptr(sp.binning),
                                                  ptr(sp.image), ptr(sp.color), ptr(sp.depth), ptr(sp.alpha), stream),
                  "splatco_blend_fwd_depth_alpha")
        else:
            check(L.splatco_blend_fwd(sp.RL, H, W, ptr(_f32c(settings.bg)), ptr(sp.geom), ptr(sp.binning), ptr(sp.image),
                                      ptr(sp.color), stream), "splatco_blend_fwd")


def publish_speculated(sp, M, outs):
    """After the sync: `outs` = the M-row tensors (xyz, color, opacity, scaling, rot) the decode returns."""
    sp.M, sp.R = M, int(sp.counter[0])
    H, W = int(sp.settings.image_height), int(sp.settings.image_width)
    _r_guess[(H, W)] = max(sp.R, 1)
    if sp.binning is None or sp.R > sp.RL:
        if M > 0 and sp.R > 0:
            sp.RL = sp.R
            _queue_binning_blend(sp, outs[0].device, H, W)
        else:
            sp.binning = None
    sp.tensors = tuple(outs)
    sp.versions = tuple(t._version for t in outs)
    _spec_slot.sp = sp


def _take_speculated(means3D, colors, opacities, scales, rotations, settings, depth_alpha=False):
    sp = getattr(_spec_slot, "sp", None)
    if sp is None:
        return None
    _spec_slot.sp = None
    ins = (means3D, colors, opacities, scales, rotations)
    if sp.settings is not settings or sp.M != int(means3D.shape[0]) or sp.depth_alpha != depth_alpha:
        return None
    for t, u, v in zip(ins, sp.tensors, sp.versions):
        # same memory, same shape, not written to since the decode produced it
        if t.data_ptr() != u.data_ptr() or t.shape != u.shape or t._version != v or not t.is_contiguous():
            return None
    return sp


def rasterize_forward_state(means3D, colors, opacities, scales, rotations, settings, depth_alpha=False) -> tuple:
    """Forward pass; returns (color [3,H,W], radii int32 [P], RasterState).  With depth_alpha the state also
    holds the depth and alpha maps [1,H,W] (`st.depth`, `st.alpha`)."""
    depth_alpha = bool(depth_alpha)
    L = _lib.lib()
    _require_cuda(means3D, colors, opacities, scales, rotations, settings.bg, settings.viewmatrix,
                  settings.projmatrix)
    dev = means3D.device
    H, W = int(settings.image_height), int(settings.image_width)
    P = int(means3D.shape[0])
    bg = _f32c(settings.bg)
    st = RasterState()
    st.P, st.PL, st.H, st.W = P, P, H, W
    st.depth_alpha, st.depth, st.alpha = depth_alpha, None, None
    sp = _take_speculated(means3D, colors, opacities, scales, rotations, settings, depth_alpha)
    if P == 0:
        st.R = st.RL = 0
        st.geom = st.binning = None
        st.image = torch.empty(L.splatco_image_bytes(H, W), dtype=torch.uint8, device=dev)
        st.radii = st.radii_full = torch.empty(0, dtype=torch.int32, device=dev)
        color = bg.reshape(3, 1, 1).expand(3, H, W).contiguous()
        if depth_alpha:
            st.depth = torch.zeros((1, H, W), dtype=torch.float32, device=dev)
            st.alpha = torch.zeros((1, H, W), dtype=torch.float32, device=dev)
        return color, st.radii, st
    stream = _stream_ptr(dev)
    with _lib.on_device(dev):
        if sp is not None and sp.binning is not None:
            # the whole forward already ran (queued inside the decode forward)
            st.PL, st.R, st.RL = sp.PL, sp.R, sp.RL
            st.geom, st.binning, st.image, st.radii_full = sp.geom, sp.binning, sp.image, sp.radii_full
            st.radii = sp.radii_full[:P]
            st.depth, st.alpha = sp.depth, sp.alpha
            _debug_sync(settings, "forward")
            return sp.color, st.radii, st
        if sp is not None:
            radii_full, geom, R, st.PL = sp.radii_full, sp.geom, sp.R, sp.PL
            radii = radii_full[:P]
        else:
            means3D = _f32c(means3D)
            colors = _f32c(colors)
            opacities = _f32c(opacities)
            rotations = _f32c(rotations)
            scales, sstride = _rows_f32(scales, 3)
            view = _f32c(settings.viewmatrix)
            proj = _f32c(settings.projmatrix)
            radii = radii_full = _lib.empty_rows(P, None, torch.int32, dev)
            geom = _lib.empty_u8(L.splatco_geom_bytes(P), dev)
            counter = _pinned_counter(dev)
            name = "splatco_preprocess_fwd_aa" if settings.antialiasing else "splatco_preprocess_fwd"
            with stage("preprocess_fwd"):
                check(getattr(L, name)(P, ptr(means3D), ptr(scales), sstride, ptr(rotations), ptr(opacities), ptr(colors),
                                       float(settings.scale_modifier), ptr(view), ptr(proj), float(settings.tanfovx),
                                       float(settings.tanfovy), H, W, ptr(radii), ptr(geom), counter.data_ptr(), stream),
                      name)
            # the one device->host sync of the forward (the reference has the same one, SURVEY §3.1)
            torch.cuda.current_stream(dev).synchronize()
            R = int(counter[0])
        _debug_sync(settings, "preprocess")
        binning = _lib.empty_u8(L.splatco_binning_bytes(R), dev)
        image = torch.empty(L.splatco_image_bytes(H, W), dtype=torch.uint8, device=dev)
        with stage("binning"):
            check(L.splatco_binning(st.PL, R, H, W, ptr(radii_full), ptr(geom), ptr(binning), ptr(image), stream),
                  "splatco_binning")
        _debug_sync(settings, "binning")
        color = torch.empty((3, H, W), dtype=torch.float32, device=dev)
        with stage("blend_fwd"):
            if depth_alpha:
                st.depth = torch.empty((1, H, W), dtype=torch.float32, device=dev)
                st.alpha = torch.empty((1, H, W), dtype=torch.float32, device=dev)
                check(L.splatco_blend_fwd_depth_alpha(R, H, W, ptr(bg), ptr(geom), ptr(binning), ptr(image), ptr(color),
                                                      ptr(st.depth), ptr(st.alpha), stream), "splatco_blend_fwd_depth_alpha")
            else:
                check(L.splatco_blend_fwd(R, H, W, ptr(bg), ptr(geom), ptr(binning), ptr(image), ptr(color), stream),
                      "splatco_blend_fwd")
        _debug_sync(settings, "blend_fwd")
    st.R, st.RL, st.geom, st.binning, st.image, st.radii, st.radii_full = R, R, geom, binning, image, radii, radii_full
    return color, radii, st


def rasterize_backward_state(st: RasterState, grad_color, means3D, scales, rotations, settings, grad_depth=None,
                             grad_alpha=None, camera=False, opacities=None):
    """Backward pass; returns dict of gradients (all fp32, same row count as the inputs).
    grad_depth / grad_alpha ([1,H,W] or None) need a depth_alpha forward.  With both None this is the colour-only
    backward (splatco_blend_bwd + splatco_preprocess_bwd); with either given, splatco_blend_bwd_depth_alpha also
    yields dL/dz_view per Gaussian (returned as "depth"), which splatco_preprocess_bwd_depth adds to dL/dmeans3D, and
    grad_color may be None.  Absent upstream gradients are passed as NULL (zero).
    camera=True: splatco_preprocess_bwd_camera replaces the preprocess backward (same per-Gaussian outputs) and the dict
    also holds "viewmatrix" and "projmatrix", fp32 [4,4]: the gradients of the contiguous fp32 copies the kernels read.
    settings.antialiasing: splatco_preprocess_bwd_aa serves all of the above; it needs the forward's `opacities` and turns
    the blend's gradient with respect to the record's compensated opacity into dL/dopacities."""
    da = grad_depth is not None or grad_alpha is not None
    aa = bool(settings.antialiasing)
    if aa and opacities is None:
        raise RuntimeError("an antialiased backward needs the forward's opacities")
    if da and not st.depth_alpha:
        raise RuntimeError("depth / alpha gradients need a forward with depth_alpha=True")
    L = _lib.lib()
    dev = means3D.device
    P, R, H, W = st.P, st.RL, st.H, st.W          # RL: the binning workspace's layout size
    # two allocations, two split calls: [mean2D 3 | conic 3 | opacity 1 | colour 3 (| depth 1)] is zero-filled for the
    # blend's REDs, [means3D 3 | scales 3 | rotations 4] is overwritten by preprocess_bwd (rotations stay 16-byte aligned)
    nz = 11 if da else 10
    parts = torch.zeros(_lib.bucket(nz * P), dtype=torch.float32, device=dev)[:nz * P].split_with_sizes(
        [3 * P, 3 * P, P, 3 * P] + ([P] if da else []))
    g_mean2D, g_conic, g_opac, g_color = parts[0].view(P, 3), parts[1].view(P, 3), parts[2].view(P, 1), parts[3].view(P, 3)
    g_depth = parts[4] if da else None
    e, f, g_ = _lib.empty_rows(12 * P, None, torch.float32, dev).split_with_sizes([4 * P, 4 * P, 4 * P])
    g_rots, g_means3D, g_scales = e.view(P, 4), f[:3 * P].view(P, 3), g_[:3 * P].view(P, 3)
    out = dict(means3D=g_means3D, means2D=g_mean2D, colors=g_color, opacities=g_opac, scales=g_scales,
               rotations=g_rots, conic=g_conic)
    if da:
        out["depth"] = g_depth
    if camera:
        g_cam = torch.zeros(32, dtype=torch.float32, device=dev) if P == 0 else torch.empty(32, dtype=torch.float32, device=dev)
        out["viewmatrix"], out["projmatrix"] = g_cam[:16].view(4, 4), g_cam[16:].view(4, 4)
    if P == 0:
        return out
    means3D = _f32c(means3D)
    rotations = _f32c(rotations)
    scales, sstride = _rows_f32(scales, 3)
    bg = _f32c(settings.bg)
    view = _f32c(settings.viewmatrix)
    proj = _f32c(settings.projmatrix)
    stream = _stream_ptr(dev)
    ws = (ptr(bg), ptr(st.geom), ptr(st.binning), ptr(st.image))
    blend_out = (ptr(g_mean2D), ptr(g_conic), ptr(g_opac), ptr(g_color))
    pre_args = (P, ptr(means3D), ptr(scales), sstride, ptr(rotations), float(settings.scale_modifier), ptr(view),
                ptr(proj), float(settings.tanfovx), float(settings.tanfovy), H, W, ptr(st.radii), ptr(g_mean2D),
                ptr(g_conic), ptr(g_means3D), ptr(g_scales), ptr(g_rots))
    with _lib.on_device(dev):
        with stage("blend_bwd"):
            if da:
                maps = [None if t is None else _f32c(t) for t in (grad_color, grad_depth, grad_alpha)]
                check(L.splatco_blend_bwd_depth_alpha(P, R, H, W, *ws, *[ptr(t) for t in maps], *blend_out, ptr(g_depth),
                                                      stream), "splatco_blend_bwd_depth_alpha")
            else:
                grad_color = _f32c(grad_color)
                check(L.splatco_blend_bwd(P, R, H, W, *ws, ptr(grad_color), *blend_out, stream), "splatco_blend_bwd")
        _debug_sync(settings, "blend_bwd")
        with stage("preprocess_bwd"):
            if aa:
                opacities = _f32c(opacities)
                cam_ws = _lib.empty_u8(L.splatco_camera_grad_ws_bytes(P), dev) if camera else None
                cam = (ptr(cam_ws), ptr(out["viewmatrix"]), ptr(out["projmatrix"])) if camera else (None, None, None)
                check(L.splatco_preprocess_bwd_aa(*pre_args, ptr(opacities), ptr(g_opac), ptr(g_depth), *cam, stream),
                      "splatco_preprocess_bwd_aa")
            elif camera:
                cam_ws = _lib.empty_u8(L.splatco_camera_grad_ws_bytes(P), dev)
                check(L.splatco_preprocess_bwd_camera(*pre_args, ptr(g_depth), ptr(cam_ws), ptr(out["viewmatrix"]),
                                                      ptr(out["projmatrix"]), stream), "splatco_preprocess_bwd_camera")
            elif da:
                check(L.splatco_preprocess_bwd_depth(*pre_args, ptr(g_depth), stream), "splatco_preprocess_bwd_depth")
            else:
                check(L.splatco_preprocess_bwd(*pre_args, stream), "splatco_preprocess_bwd")
        _debug_sync(settings, "preprocess_bwd")
    return out


def _check_supported(sh, cov3Ds_precomp):
    if sh is not None and sh.numel() > 0:
        raise NotImplementedError("splatco_b200: SH colours are not on SplatCo's path (it passes colors_precomp)")
    if cov3Ds_precomp is not None and cov3Ds_precomp.numel() > 0:
        raise NotImplementedError("splatco_b200: cov3D_precomp is not on SplatCo's path (it passes scales+rotations)")


def _save_for_backward(ctx, st, raster_settings, radii, means3D, scales, rotations, opacities):
    ctx.raster_settings = raster_settings
    ctx.state = st
    # the antialiased backward also reads the opacities (dL/dopacities = rho dL/d(record opacity))
    ctx.save_for_backward(means3D, scales, rotations, *((opacities,) if raster_settings.antialiasing else ()))
    ctx.mark_non_differentiable(radii)
    ctx.set_materialize_grads(False)          # no zero-filled gradient tensor for `radii` (or an unused map)


def _saved(ctx):
    """(means3D, scales, rotations, opacities or None)"""
    t = ctx.saved_tensors
    return (*t, None) if len(t) == 3 else t


class _RasterizeGaussians(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                raster_settings):
        _check_supported(sh, cov3Ds_precomp)
        color, radii, st = rasterize_forward_state(means3D, colors_precomp, opacities, scales, rotations,
                                                   raster_settings)
        _save_for_backward(ctx, st, raster_settings, radii, means3D, scales, rotations, opacities)
        return color, radii

    @staticmethod
    def backward(ctx, grad_out_color, _grad_radii):
        if grad_out_color is None:
            return (None,) * 9
        means3D, scales, rotations, opacities = _saved(ctx)
        g = rasterize_backward_state(ctx.state, grad_out_color, means3D, scales, rotations, ctx.raster_settings,
                                     opacities=opacities)
        # (means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, settings)
        return (g["means3D"], g["means2D"], None, g["colors"], g["opacities"], g["scales"], g["rotations"],
                None, None)


def rasterize_gaussians(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                        raster_settings):
    return _RasterizeGaussians.apply(means3D, means2D, sh, colors_precomp, opacities, scales, rotations,
                                     cov3Ds_precomp, raster_settings)


class _RasterizeGaussiansDepthAlpha(torch.autograd.Function):
    """_RasterizeGaussians that also returns the depth and alpha maps [1,H,W] (see GaussianRasterizer.forward)."""

    @staticmethod
    def forward(ctx, means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                raster_settings):
        _check_supported(sh, cov3Ds_precomp)
        color, radii, st = rasterize_forward_state(means3D, colors_precomp, opacities, scales, rotations,
                                                   raster_settings, depth_alpha=True)
        depth, alpha = st.depth, st.alpha
        st.depth = st.alpha = None                  # the state outlives the outputs in ctx; it does not need them
        _save_for_backward(ctx, st, raster_settings, radii, means3D, scales, rotations, opacities)
        return color, radii, depth, alpha

    @staticmethod
    def backward(ctx, grad_out_color, _grad_radii, grad_depth, grad_alpha):
        if grad_out_color is None and grad_depth is None and grad_alpha is None:
            return (None,) * 9
        means3D, scales, rotations, opacities = _saved(ctx)
        # both map gradients None: exactly the colour-only backward (splatco_blend_bwd + splatco_preprocess_bwd)
        g = rasterize_backward_state(ctx.state, grad_out_color, means3D, scales, rotations, ctx.raster_settings,
                                     grad_depth=grad_depth, grad_alpha=grad_alpha, opacities=opacities)
        return (g["means3D"], g["means2D"], None, g["colors"], g["opacities"], g["scales"], g["rotations"],
                None, None)


class _RasterizeGaussiansCamera(torch.autograd.Function):
    """_RasterizeGaussians (depth_alpha False) or _RasterizeGaussiansDepthAlpha (True) with the view and projection
    matrices of the settings as differentiable inputs: GaussianRasterizer.forward routes here when either of them
    requires grad.  Their gradients are taken with respect to the [4,4] elements, whatever dtype and strides the
    tensors have; `campos` gets none (there are no SH colours)."""

    @staticmethod
    def forward(ctx, means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                raster_settings, viewmatrix, projmatrix, depth_alpha):
        _check_supported(sh, cov3Ds_precomp)
        color, radii, st = rasterize_forward_state(means3D, colors_precomp, opacities, scales, rotations,
                                                   raster_settings, depth_alpha=depth_alpha)
        _save_for_backward(ctx, st, raster_settings, radii, means3D, scales, rotations, opacities)
        ctx.cam_dtypes = (viewmatrix.dtype, projmatrix.dtype)
        if not depth_alpha:
            return color, radii
        depth, alpha = st.depth, st.alpha
        st.depth = st.alpha = None
        return color, radii, depth, alpha

    @staticmethod
    def backward(ctx, grad_out_color, _grad_radii, grad_depth=None, grad_alpha=None):
        if grad_out_color is None and grad_depth is None and grad_alpha is None:
            return (None,) * 12
        means3D, scales, rotations, opacities = _saved(ctx)
        g = rasterize_backward_state(ctx.state, grad_out_color, means3D, scales, rotations, ctx.raster_settings,
                                     grad_depth=grad_depth, grad_alpha=grad_alpha, camera=True, opacities=opacities)
        g_view = g["viewmatrix"].to(ctx.cam_dtypes[0]) if ctx.needs_input_grad[9] else None
        g_proj = g["projmatrix"].to(ctx.cam_dtypes[1]) if ctx.needs_input_grad[10] else None
        return (g["means3D"], g["means2D"], None, g["colors"], g["opacities"], g["scales"], g["rotations"],
                None, None, g_view, g_proj, None)


class GaussianRasterizer(nn.Module):
    def __init__(self, raster_settings: GaussianRasterizationSettings):
        super().__init__()
        self.raster_settings = raster_settings

    def markVisible(self, positions):
        raise NotImplementedError("splatco_b200: markVisible is not on SplatCo's path (use visible_filter)")

    def forward(self, means3D, means2D, opacities, shs=None, colors_precomp=None, scales=None, rotations=None,
                cov3D_precomp=None, *, depth_alpha=False):
        """(color [3,H,W], radii [P]); with depth_alpha=True (color, radii, depth [1,H,W], alpha [1,H,W]):
        depth = sum_i z_i alpha_i T_i, the accumulated view-space depth with background 0, and alpha = 1 - T_final,
        both from the walk that forms the colour and both differentiable.  The expected (normalised) depth is
        depth / alpha where alpha > 0; the caller forms it.
        When the settings' viewmatrix or projmatrix requires grad (and grad mode is on), they receive gradients too."""
        raster_settings = self.raster_settings
        if (shs is None and colors_precomp is None) or (shs is not None and colors_precomp is not None):
            raise Exception('Please provide excatly one of either SHs or precomputed colors!')
        if ((scales is None or rotations is None) and cov3D_precomp is None) or \
                ((scales is not None or rotations is not None) and cov3D_precomp is not None):
            raise Exception('Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!')
        if torch.is_grad_enabled() and (raster_settings.viewmatrix.requires_grad or
                                        raster_settings.projmatrix.requires_grad):
            return _RasterizeGaussiansCamera.apply(means3D, means2D, shs, colors_precomp, opacities, scales, rotations,
                                                   cov3D_precomp, raster_settings, raster_settings.viewmatrix,
                                                   raster_settings.projmatrix, bool(depth_alpha))
        if depth_alpha:
            return _RasterizeGaussiansDepthAlpha.apply(means3D, means2D, shs, colors_precomp, opacities, scales,
                                                       rotations, cov3D_precomp, raster_settings)
        return rasterize_gaussians(means3D, means2D, shs, colors_precomp, opacities, scales, rotations,
                                   cov3D_precomp, raster_settings)

    def visible_filter(self, means3D, scales=None, rotations=None, cov3D_precomp=None):
        """Per-anchor radii (int32 [N]); radii > 0 <=> the anchor's Gaussian touches the view
        (gaussian_renderer/__init__.py:239-244)."""
        rs = self.raster_settings
        if cov3D_precomp is not None and (not torch.is_tensor(cov3D_precomp) or cov3D_precomp.numel() > 0):
            raise NotImplementedError("splatco_b200: visible_filter with cov3D_precomp is not supported")
        if scales is None or rotations is None:
            raise Exception('Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!')
        with torch.no_grad():
            L = _lib.lib()
            _require_cuda(means3D, scales, rotations, rs.viewmatrix, rs.projmatrix)
            dev = means3D.device
            N = int(means3D.shape[0])
            radii = torch.empty(N, dtype=torch.int32, device=dev)
            if N == 0:
                return radii
            means3D = _f32c(means3D.detach())
            rotations = _f32c(rotations.detach())
            scales, sstride = _rows_f32(scales.detach(), 3)
            view, proj = _f32c(rs.viewmatrix), _f32c(rs.projmatrix)
            with _lib.on_device(dev), stage("visible_filter"):
                check(L.splatco_visible_filter(N, ptr(means3D), ptr(scales), sstride, ptr(rotations),
                                               float(rs.scale_modifier), ptr(view), ptr(proj), float(rs.tanfovx),
                                               float(rs.tanfovy), int(rs.image_height), int(rs.image_width),
                                               ptr(radii), _stream_ptr(dev)), "splatco_visible_filter")
            _debug_sync(rs, "visible_filter")
            return radii


# ---- prefilter with the index list render() needs next -------------------------------------------------------
class _Compaction:
    __slots__ = ("mask", "version", "idx", "counter", "event", "ws", "count_ptr")


def visible_mask_compact(means3D, scales, rotations, raster_settings):
    """bool[N] mask of the anchors whose Gaussian touches the view (radii > 0) -- what prefilter_voxel returns --
    computed together with the ascending index list of the visible anchors; the list is handed to the decode by
    `take_compaction(mask)` when render() is called with this very mask, replacing torch.nonzero and its syncs."""
    rs = raster_settings
    with torch.no_grad():
        L = _lib.lib()
        _require_cuda(means3D, scales, rotations, rs.viewmatrix, rs.projmatrix)
        dev = means3D.device
        N = int(means3D.shape[0])
        mask_u8 = torch.empty(N, dtype=torch.uint8, device=dev)
        if N == 0:
            return mask_u8.view(torch.bool)
        means3D = _f32c(means3D.detach())
        rotations = _f32c(rotations.detach())
        scales, sstride = _rows_f32(scales.detach(), 3)
        view, proj = _f32c(rs.viewmatrix), _f32c(rs.projmatrix)
        cp = _Compaction()
        with _lib.on_device(dev), stage("visible_filter"):
            radii = torch.empty(N, dtype=torch.int32, device=dev)
            cp.idx = torch.empty(N, dtype=torch.int32, device=dev)
            ws = torch.empty(L.splatco_visible_compact_ws_bytes(N), dtype=torch.uint8, device=dev)
            cp.counter = _pinned_counter(dev, 2)
            check(L.splatco_visible_filter_compact(N, ptr(means3D), ptr(scales), sstride, ptr(rotations),
                                                   float(rs.scale_modifier), ptr(view), ptr(proj), float(rs.tanfovx),
                                                   float(rs.tanfovy), int(rs.image_height), int(rs.image_width),
                                                   ptr(radii), ptr(mask_u8), ptr(cp.idx), ptr(ws), cp.counter.data_ptr(),
                                                   _stream_ptr(dev)), "splatco_visible_filter_compact")
            cp.event = torch.cuda.Event()
            cp.event.record(torch.cuda.current_stream(dev))
            cp.ws = ws                                       # holds the device-side count (cp.count_ptr)
            cp.count_ptr = L.splatco_visible_compact_count_ptr(ptr(ws), N)
        _debug_sync(rs, "visible_filter")
        cp.mask = mask_u8.view(torch.bool)
        cp.version = cp.mask._version
        _spec_slot.compaction = cp
        return cp.mask


def pending_compaction(visible_mask):
    """The pending compaction record of `visible_mask` WITHOUT waiting for it: `.idx` (int32 [N], the first V entries
    valid once the filter has run), `.count_ptr` (device address of V), `.counter` / `.event` (the pinned read-back).
    The decode queues itself on these and reads V after its own sync.  None if the mask is not the last prefilter's."""
    cp = getattr(_spec_slot, "compaction", None)
    if cp is None or cp.mask is not visible_mask or visible_mask._version != cp.version:
        return None
    return cp


def clear_compaction(cp):
    if getattr(_spec_slot, "compaction", None) is cp:
        _spec_slot.compaction = None


def take_compaction(visible_mask):
    """(idx int32 [V], V) if `visible_mask` is the untouched tensor the last visible_mask_compact returned, else None.
    Waits for the filter's read-back only (an event), not for the stream."""
    cp = getattr(_spec_slot, "compaction", None)
    if cp is None or cp.mask is not visible_mask or visible_mask._version != cp.version:
        return None
    _spec_slot.compaction = None
    cp.event.synchronize()
    V = int(cp.counter[0])
    return cp.idx[:V], V
