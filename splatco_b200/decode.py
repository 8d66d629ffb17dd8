"""Fused anchor decode: host side of splatco_decode_* (include/splatco_b200.h).

Mirrors the contract of the reference's `generate_neural_gaussians`
(gaussian_renderer/__init__.py:18-116): same inputs read off the same `pc` attributes, same 7-tuple
(train) / 5-tuple (eval) of outputs, gradients delivered to the same leaves through autograd.
All arithmetic runs in libsplatco_b200.so, TriPlaneAttention over the whole planes included (a dense,
view-independent pass — SURVEY §8 row f2 — evaluated once per iteration by splatco_ta_fwd/_bwd and cached
across the mv views, `_TACache`).
"""
from __future__ import annotations

import ctypes as C
import threading
import weakref

import torch

from . import _gradacc, _lib
from ._lib import check
from .profiling import stage

_fp = C.POINTER(C.c_float)
_vp = C.c_void_p


class DecodeDesc(C.Structure):
    _fields_ = [
        ("N", C.c_int32), ("V", C.c_int32), ("K", C.c_int32), ("rc", C.c_int32), ("level", C.c_int32),
        ("app_dim", C.c_int32),
        ("E", C.c_int32 * 3), ("use_dist", C.c_int32 * 3), ("update_running", C.c_int32),
        ("xyz_min", _vp), ("xyz_max", _vp), ("cam", _vp),
        ("bn_eps", C.c_float), ("bn_momentum", C.c_float),
        ("anchor_feat", _vp), ("anchor", _vp), ("offset", _vp), ("scaling", _vp), ("vis", _vp),
        ("plane", _vp * 9), ("att", _vp * 3),
        ("bn_w", _vp * 3), ("bn_b", _vp * 3), ("lin_w", _vp * 3), ("lin_b", _vp * 3),
        ("cbn_w", _vp * 3), ("cbn_b", _vp * 3), ("clin_w", _vp * 3), ("clin_b", _vp * 3),
        ("bn_rm", _vp * 3), ("bn_rv", _vp * 3), ("cbn_rm", _vp * 3), ("cbn_rv", _vp * 3),
        ("bn_nbt", _vp * 3), ("cbn_nbt", _vp * 3),
        ("w1", _vp * 3), ("b1", _vp * 3), ("w2", _vp * 3), ("b2", _vp * 3),
        ("app_vec", _vp), ("noise", _vp), ("noise_q", C.c_float), ("noise_seed", C.c_uint64), ("plane_layout", C.c_int32),
        ("V_dev", _vp), ("V_layout", C.c_int32),
    ]


class DecodeGrads(C.Structure):
    _fields_ = [
        ("anchor_feat", _vp), ("anchor", _vp), ("offset", _vp), ("scaling", _vp),
        ("plane", _vp * 9), ("att", _vp * 3),
        ("bn_w", _vp * 3), ("bn_b", _vp * 3), ("lin_w", _vp * 3), ("lin_b", _vp * 3),
        ("cbn_w", _vp * 3), ("cbn_b", _vp * 3), ("clin_w", _vp * 3), ("clin_b", _vp * 3),
        ("w1", _vp * 3), ("b1", _vp * 3), ("w2", _vp * 3), ("b2", _vp * 3),
        ("app_vec", _vp),
    ]


_registered = False


def _register():
    return _lib.lib()       # signatures live in _lib.SIGNATURES


_tls = threading.local()


def _pinned_counter(dev):
    cache = getattr(_tls, "c", None)
    if cache is None:
        cache = _tls.c = {}
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in cache:
        cache[key] = torch.zeros(1, dtype=torch.int32).pin_memory()
    return cache[key]


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _c(t):
    t = t.detach()
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


class DecodeConfig:
    """Everything that is not a differentiable tensor input."""
    __slots__ = ("N", "K", "rc", "level", "E", "use_dist", "app_dim", "xyz_min", "xyz_max", "cam",
                 "bn_eps", "bn_momentum", "update_running", "buffers", "vis_idx", "noise", "noise_q", "noise_seed", "plan", "raster", "packed",
                 "pending", "depth_alpha", "cam_grad")


# order of the differentiable parameter list handed to the autograd Function
PER_LEVEL = ("xy", "xz", "yz", "bn_w", "bn_b", "lin_w", "lin_b", "cbn_w", "cbn_b", "clin_w", "clin_b")
PER_HEAD = ("w1", "b1", "w2", "b2")


_NGRAD = 53
_GradPtrs = C.c_void_p * _NGRAD
assert C.sizeof(_GradPtrs) == C.sizeof(DecodeGrads)
_slot_cache = {}


def _grad_slots(nl):
    """forward-argument index (anchor_feat, anchor, offset, scaling, att x3, app_vec, per-level x11, heads x4)
    -> pointer slot of splatco_decode_grads."""
    m = _slot_cache.get(nl)
    if m is None:
        m = [0, 1, 2, 3, 13, 14, 15, 52]
        for l in range(nl):
            m += [4 + 3 * l, 5 + 3 * l, 6 + 3 * l] + [16 + 3 * j + l for j in range(8)]
        for h in range(3):
            m += [40 + 3 * j + h for j in range(4)]
        _slot_cache[nl] = m
    return m


def _plain(t):
    return t.dtype == torch.float32 and t.is_contiguous()


def _fill_desc(cfg: DecodeConfig, V, anchor_feat, anchor, offset, scaling, att, app_vec, params):
    """Descriptor for one view.  The ~100 parameter / buffer pointers only change when the optimizer or
    densification swaps tensors, so a filled template is cached on the config's plan and copied."""
    plan = cfg.plan
    key = (tuple([t.data_ptr() for t in params]), tuple(cfg.use_dist), cfg.app_dim, cfg.level, cfg.N, id(cfg.buffers),
           cfg.xyz_min.data_ptr())
    if plan.desc_key != key:
        d = DecodeDesc()
        d.N, d.K, d.rc, d.level, d.app_dim = cfg.N, cfg.K, cfg.rc, cfg.level, cfg.app_dim
        for q in range(3):
            d.E[q] = cfg.E[q]
            d.use_dist[q] = int(cfg.use_dist[q])
        d.xyz_min, d.xyz_max = cfg.xyz_min.data_ptr(), cfg.xyz_max.data_ptr()
        d.bn_eps, d.bn_momentum = cfg.bn_eps, cfg.bn_momentum
        nl = cfg.level + 1
        for l in range(nl):
            lp = dict(zip(PER_LEVEL, params[l * len(PER_LEVEL):(l + 1) * len(PER_LEVEL)]))
            d.plane[3 * l], d.plane[3 * l + 1], d.plane[3 * l + 2] = (lp[k].data_ptr() for k in ("xy", "xz", "yz"))
            for k in ("bn_w", "bn_b", "lin_w", "lin_b", "cbn_w", "cbn_b", "clin_w", "clin_b"):
                getattr(d, k)[l] = lp[k].data_ptr()
            bufs = cfg.buffers[l]
            for k in ("bn_rm", "bn_rv", "cbn_rm", "cbn_rv", "bn_nbt", "cbn_nbt"):
                getattr(d, k)[l] = bufs[k].data_ptr() if bufs.get(k) is not None else None
        base = nl * len(PER_LEVEL)
        for h in range(3):
            for n, k in enumerate(PER_HEAD):
                getattr(d, k)[h] = params[base + h * 4 + n].data_ptr()
        plan.desc_key, plan.desc = key, d
    d = DecodeDesc.from_buffer_copy(plan.desc)
    d.N, d.V = cfg.N, V
    d.update_running = int(cfg.update_running)
    d.cam = cfg.cam.data_ptr()
    d.anchor_feat, d.anchor, d.offset, d.scaling = (anchor_feat.data_ptr(), anchor.data_ptr(), offset.data_ptr(),
                                                    scaling.data_ptr())
    d.vis = cfg.vis_idx.data_ptr()
    d.att[0], d.att[1], d.att[2] = att[0].data_ptr(), att[1].data_ptr(), att[2].data_ptr()
    d.app_vec = app_vec.data_ptr() if app_vec is not None else None
    d.noise = cfg.noise.data_ptr() if cfg.noise is not None else None
    d.noise_q, d.noise_seed = cfg.noise_q, cfg.noise_seed
    d.plane_layout = 1 if cfg.packed else 0
    d.V_dev, d.V_layout = None, 0
    return d


class _FusedDecode(torch.autograd.Function):
    @staticmethod
    def forward(ctx, cfg: DecodeConfig, anchor_feat, anchor, offset, scaling, att_xy, att_xz, att_yz, app_vec,
                *params):
        # cfg.cam_grad: the last input is the camera centre (the tensor cfg.cam was read from), which wants a gradient
        if cfg.cam_grad:
            ctx.cam_meta = (params[-1].shape, params[-1].dtype)
            params = params[:-1]
        L = _register()
        dev = anchor.device
        # kernels read fp32 contiguous memory; tensors that already are (the normal case) are used in place
        tensors = [t if _plain(t) else _c(t) for t in (anchor_feat, anchor, offset, scaling, att_xy, att_xz, att_yz)]
        anchor_feat_c, anchor_c, offset_c, scaling_c, a_xy, a_xz, a_yz = tensors
        app_c = None if app_vec is None else (app_vec if _plain(app_vec) else _c(app_vec))
        plan = cfg.plan
        ids = tuple(map(id, params))
        if plan.param_ids == ids:
            pc = params                                       # same Parameter objects as last view: all fp32 contiguous
        else:
            pc = [t if _plain(t) else _c(t) for t in params]
            plan.param_ids = ids if all(a is b for a, b in zip(pc, params)) else None
        K = cfg.K
        cp = cfg.pending if (cfg.raster is not None and 1 <= cfg.rc <= 5) else None
        if cfg.pending is not None and cp is None:       # not the two-stage decode after all: the round-1 order
            from .diff_gaussian_rasterization import clear_compaction
            cfg.pending.event.synchronize()
            cfg.vis_idx = cfg.pending.idx[:int(cfg.pending.counter[0])]
            clear_compaction(cfg.pending)
            cfg.pending = None
        # V: exact, or (cp: count still on the device) the capacity N every buffer of this view is sized for
        V = int(cfg.vis_idx.shape[0])
        desc = _fill_desc(cfg, V, anchor_feat_c, anchor_c, offset_c, scaling_c, (a_xy, a_xz, a_yz), app_c, pc)
        if cp is not None:
            desc.V_dev, desc.V_layout = cp.count_ptr, V
        stream = _lib.raw_stream(dev)
        with _lib.on_device(dev):
            ws = _lib.empty_u8(L.splatco_decode_fwd_ws_bytes(V, cfg.rc, cfg.level), dev)
            nopac = _lib.empty_rows(V * K, 1, torch.float32, dev)
            mask = _lib.empty_rows(V * K, None, torch.bool, dev)
            counter = _pinned_counter(dev)
            with stage("decode_fwd"):
                check(L.splatco_decode_fwd(C.byref(desc), _p(ws), _p(nopac), _p(mask), counter.data_ptr(), stream),
                      "splatco_decode_fwd")
            f32 = dict(dtype=torch.float32, device=dev)
            if cfg.raster is not None and V > 0:
                # render() path: compaction and the rasterizer's preprocess are queued on VK-row buffers with the
                # survivor count still on the device, then ONE sync returns both M and the instance count R
                # (the reference syncs twice here: boolean indexing, then num_rendered)
                from . import diff_gaussian_rasterization as _dgr
                VK = V * K
                bufs = [_lib.empty_rows(VK, c, torch.float32, dev) for c in (3, 3, 1, 3, 4)]
                with stage("decode_emit"):
                    check(L.splatco_decode_emit(C.byref(desc), _p(ws), VK, *[_p(b) for b in bufs], stream),
                          "splatco_decode_emit")
                sp = _dgr.preprocess_speculative(*bufs, L.splatco_decode_count_ptr(_p(ws), V, cfg.rc, cfg.level), cfg.raster,
                                                  depth_alpha=cfg.depth_alpha)
                sp.event.synchronize()             # M, R (and V) have landed; binning + blend keep running behind it
                M = int(counter[0])
                if cp is not None:
                    from .diff_gaussian_rasterization import clear_compaction
                    clear_compaction(cp)
                    V_cap, V = V, int(cp.counter[0])
                    if V == 1:                      # (V = 0: an empty view, legal as before)
                        raise RuntimeError(f"splatco_decode_fwd failed (-1): decode: BatchNorm in train mode needs more than 1 "
                                           f"visible anchor (got {V})")
                    desc.V, desc.V_dev = V, None   # the backward (and everything after the sync) works with the exact V
                    cfg.vis_idx = cp.idx[:V]
                    nopac, mask = nopac[:V * K], mask[:V * K]
                    cfg.pending = None
                xyz, color, opacity, scl, rot = [b[:M] for b in bufs]
                _dgr.publish_speculated(sp, M, (xyz, color, opacity, scl, rot))
            else:
                torch.cuda.current_stream(dev).synchronize()      # M sizes the outputs (the reference syncs here too: boolean indexing)
                M = int(counter[0]) if V > 0 else 0
                xyz, color, opacity, scl, rot = [torch.empty((M, c), **f32) for c in (3, 3, 1, 3, 4)]
                with stage("decode_emit"):
                    check(L.splatco_decode_emit(C.byref(desc), _p(ws), M, _p(xyz), _p(color), _p(opacity), _p(scl), _p(rot),
                                                stream), "splatco_decode_emit")
        ctx.cfg, ctx.desc, ctx.ws, ctx.M, ctx.V = cfg, desc, ws, M, V
        ctx.V_rows = int(desc.V_layout) or V                    # rows the workspaces are laid out for
        _v_last[id(cfg.plan)] = V
        # everything a pointer in desc refers to stays alive with the node
        ctx.keep = (tensors, app_c, pc, cfg.vis_idx, cfg.noise, cfg.xyz_min, cfg.xyz_max, cfg.cam)
        # the forward input OBJECTS: their identity keys the shared gradient buffers of a backward pass
        ctx.origs = (anchor_feat, anchor, offset, scaling, att_xy, att_xz, att_yz, app_vec) + tuple(params)
        ctx.mark_non_differentiable(mask)
        ctx.set_materialize_grads(False)          # unused outputs (neural_opacity, the mask) get no zero-filled gradients
        return xyz, color, opacity, scl, rot, nopac, mask

    @staticmethod
    def backward(ctx, g_xyz, g_color, g_opacity, g_scl, g_rot, g_nopac, _g_mask):
        L = _register()
        cfg, desc, V, M = ctx.cfg, ctx.desc, ctx.V, ctx.M
        tensors, app_c, pc = ctx.keep[:3]
        dev = tensors[1].device
        nl = cfg.level + 1
        # One destination per differentiable input, in forward-argument order.  splatco_decode_bwd
        # accumulates, so nodes of the same backward pass that were fed the same tensor share one
        # zero-filled buffer (_gradacc): no per-view N-row / plane-sized temporaries, no autograd adds.
        origs = ctx.origs                      # forward inputs 1.. (anchor_feat, ..., app_vec, *params)
        need = ctx.needs_input_grad[1:]
        shapes = [t.shape for t in tensors] + [app_c.shape if app_c is not None else None] + [t.shape for t in pc]
        reqs, where = [], []
        for n, (o, shp) in enumerate(zip(origs, shapes)):
            if shp is None:
                continue
            reqs.append((id(o) if need[n] else None, shp, bool(getattr(o, "is_leaf", True))))
            where.append(n)
        with _lib.on_device(dev):
            got = _gradacc.acquire(dev, reqs)
        slots = _grad_slots(nl)
        vals = [None] * _NGRAD
        rets = [None] * len(origs)                 # (a camera centre input is last; its gradient is appended below)
        for n, (ptr_n, ret) in zip(where, got):
            vals[slots[n]] = ptr_n
            rets[n] = ret if need[n] else None
        del got
        gd = _GradPtrs(*vals)                  # same memory layout as splatco_decode_grads (all pointers)
        cam = cfg.cam_grad and ctx.needs_input_grad[-1]
        d_cam = torch.zeros(3, dtype=torch.float32, device=dev) if cam else None
        if V > 0:
            ups = [_c(t) if t is not None else None for t in (g_xyz, g_color, g_opacity, g_scl, g_rot, g_nopac)]
            if M > 0:
                z = lambda *s: torch.zeros(*s, dtype=torch.float32, device=dev)
                ups = [u if u is not None else z(*s) for u, s in zip(ups[:5], ((M, 3), (M, 3), (M, 1), (M, 3), (M, 4)))] + [ups[5]]
            stream = _lib.raw_stream(dev)
            with _lib.on_device(dev):
                bws = _lib.empty_u8(L.splatco_decode_bwd_ws_bytes(ctx.V_rows, cfg.rc, cfg.level), dev)
                with stage("decode_bwd"):
                    if cam:
                        cam_ws = _lib.empty_u8(L.splatco_camera_grad_ws_bytes(V), dev)
                        check(L.splatco_decode_bwd_camera(C.byref(desc), _p(ctx.ws), _p(bws), M, *[_p(u) for u in ups],
                                                          gd, _p(cam_ws), _p(d_cam), stream), "splatco_decode_bwd_camera")
                    else:
                        check(L.splatco_decode_bwd(C.byref(desc), _p(ctx.ws), _p(bws), M, *[_p(u) for u in ups],
                                                   gd, stream), "splatco_decode_bwd")
        if not cfg.cam_grad:
            return (None, *rets)
        shape, dtype = ctx.cam_meta
        return (None, *rets, d_cam.to(dtype).reshape(shape) if cam else None)


def _bn_lin(seq):
    bn, lin = seq[0], seq[1]
    return bn, lin


class _TriPlaneAttention(torch.autograd.Function):
    """TriPlaneAttention.forward (scene/grids.py:22-64) on the three TA-level planes, in
    libsplatco_b200.so (csrc/triplane_attention.cu).  Inputs: xy/xz/yz planes [1, rc, E, E] and the
    three Conv2d weights of the module; outputs: the three attended planes."""

    @staticmethod
    def forward(ctx, xy, xz, yz, w_ca1, w_ca2, w_sa):
        L = _register()
        if not xy.is_cuda:
            raise RuntimeError("splatco_b200 TriPlaneAttention needs CUDA tensors (no CPU fallback)")
        dev = xy.device
        ins = [t if _plain(t) else _c(t) for t in (xy, xz, yz, w_ca1, w_ca2, w_sa)]
        rc, E = int(xy.shape[1]), int(xy.shape[2])
        hidden, ksize = int(w_ca1.shape[0]), int(w_sa.shape[-1])
        if not (xy.shape == xz.shape == yz.shape and xy.shape[2] == xy.shape[3]):
            raise NotImplementedError("splatco_b200 TriPlaneAttention supports equal square planes only")
        with _lib.on_device(dev):
            ws = torch.empty(L.splatco_ta_fwd_ws_bytes(rc, E), dtype=torch.uint8, device=dev)
            outs = [torch.empty_like(ins[q]) for q in range(3)]
            with stage("triplane_attention_fwd"):
                check(L.splatco_ta_fwd(rc, E, hidden, ksize, *[_p(t) for t in ins], _p(ws), *[_p(t) for t in outs],
                                       _lib.raw_stream(dev)), "splatco_ta_fwd")
        ctx.ins, ctx.ws, ctx.dims = ins, ws, (rc, E, hidden, ksize)
        ctx.origs = (xy, xz, yz, w_ca1, w_ca2, w_sa)
        return tuple(outs)

    @staticmethod
    def backward(ctx, g_xy, g_xz, g_yz):
        L = _register()
        rc, E, hidden, ksize = ctx.dims
        ins = ctx.ins
        dev = ins[0].device
        need = ctx.needs_input_grad
        # plane gradients go into the same per-backward-pass buffers the decode nodes scatter their
        # direct (un-attended) level-0 plane gradients into (_gradacc)
        with _lib.on_device(dev):
            got = _gradacc.acquire(dev, [(id(o) if need[n] else None, t.shape, bool(o.is_leaf)) for n, (o, t) in enumerate(zip(ctx.origs, ins))])
            ptrs = [g[0] for g in got]
            rets = [g[1] if need[n] else None for n, g in enumerate(got)]
            del got
            gs = [g if g is not None else torch.zeros_like(ins[q]) for q, g in enumerate((g_xy, g_xz, g_yz))]
            gs = [g if _plain(g) else _c(g) for g in gs]
            bws = torch.empty(L.splatco_ta_bwd_ws_bytes(rc, E), dtype=torch.uint8, device=dev)
            with stage("triplane_attention_bwd"):
                check(L.splatco_ta_bwd(rc, E, hidden, ksize, *[_p(t) for t in ins], _p(ctx.ws), _p(bws),
                                       *[_p(g) for g in gs], *ptrs,
                                       _lib.raw_stream(dev)), "splatco_ta_bwd")
        return tuple(rets)


class _PackPlanes(torch.autograd.Function):
    """Channel-last copies [E,E,8] of three [1,rc,E,E] planes (splatco_pack_planes); backward adds the
    channel-last gradients back into the planes' gradient buffers of this backward pass."""

    @staticmethod
    def forward(ctx, xy, xz, yz):
        L = _register()
        dev = xy.device
        ins = [t if _plain(t) else _c(t) for t in (xy, xz, yz)]
        rc, E = int(xy.shape[1]), int(xy.shape[2])
        with _lib.on_device(dev):
            outs = [torch.empty((E, E, 8), dtype=torch.float32, device=dev) for _ in range(3)]
            with stage("pack_planes"):
                check(L.splatco_pack_planes(rc, E, *[_p(t) for t in ins], *[_p(t) for t in outs], _lib.raw_stream(dev)),
                      "splatco_pack_planes")
        ctx.dims, ctx.origs, ctx.shapes = (rc, E), (xy, xz, yz), [t.shape for t in ins]
        return tuple(outs)

    @staticmethod
    def backward(ctx, g_xy, g_xz, g_yz):
        L = _register()
        rc, E = ctx.dims
        dev = ctx.origs[0].device
        need = ctx.needs_input_grad
        with _lib.on_device(dev):
            got = _gradacc.acquire(dev, [(id(o) if need[n] else None, shp, bool(o.is_leaf)) for n, (o, shp) in enumerate(zip(ctx.origs, ctx.shapes))])
            ptrs = [g[0] for g in got]
            rets = [g[1] if need[n] else None for n, g in enumerate(got)]
            del got
            gs = [g if g is not None else torch.zeros((E, E, 8), dtype=torch.float32, device=dev) for g in (g_xy, g_xz, g_yz)]
            gs = [g if _plain(g) else _c(g) for g in gs]
            with stage("unpack_planes"):
                check(L.splatco_unpack_planes_add(rc, E, *[_p(g) for g in gs], *ptrs, _lib.raw_stream(dev)),
                      "splatco_unpack_planes_add")
        return tuple(rets)


# "auto": pack when the mv views of an iteration amortise the two extra passes over the planes; True / False force it
# (SPLATCO_PACK_PLANES=0|1 in the environment forces it for A/B timing)
import os as _os
PACK_PLANES = {"0": False, "1": True}.get(_os.environ.get("SPLATCO_PACK_PLANES", ""), "auto")


class _PackCache:
    """Channel-last plane copies are view-independent like TriPlaneAttention's output: built on the first
    view of an iteration, reused by the others, dropped when a plane changes (optimizer step) or once a
    backward pass has flowed through them.  `uses` of the previous generation estimates mv."""

    def __init__(self):
        self.key, self.value, self.uses, self.last_uses = None, None, 0, 1

    def get(self, planes, V):
        key = (torch.is_grad_enabled(),) + tuple((id(t), t._version, t.data_ptr()) for t in planes)
        if self.key == key:
            self.uses += 1
            return self.value
        if self.key is not None:
            self.last_uses = max(self.uses, 1)
        self.key, self.uses = key, 1
        want = PACK_PLANES
        if want == "auto":
            # measured on B200 (round 2, C2): with the one-thread-per-anchor gather / scatter kernels (16-byte texel
            # loads, vector REDs) the channel-last layout saves ~1.2 ns per visible anchor and view; packing, unpacking
            # and zero-filling cost ~0.6 us per MB of planes per iteration -> worth it from ~500 anchor-views per MB
            # (C2 at mv = 4: 1850 per MB, yes: 2.26 -> 2.16 ms/view)
            plane_mb = sum(t.numel() for t in planes) * 4 / 1e6
            want = V * self.last_uses > 600.0 * plane_mb
        if not want or int(planes[0].shape[1]) > 8:
            self.value = None
            return None
        packed = []
        for q in range(0, len(planes), 3):
            packed += list(_PackPlanes.apply(*planes[q:q + 3]))
        if packed[0].requires_grad:
            packed[0].register_hook(self._invalidate)
        self.value = tuple(packed)
        return self.value

    def _invalidate(self, grad):
        self.key, self.value = None, None
        return grad


_pack_caches = {}


def _pack_cache_for(owner) -> _PackCache:
    c = _pack_caches.get(id(owner))
    if c is None:
        if len(_pack_caches) > 8:
            _pack_caches.clear()
        c = _pack_caches[id(owner)] = _PackCache()
    return c


class _TACache:
    """TriPlaneAttention is view-independent (it only reads the level-0 planes and its own weights) but
    the reference recomputes it for every view (SURVEY §8 row a4/f2).  Its output is cached here and
    re-used by all views of an iteration: autograd then sums the views' gradients into the ONE cached
    node and runs the attention backward once.  The entry is dropped when any input tensor is modified
    in place (optimizer.step bumps `_version`), replaced (densification swaps Parameters), when the grad
    mode changes, or as soon as a backward pass has flowed through it (the graph is gone after that)."""

    def __init__(self):
        self.key = None
        self.value = None

    def get(self, planes, weights):
        ts = list(planes) + list(weights)
        key = (torch.is_grad_enabled(),) + tuple((id(t), t._version, t.data_ptr(), tuple(t.shape)) for t in ts)
        if self.key == key and self.value is not None:
            return self.value
        att = _TriPlaneAttention.apply(*planes, *weights)
        if att[0].requires_grad:
            att[0].register_hook(self._invalidate)
        self.key, self.value = key, att
        return att

    def _invalidate(self, grad):
        self.key, self.value = None, None
        return grad


_ta_caches = {}


def _ta_cache_for(owner) -> _TACache:
    c = _ta_caches.get(id(owner))
    if c is None:
        if len(_ta_caches) > 8:
            _ta_caches.clear()
        c = _ta_caches[id(owner)] = _TACache()
    return c


class _ModelPlan:
    """Per-model state that survives between views: handles of the modules the decode reads (so the ~50
    parameter tensors are fetched with dict lookups instead of nn.Module attribute resolution), the
    static sizes, and the descriptor template (_fill_desc)."""
    __slots__ = ("feat_ref", "level", "heads", "levels", "rc", "E", "xyz_min", "xyz_max", "bn_eps", "bn_momentum",
                 "buffers", "ta_weights", "desc_key", "desc", "param_ids", "bbox_src")


_plans = {}


def _par(module, name):
    try:
        return module._parameters[name]
    except (AttributeError, KeyError):
        return getattr(module, name)


def _plan_for(pc, feat, level, heads) -> _ModelPlan:
    plan = _plans.get(id(pc))
    if (plan is not None and plan.feat_ref() is feat and plan.level == level
            and all(a is b for a, b in zip(plan.heads, heads))
            # buffers are captured as tensor objects: module.to() / load_state_dict(assign=True) replace them
            and all(lv[1]._buffers.get("running_mean") is bf["bn_rm"] and lv[3]._buffers.get("running_mean") is bf["cbn_rm"]
                    for lv, bf in zip(plan.levels, plan.buffers))
            and plan.bbox_src[0] is feat.k0s[0].xyz_min and plan.bbox_src[1] is feat.k0s[0].xyz_max):
        return plan
    k0s = feat.k0s
    for l in range(level + 1):
        pl = k0s[l]
        if not (pl.xy_plane.shape[2] == pl.xy_plane.shape[3] == pl.xz_plane.shape[3] == pl.yz_plane.shape[2]):
            raise NotImplementedError("splatco_b200 decode supports cubic plane grids only (world_size = [s, s, s])")
    plan = _ModelPlan()
    plan.feat_ref, plan.level, plan.heads = weakref.ref(feat), level, tuple(heads)
    plan.rc = int(k0s[0].xy_plane.shape[1])
    plan.E = [int(k0s[min(l, len(k0s) - 1)].xy_plane.shape[2]) for l in range(3)]
    plan.xyz_min, plan.xyz_max = _c(k0s[0].xyz_min), _c(k0s[0].xyz_max)      # stay on the device: no host sync
    plan.bbox_src = (k0s[0].xyz_min, k0s[0].xyz_max)
    bn0 = feat.models[0][0]
    plan.bn_eps, plan.bn_momentum = float(bn0.eps), float(bn0.momentum if bn0.momentum is not None else 0.1)
    plan.levels, plan.buffers = [], []
    for l in range(level + 1):
        bn, lin = _bn_lin(feat.models[l])
        cbn, clin = _bn_lin(feat.CTX_models[l])
        plan.levels.append((k0s[l], bn, lin, cbn, clin))
        plan.buffers.append(dict(bn_rm=bn.running_mean, bn_rv=bn.running_var, cbn_rm=cbn.running_mean,
                                 cbn_rv=cbn.running_var, bn_nbt=bn.num_batches_tracked,
                                 cbn_nbt=cbn.num_batches_tracked))
    ta = k0s[0].TA
    plan.ta_weights = (ta.ca.sharedMLP[0], ta.ca.sharedMLP[2], ta.sa.conv)
    plan.desc_key = plan.desc = plan.param_ids = None
    if len(_plans) > 8:
        _plans.clear()
    _plans[id(pc)] = plan
    return plan


_v_last = {}        # id(model) -> visible-anchor count of its last view (sizing heuristics only)


def collect_model(pc, viewpoint_camera, visible_mask, update_running=True, defer_count=False):
    """Read the reference model's attributes (duck-typed GaussianModel, SURVEY §8b) into
    (cfg, differentiable inputs)."""
    if getattr(pc, "use_feat_bank", False):
        raise NotImplementedError(
            "use_feat_bank is unusable in the reference itself (mlp_feature_bank is Linear(4, .) but is fed 68 "
            "columns, scene/gaussian_model.py:307-313 vs gaussian_renderer/__init__.py:42-44)")
    anchor = pc.get_anchor
    dev = anchor.device
    if not anchor.is_cuda:
        raise RuntimeError("splatco_b200 decode needs CUDA tensors (no CPU fallback)")
    feat = pc.feat_planes._feat
    level = int(feat.activate_level)
    heads = (pc.get_opacity_mlp, pc.get_cov_mlp, pc.get_color_mlp)
    plan = _plan_for(pc, feat, level, heads)
    cfg = DecodeConfig()
    cfg.plan = plan
    cfg.N = int(anchor.shape[0])
    cfg.K = int(pc.n_offsets)
    cfg.level, cfg.rc, cfg.E = level, plan.rc, plan.E
    cfg.use_dist = [bool(pc.add_opacity_dist), bool(pc.add_cov_dist), bool(pc.add_color_dist)]
    cfg.app_dim = int(pc.appearance_dim) if pc.appearance_dim else 0
    cfg.xyz_min, cfg.xyz_max = plan.xyz_min, plan.xyz_max
    cam = viewpoint_camera.camera_center
    cfg.cam = cam if _plain(cam) else _c(cam)
    cfg.bn_eps, cfg.bn_momentum = plan.bn_eps, plan.bn_momentum
    cfg.update_running = bool(update_running)
    cfg.buffers = plan.buffers
    params = []
    for pl, bn, lin, cbn, clin in plan.levels:
        params += [_par(pl, "xy_plane"), _par(pl, "xz_plane"), _par(pl, "yz_plane"), _par(bn, "weight"), _par(bn, "bias"),
                   _par(lin, "weight"), _par(lin, "bias"), _par(cbn, "weight"), _par(cbn, "bias"),
                   _par(clin, "weight"), _par(clin, "bias")]
    for mlp in heads:
        m0, m2 = mlp[0], mlp[2]
        params += [_par(m0, "weight"), _par(m0, "bias"), _par(m2, "weight"), _par(m2, "bias")]
    # TriPlaneAttention over the level-0 planes (scene/grids.py:166-169)
    att = _ta_cache_for(plan.levels[0][0]).get(tuple(params[0:3]), tuple(_par(m, "weight") for m in plan.ta_weights))
    # the visible-anchor list LAST: everything above is independent of it and overlaps with the GPU finishing the
    # prefilter (and whatever was queued before it); prefilter_voxel already compacted the indices on the device
    cfg.pending = None
    if visible_mask is None:
        cfg.vis_idx = torch.arange(cfg.N, dtype=torch.int32, device=dev)
        v_est = cfg.N
    else:
        from .diff_gaussian_rasterization import pending_compaction, take_compaction
        cp = pending_compaction(visible_mask) if defer_count else None
        if cp is not None:
            # render() path on the two-stage decode: the visible-anchor COUNT stays on the device (desc.V_dev), the decode
            # is queued on N-row buffers, and the host learns V together with M and R at the ONE sync of the view
            cfg.pending = cp
            cfg.vis_idx = cp.idx
            v_est = _v_last.get(id(plan), (3 * cfg.N) // 4)
        else:
            got = take_compaction(visible_mask)
            cfg.vis_idx = got[0] if got is not None else torch.nonzero(visible_mask).squeeze(1).to(torch.int32)
            v_est = int(cfg.vis_idx.shape[0])
    # channel-last copies of every sampled plane (direct planes of the active levels + the attended ones)
    nper = len(PER_LEVEL)
    planes = [params[l * nper + q] for l in range(level + 1) for q in range(3)] + list(att)
    packed = _pack_cache_for(plan.levels[0][0]).get(planes, v_est)
    cfg.packed = packed is not None
    if cfg.packed:
        for l in range(level + 1):
            params[l * nper: l * nper + 3] = packed[3 * l: 3 * l + 3]
        att = packed[3 * (level + 1):]
    app_vec = None
    if cfg.app_dim > 0:
        app_vec = pc.get_appearance.embedding.weight[int(viewpoint_camera.uid)]
    return cfg, att, app_vec, params


_noise_calls = 0
# SPLATCO_DEFER_COUNT=0: wait for the prefilter's count before the decode is queued (the round-1 order; A/B timing)
DEFER_COUNT = _os.environ.get("SPLATCO_DEFER_COUNT", "1") != "0"


def generate_neural_gaussians(viewpoint_camera, pc, visible_mask=None, is_training=False, _raster_settings=None,
                              _scaling=None, _depth_alpha=False):
    """Drop-in for gaussian_renderer.generate_neural_gaussians (reference :18-116).  `_raster_settings`
    is render()'s private hint: the GaussianRasterizationSettings it is about to rasterize the result
    with, which lets the decode queue the rasterizer's preprocess before its own row count is known;
    `_depth_alpha` says whether that rasterization also produces the depth and alpha maps."""
    # the per-anchor inputs first (pc.get_scaling launches two kernels): collect_model ends by waiting for the
    # prefilter's visible-anchor count, and everything queued before that wait overlaps with the GPU's backlog
    scaling_in = _scaling if _scaling is not None else pc.get_scaling
    # (an explicit noise tensor -- tests -- is [V, ncol]: it needs V on the host first)
    defer = (_raster_settings is not None and DEFER_COUNT and getattr(pc.feat_planes, "_splatco_noise", None) is None
             and _register().splatco_decode_get_impl() == 2)
    cfg, att, app_vec, params = collect_model(pc, viewpoint_camera, visible_mask, defer_count=defer)
    cfg.raster = _raster_settings
    cfg.depth_alpha = bool(_depth_alpha)
    # a camera centre that requires grad (a pose being optimised) becomes a differentiable input of the decode
    cam = viewpoint_camera.camera_center
    cam_in = (cam,) if torch.is_grad_enabled() and cam.requires_grad else ()
    cfg.cam_grad = bool(cam_in)
    # GaussianLearner.inference always passes Q = self.Q0 (0.03 while training, 0 in render.py):
    # U(-.5,.5)*Q is added to the plane features of the non-TA levels (scene/grids.py:159-164)
    Q = float(getattr(pc.feat_planes, "Q0", 0.0) or 0.0)
    cfg.noise = getattr(pc.feat_planes, "_splatco_noise", None)      # tests inject an explicit [V, ncol] noise tensor here
    cfg.noise_q, cfg.noise_seed = 0.0, 0
    if cfg.noise is None and Q != 0.0 and cfg.level >= 1:
        # generated inside the gather kernel from (torch's seed, call counter): no [V, ncol] tensor, no torch launches
        global _noise_calls
        _noise_calls += 1
        cfg.noise_q = Q
        cfg.noise_seed = (torch.initial_seed() * 0x9E3779B97F4A7C15 + _noise_calls * 0xD1B54A32D192ED03) & 0xFFFFFFFFFFFFFFFF
    outs = _FusedDecode.apply(cfg, pc._anchor_feat, pc.get_anchor, pc._offset, scaling_in, att[0], att[1], att[2],
                              app_vec, *params, *cam_in)
    xyz, color, opacity, scaling, rot, neural_opacity, mask = outs
    if is_training:
        return xyz, color, opacity, scaling, rot, neural_opacity, mask
    return xyz, color, opacity, scaling, rot
