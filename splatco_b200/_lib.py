"""ctypes binding of libsplatco_b200.so (C ABI in include/splatco_b200.h).

There is deliberately NO fallback: if the library is missing or a call fails, a RuntimeError is
raised (the reference surfaces C++ exceptions from its pybind module the same way, SURVEY.md §8b).
ctypes releases the GIL for the duration of each call, and the library keeps no thread-affine state,
so forward (main thread) and backward (autograd thread) can both call in.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsplatco_b200.so")
_lib = None

_vp, _i, _i64, _f, _sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t

# name -> (restype, argtypes); must list every symbol declared in include/splatco_b200.h
SIGNATURES = {
    "splatco_abi_version": (_i, []),
    "splatco_last_error": (C.c_char_p, []),
    "splatco_launch_count": (C.c_uint64, []),
    "splatco_geom_bytes": (_sz, [_i]),
    "splatco_binning_bytes": (_sz, [_i64]),
    "splatco_image_bytes": (_sz, [_i, _i]),
    "splatco_geom_layout": (_i, [_i, C.POINTER(_sz), _i]),
    "splatco_binning_layout": (_i, [_i64, C.POINTER(_sz), _i]),
    "splatco_image_layout": (_i, [_i, _i, C.POINTER(_sz), _i]),
    "splatco_sorted_buffer_index": (_i, [_i, _i]),
    "splatco_visible_filter": (_i, [_i, _vp, _vp, _i, _vp, _f, _vp, _vp, _f, _f, _i, _i, _vp, _vp]),
    "splatco_visible_compact_ws_bytes": (_sz, [_i]),
    "splatco_visible_compact_count_ptr": (_vp, [_vp, _i]),
    "splatco_visible_filter_compact": (_i, [_i, _vp, _vp, _i, _vp, _f, _vp, _vp, _f, _f, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "splatco_preprocess_fwd": (_i, [_i, _vp, _vp, _i, _vp, _vp, _vp, _f, _vp, _vp, _f, _f, _i, _i, _vp, _vp, _vp, _vp]),
    "splatco_preprocess_fwd_counted": (_i, [_i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _f, _vp, _vp, _f, _f, _i, _i, _vp, _vp, _vp, _vp]),
    "splatco_binning": (_i, [_i, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "splatco_binning_accepts_capacity": (_i, [_i, _i64, _i, _i]),
    "splatco_binning_radix": (_i, [_i, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "splatco_duplicate_with_keys": (_i, [_i, _i64, _i, _i, _vp, _vp, _vp, _vp]),
    "splatco_sort_pairs": (_i, [_i64, _i, _i, _vp, _vp]),
    "splatco_identify_tile_ranges": (_i, [_i64, _i, _i, _vp, _vp, _vp]),
    "splatco_blend_fwd": (_i, [_i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "splatco_blend_bwd": (_i, [_i, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "splatco_blend_fwd_upstream": (_i, [_i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "splatco_blend_bwd_upstream": (_i, [_i, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "splatco_blend_census": (_i, [_i64, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "splatco_preprocess_bwd": (_i, [_i, _vp, _vp, _i, _vp, _f, _vp, _vp, _f, _f, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "splatco_blend_fwd_depth_alpha": (_i, [_i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "splatco_blend_bwd_depth_alpha": (_i, [_i, _i64, _i, _i] + [_vp] * 13),
    "splatco_preprocess_bwd_depth": (_i, [_i, _vp, _vp, _i, _vp, _f, _vp, _vp, _f, _f, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "splatco_camera_grad_ws_bytes": (_sz, [_i]),
    "splatco_preprocess_bwd_camera": (_i, [_i, _vp, _vp, _i, _vp, _f, _vp, _vp, _f, _f, _i, _i] + [_vp] * 11),
    "splatco_preprocess_fwd_aa": (_i, [_i, _vp, _vp, _i, _vp, _vp, _vp, _f, _vp, _vp, _f, _f, _i, _i, _vp, _vp, _vp, _vp]),
    "splatco_preprocess_fwd_aa_counted": (_i, [_i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _f, _vp, _vp, _f, _f, _i, _i, _vp, _vp, _vp, _vp]),
    "splatco_preprocess_bwd_aa": (_i, [_i, _vp, _vp, _i, _vp, _f, _vp, _vp, _f, _f, _i, _i] + [_vp] * 13),
    # decode: descriptor / gradient structs are passed with ctypes.byref (see decode.py)
    "splatco_pack_planes": (_i, [_i, _i] + [_vp] * 7),
    "splatco_unpack_planes_add": (_i, [_i, _i] + [_vp] * 7),
    "splatco_decode_fwd_ws_bytes": (_sz, [_i, _i, _i]),
    "splatco_decode_bwd_ws_bytes": (_sz, [_i, _i, _i]),
    "splatco_decode_count_ptr": (_vp, [_vp, _i, _i, _i]),
    "splatco_decode_gathered_rows": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "splatco_blend_set_impl": (_i, [_i, _i]),
    "splatco_decode_set_impl": (_i, [_i]),
    "splatco_decode_profile": (_i, [_i]),
    "splatco_decode_profile_read": (_i, [_vp, _vp]),
    "splatco_decode_trace_read": (_i, [_vp]),
    "splatco_decode_get_impl": (_i, []),
    "splatco_decode_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "splatco_decode_emit": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "splatco_decode_bwd": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "splatco_decode_bwd_camera": (_i, [_vp, _vp, _vp, _i] + [_vp] * 10),
    "splatco_ta_fwd_ws_bytes": (_sz, [_i, _i]),
    "splatco_ta_bwd_ws_bytes": (_sz, [_i, _i]),
    "splatco_ta_fwd": (_i, [_i, _i, _i, _i] + [_vp] * 11),
    "splatco_ta_bwd": (_i, [_i, _i, _i, _i] + [_vp] * 18),
    "splatco_loss_ws_bytes": (_sz, [_i, _i, _i]),
    "splatco_l1_ssim_fwd": (_i, [_i, _i, _i, _vp, _vp, _f, _vp, _vp, _vp]),
    "splatco_l1_ssim_bwd": (_i, [_i, _i, _i, _vp, _vp, _f, _vp, _vp, _vp, _vp]),
    "splatco_scaling_reg_fwd": (_i, [_i, _vp, _vp, _vp, _vp]),
    "splatco_scaling_reg_bwd": (_i, [_i, _vp, _vp, _vp, _vp]),
    "splatco_mv_consistency_ws_bytes": (_sz, [_i]),
    "splatco_mv_consistency_fwd": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp]),
    "splatco_mv_consistency_bwd": (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "splatco_tv_add_grad": (_i, [_i, _i, _i, _vp, _vp, _f, _vp]),
    "splatco_grow_ws_bytes": (_sz, [_i64]),
    "splatco_grow_count": (_i, [_i64, _vp, _vp, _f, _vp, _vp, _f, _vp, _vp]),
    "splatco_grow_unique": (_i, [_i, _i, _i64, _vp, _vp, _vp, _i, _vp, _vp, _f, _vp, _vp, _f, _f, _i, _i64, _vp, _vp, _vp]),
    "splatco_grow_emit": (_i, [_i, _i, _f, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "splatco_cvpm_ws_bytes": (_sz, []),
    "splatco_cvpm_mask": (_i, [_i, _vp, _vp, _vp, _vp, _f, _f, _f, _f, _vp, _vp, _vp, _vp]),
    "splatco_adam_step": (_i, [_i, _vp, C.c_double, C.c_double, C.c_double, _vp]),
    "splatco_training_statis": (_i, [_i, _i] + [_vp] * 11),
    "splatco_tc_gemm_selftest": (_i, [_i, _i, _i, _vp, _vp, _vp, _i, _vp]),
    "splatco_tc_wgrad_selftest": (_i, [_i, _vp, _vp, _vp, _i, _vp]),
}


def lib():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m splatco_b200.build` "
                "(splatco_b200 has no CPU/PyTorch fallback)")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        if l.splatco_abi_version() != 1:
            raise RuntimeError("libsplatco_b200.so ABI version mismatch")
        _lib = l
    return _lib


def check(rc: int, what: str):
    if rc != 0:
        msg = lib().splatco_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (rc={rc}): {msg}")


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


# ---- cheap per-call plumbing (these run dozens of times per view; the torch.cuda wrappers cost ~10 us each) ----
import contextlib as _contextlib

import torch as _torch

_NULL = _contextlib.nullcontext()


def raw_stream(device) -> int:
    """cudaStream_t of torch's current stream on `device`, as an int."""
    idx = device.index
    if idx is None:
        idx = _torch.cuda.current_device()
    return _torch._C._cuda_getCurrentRawStream(idx)


def on_device(device):
    """Context that makes `device` current; a no-op object when it already is (the common case)."""
    idx = device.index
    if idx is None or idx == _torch.cuda.current_device():
        return _NULL
    return _torch.cuda.device(device)


# ---- size-bucketed allocations -------------------------------------------------------------------------------------
# V, M and R change a little from view to view and, once the optimizer moves the anchors, from iteration to iteration.
# torch's caching allocator only reuses a block for a request it fits, so workspaces sized to the exact byte keep
# missing the cache and fall through to cudaMalloc (milliseconds, and device-synchronising when it has to free first):
# measured as 25-45 ms outlier iterations in a training loop.  Sizes are therefore rounded up to 4 steps per octave
# (<= 25 % slack), which makes consecutive requests land on the same few block sizes.
# (4 steps per octave since round 2: with several GPUs in one process group every cudaMalloc also maps the new block into
# the peers' address spaces and costs 10-100 ms -- a stall all ranks then share through the gradient all-reduce)
BUCKET_BITS = int(os.environ.get("SPLATCO_BUCKET_BITS", "3"))      # 2^(BITS-1) size steps per octave


def bucket(n: int) -> int:
    if n <= 4096:
        return n
    step = 1 << (n.bit_length() - BUCKET_BITS)
    return (n + step - 1) // step * step


def empty_u8(nbytes: int, device):
    return _torch.empty(bucket(max(int(nbytes), 256)), dtype=_torch.uint8, device=device)


def empty_rows(rows: int, cols, dtype, device):
    """[rows, cols] (or [rows] when cols is None) as a prefix view of a bucketed allocation."""
    shape = (bucket(rows),) if cols is None else (bucket(rows), cols)
    return _torch.empty(shape, dtype=dtype, device=device)[:rows]
