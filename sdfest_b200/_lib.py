"""ctypes binding of libsdfrender.so -- the only native entry point of the package.

There is NO fallback: if the library is missing or a call fails, a RuntimeError is raised.
Signatures mirror include/sdfrender.h one to one.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_float, c_int, c_longlong, c_uint, c_void_p

# SDFR_LIB_PATH: load another build of the same ABI instead, e.g. a parent commit's, to compare
# two builds in one process (scripts/ab/)
LIB_PATH = os.environ.get("SDFR_LIB_PATH") or os.path.join(
    os.path.dirname(os.path.abspath(__file__)), "libsdfrender.so")

ABI_VERSION = 12

GRAD_SDF = 0x01
GRAD_POSITION = 0x02
GRAD_ORIENTATION = 0x04
GRAD_INV_SCALE = 0x08
GRAD_ALL = 0x0F
SDF_GRAD_EXACT = 0x10
ZERO_GRADS = 0x20
LOSS_WEIGHTED = 0x40  # sdfr_point_loss_fused: loss_sum += upstream[b] * sum
STEP_CLEAR_INPUTS = 0x100
STEP_NO_UPDATE = 0x200
TRACK_KEEP_VALID = 0x400  # sdfr_track_best: CLEAR_INPUTS zeroes n_inlier only
LAYOUT_DENSE = 0
LAYOUT_SKEWED = 1

_P = c_void_p
_CAM = [c_int, c_int, c_float, c_float, c_float, c_float]  # W, H, cx, cy, fx, fy
_POSE = [_P, _P, _P]  # position, orientation, inv_scale
_GRADS = [_P, c_longlong, _P, _P, _P]  # grad_sdf, grad_sdf_stride, g_pos, g_quat, g_inv_scale

SIGNATURES = {
    "sdfr_abi_version": (c_int, []),
    "sdfr_last_error": (ctypes.c_char_p, []),
    "sdfr_build_info": (ctypes.c_char_p, []),
    "sdfr_max_steps": (c_int, []),
    # the trailing (_P, _P) of the render entry points are (bounds or NULL, stream)
    "sdfr_grid_bounds": (c_int, [_P, c_int, c_longlong, c_int, _P, _P, c_int, c_float, _P, _P]),
    "sdfr_grid_slab_minima": (c_int, [_P, c_int, c_longlong, c_int, c_int, _P, _P]),
    "sdfr_bounds_from_minima": (c_int, [_P, c_int, c_int, _P, _P, c_int, c_float, _P, _P]),
    "sdfr_skew_grids_bounds": (c_int, [_P, c_int, c_longlong, c_int, _P, c_longlong, _P, _P, c_float, _P, _P]),
    "sdfr_forward": (c_int, [_P, c_int, c_longlong, c_int, *_POSE, c_int, *_CAM, c_float, _P, _P, _P]),
    "sdfr_forward_stats": (
        c_int, [_P, c_int, c_longlong, c_int, *_POSE, c_int, *_CAM, c_float, _P, _P, _P, _P]),
    "sdfr_backward": (
        c_int, [_P, _P, _P, c_int, c_longlong, c_int, *_POSE, c_int, *_CAM, *_GRADS, c_uint, _P, _P]),
    "sdfr_compare_forward": (
        c_int, [_P, c_int, c_longlong, c_int, *_POSE, c_int, *_CAM, c_float, _P, c_longlong, _P, _P, _P,
                c_uint, _P, _P]),
    "sdfr_compare_backward": (
        c_int, [_P, _P, c_longlong, _P, _P, _P, c_int, c_longlong, c_int, *_POSE, c_int, *_CAM, *_GRADS,
                c_uint, _P, _P]),
    "sdfr_compare_fused": (
        c_int, [_P, c_int, c_longlong, c_int, *_POSE, c_int, *_CAM, c_float, _P, c_longlong, _P, _P, _P,
                *_GRADS, c_uint, _P, _P]),
    "sdfr_compare_fused_inliers": (
        c_int, [_P, c_int, c_longlong, c_int, *_POSE, c_int, *_CAM, c_float, _P, c_longlong, _P, _P, _P,
                c_float, _P, *_GRADS, c_uint, _P, _P]),
    "sdfr_skewed_pitches": (c_int, [c_int, _P, _P, _P]),
    "sdfr_skew_grids": (c_int, [_P, c_int, c_longlong, c_int, _P, c_longlong, _P]),
    "sdfr_scale_grads": (c_int, [_P, _P, c_int, c_int, *_GRADS, c_uint, _P, c_longlong, _P]),
    "sdfr_point_loss_forward": (
        c_int, [_P, c_longlong, c_int, _P, c_int, c_longlong, c_int, *_POSE, c_int, _P, c_uint, _P]),
    "sdfr_point_loss_backward": (
        c_int, [_P, c_longlong, c_int, _P, c_int, c_longlong, c_int, *_POSE, c_int, _P, *_GRADS,
                c_uint, _P]),
    "sdfr_point_loss_fused": (
        c_int, [_P, c_longlong, c_int, _P, c_int, c_longlong, c_int, *_POSE, c_int, _P, _P, *_GRADS,
                c_uint, _P]),
    "sdfr_hypothesis_step": (
        c_int, [_P, _P, _P, _P, c_int, c_int, _P, _P, _P, _P, _P, c_float, _P, c_float, _P, _P, _P, _P,
                _P, _P, _P, _P, _P, ctypes.POINTER(c_float), c_float, c_float, c_float, _P, _P, _P, c_uint, _P]),
    "sdfr_view_poses": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, _P, _P, _P, _P]),
    "sdfr_views_pull_back": (
        c_int, [_P, _P, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P, c_float, _P, _P, _P, _P, _P, c_uint, _P]),
    "sdfr_point_constraint": (
        c_int, [_P, c_int, ctypes.POINTER(c_float), ctypes.POINTER(c_float), c_float, _P, _P, _P]),
    "sdfr_inlier_count": (
        c_int, [_P, _P, c_longlong, c_int, c_int, c_int, c_float, _P, _P, c_uint, _P]),
    "sdfr_track_best": (
        c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P, c_uint, _P]),
    "sdfr_decoder_tail_forward": (
        c_int, [_P, c_int, c_int, _P, _P, _P, c_int, c_int, _P, c_longlong, c_int, _P]),
    "sdfr_decoder_tail_forward_bounds": (
        c_int, [_P, c_int, c_int, _P, _P, _P, c_int, c_int, _P, c_longlong, c_int, _P, _P, c_float, _P, _P]),
    "sdfr_decoder_tail_backward": (
        c_int, [_P, c_longlong, _P, _P, _P, c_longlong, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "sdfr_upsample3d_forward": (c_int, [_P, c_int, c_int, c_int, _P, _P]),
    "sdfr_upsample3d_backward": (c_int, [_P, c_int, c_int, c_int, _P, _P]),
    "sdfr_conv3d_forward": (c_int, [_P, c_int, c_int, c_int, _P, _P, c_int, c_int, c_int, _P, _P]),
    "sdfr_conv3d_backward_data": (c_int, [_P, _P, c_int, c_int, c_int, _P, c_int, c_int, _P, _P]),
    "sdfr_depth_to_points_scratch": (c_int, [c_int, c_int, c_int, _P]),
    "sdfr_depth_to_points": (
        c_int, [_P, c_longlong, _P, c_int, c_int, c_int, c_float, c_float, c_float, c_float, c_float, _P, _P,
                c_int, _P, _P, _P]),
    "sdfr_forward_composite": (
        c_int, [_P, c_int, c_longlong, c_int, *_POSE, c_int, *_CAM, c_float, _P, _P, _P, _P]),
    "sdfr_backward_composite": (
        c_int, [_P, _P, _P, _P, c_int, c_longlong, c_int, *_POSE, c_int, *_CAM, *_GRADS, c_uint, _P]),
}

_lib = None


def lib() -> ctypes.CDLL:
    """Load (once) and return the native library; raises if it is not built."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m sdfest_b200.build` "
                "(needs nvcc; there is no CPU or PyTorch fallback for the renderer)")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the ABI lost a symbol
            fn.restype = restype
            fn.argtypes = argtypes
        got = handle.sdfr_abi_version()
        if got != ABI_VERSION:
            raise RuntimeError(f"libsdfrender ABI {got} != binding ABI {ABI_VERSION}; rebuild")
        _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().sdfr_last_error().decode(errors="replace")
        kind = "argument error" if rc < 0 else "CUDA error"
        raise RuntimeError(f"{what} failed ({kind} {rc}): {msg}")
