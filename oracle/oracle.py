"""numpy front-end of the CPU oracle (``liboracle.so``) -- TEST INFRASTRUCTURE ONLY.

All camera parameters are in the pixel-centre-0.5 convention the reference hands
to its kernels (``sdf_renderer.py:116-133, 310``).  ``dtype=np.float32`` mirrors the
reference CUDA kernels, ``np.float64`` the reference numpy renderer.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "liboracle.so")
_lib = None

POSE_KEYS = ("x", "y", "z", "qx", "qy", "qz", "qw", "s_inv")


def build(force: bool = False) -> str:
    """Compile liboracle.so with gcc (seconds)."""
    srcs = [os.path.join(_HERE, f) for f in ("sdf_oracle.c", "sdf_oracle_impl.h")]
    if force or not os.path.isfile(_SO) or any(
        os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs
    ):
        # the image exports CC=/opt/gcc/bin/gcc (a wrapper without libgomp): use the system gcc
        gcc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        base = [gcc, "-O2", "-ffp-contract=off", "-fPIC", "-shared", srcs[0], "-o", _SO, "-lm"]
        if subprocess.call(base + ["-fopenmp"], stderr=subprocess.DEVNULL) != 0:
            subprocess.check_call(base)  # no OpenMP runtime: single-threaded oracle
    return _SO


def _load():
    global _lib
    if _lib is None:
        build()
        _lib = ctypes.CDLL(_SO)
        for suf in ("f32", "f64"):
            getattr(_lib, f"oracle_render_{suf}").restype = ctypes.c_int
            getattr(_lib, f"oracle_backward_{suf}").restype = ctypes.c_int
    return _lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _suffix(dtype):
    dtype = np.dtype(dtype)
    if dtype == np.float32:
        return "f32"
    if dtype == np.float64:
        return "f64"
    raise ValueError("oracle dtype must be float32 or float64")


def _pose(position, orientation, inv_scale, dtype):
    p = np.ascontiguousarray(np.asarray(position, dtype=dtype).reshape(-1)[:3])
    q = np.ascontiguousarray(np.asarray(orientation, dtype=dtype).reshape(-1)[:4])
    s = np.ascontiguousarray(np.asarray(inv_scale, dtype=dtype).reshape(-1)[:1])
    return p, q, s


def _cam(cx, cy, fx, fy, dtype):
    # the CUDA launchers take cx,cy,fx,fy as C floats (sdf_renderer_cuda.cu:478-481)
    if np.dtype(dtype) == np.float32:
        cx, cy, fx, fy = (float(np.float32(v)) for v in (cx, cy, fx, fy))
    return [ctypes.c_double(float(v)) for v in (cx, cy, fx, fy)]


def render(sdf, position, orientation, inv_scale, width, height, cx, cy, fx, fy,
           threshold, dtype=np.float32, nthreads=1, max_steps=0, extras=False):
    """Depth image (H, W); with ``extras`` also per-pixel step counts and hit t."""
    lib = _load()
    dtype = np.dtype(dtype)
    suf = _suffix(dtype)
    sdf = np.ascontiguousarray(sdf, dtype=dtype)
    assert sdf.ndim == 3 and sdf.shape[0] == sdf.shape[1] == sdf.shape[2]
    p, q, s = _pose(position, orientation, inv_scale, dtype)
    depth = np.empty((height, width), dtype=dtype)
    steps = np.empty((height, width), dtype=np.int32) if extras else None
    t_hit = np.empty((height, width), dtype=dtype) if extras else None
    thr = float(np.float32(threshold)) if suf == "f32" else float(threshold)
    rc = getattr(lib, f"oracle_render_{suf}")(
        _ptr(sdf), ctypes.c_int(sdf.shape[0]), _ptr(p), _ptr(q), _ptr(s),
        ctypes.c_int(width), ctypes.c_int(height), *_cam(cx, cy, fx, fy, dtype),
        ctypes.c_double(thr), _ptr(depth), _ptr(steps), _ptr(t_hit),
        ctypes.c_int(max_steps), ctypes.c_int(nthreads))
    if rc != 0:
        raise RuntimeError(f"oracle_render_{suf} failed: {rc}")
    return (depth, steps, t_hit) if extras else depth


def render_backward(grad_depth, depth, sdf, position, orientation, inv_scale, width, height,
                    cx, cy, fx, fy, sdf_grad_mode="reference", dtype=np.float32, nthreads=1,
                    want_sdf=True, want_deriv=False):
    """Gradients of sum(grad_depth * depth) w.r.t. sdf, position, orientation, inv_scale.

    Returns a dict with float64 ``g_sdf`` (R,R,R) or None, ``g_position`` (3,),
    ``g_orientation`` (4, order x,y,z,w), ``g_inv_scale`` (scalar) and, with
    ``want_deriv``, ``deriv`` (8,H,W) in ``POSE_KEYS`` order.
    """
    lib = _load()
    dtype = np.dtype(dtype)
    suf = _suffix(dtype)
    sdf = np.ascontiguousarray(sdf, dtype=dtype)
    R = sdf.shape[0]
    depth = np.ascontiguousarray(depth, dtype=dtype)
    gd = None if grad_depth is None else np.ascontiguousarray(grad_depth, dtype=dtype)
    p, q, s = _pose(position, orientation, inv_scale, dtype)
    g_sdf = np.zeros((R, R, R), dtype=np.float64) if want_sdf else None
    g_pose = np.zeros(8, dtype=np.float64)
    deriv = np.empty((8, height, width), dtype=dtype) if want_deriv else None
    mode = {"reference": 0, "exact": 1}[sdf_grad_mode]
    rc = getattr(lib, f"oracle_backward_{suf}")(
        _ptr(gd), _ptr(depth), _ptr(sdf), ctypes.c_int(R), _ptr(p), _ptr(q), _ptr(s),
        ctypes.c_int(width), ctypes.c_int(height), *_cam(cx, cy, fx, fy, dtype),
        ctypes.c_int(mode), _ptr(g_sdf), _ptr(g_pose), _ptr(deriv), ctypes.c_int(nthreads))
    if rc != 0:
        raise RuntimeError(f"oracle_backward_{suf} failed: {rc}")
    return {
        "g_sdf": g_sdf,
        "g_position": g_pose[0:3].copy(),
        "g_orientation": g_pose[3:7].copy(),
        "g_inv_scale": float(g_pose[7]),
        "deriv": deriv,
    }


# ---------------------------------------------------------------------------------
# composition helpers (plain numpy; the reference has no counterpart for these --
# they state the semantics the batched / multi-object CUDA entry points must match)
# ---------------------------------------------------------------------------------
def composite_min_depth(depths):
    """Per-pixel minimum positive depth over K object layers (K,H,W).

    Returns (depth (H,W), winner (H,W) int32 with -1 where nothing was hit).  Ties go
    to the lowest object index.
    """
    depths = np.asarray(depths)
    big = np.where(depths > 0, depths, np.inf)
    winner = np.argmin(big, axis=0).astype(np.int32)
    best = np.take_along_axis(big, winner[None].astype(np.int64), axis=0)[0]
    hit = np.isfinite(best)
    return np.where(hit, best, 0).astype(depths.dtype), np.where(hit, winner, -1).astype(np.int32)


def render_composite(sdfs, positions, orientations, inv_scales, width, height, cx, cy, fx, fy,
                     threshold, dtype=np.float32, nthreads=1):
    layers = np.stack([
        render(sdfs[k], positions[k], orientations[k], inv_scales[k], width, height,
               cx, cy, fx, fy, threshold, dtype=dtype, nthreads=nthreads)
        for k in range(len(sdfs))])
    depth, winner = composite_min_depth(layers)
    return depth, winner


def render_composite_backward(grad_depth, depth, winner, sdfs, positions, orientations,
                              inv_scales, width, height, cx, cy, fx, fy,
                              sdf_grad_mode="reference", dtype=np.float32, nthreads=1,
                              want_deriv=False):
    """Per-object gradients of a min-depth composite: each pixel back-propagates to its winner."""
    out = []
    for k in range(len(sdfs)):
        dk = np.where(winner == k, depth, 0).astype(dtype)
        out.append(render_backward(grad_depth, dk, sdfs[k], positions[k], orientations[k],
                                   inv_scales[k], width, height, cx, cy, fx, fy,
                                   sdf_grad_mode=sdf_grad_mode, dtype=dtype, nthreads=nthreads,
                                   want_deriv=want_deriv))
    return out


def l1_depth_loss(depth_est, depth_obs):
    """Masked L1 depth loss of the reference pipeline (estimation/simple_setup.py:125-131).

    loss = mean |est - obs| over pixels with obs > 0 and est > 0; returns
    (loss, d loss / d est, n_overlap).  sign(0) = 0 as torch.abs' gradient.
    With no overlap the reference's mean over an empty selection is NaN; the oracle
    returns (0, zeros, 0) and callers must special-case it.
    """
    est = np.asarray(depth_est, dtype=np.float64)
    obs = np.asarray(depth_obs, dtype=np.float64)
    mask = (obs > 0) & (est > 0)
    n = int(mask.sum())
    if n == 0:
        return 0.0, np.zeros_like(est), 0
    diff = est - obs
    loss = float(np.abs(diff[mask]).sum() / n)
    grad = np.where(mask, np.sign(diff), 0.0) / n
    return loss, grad, n
