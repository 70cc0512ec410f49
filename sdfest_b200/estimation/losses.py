"""Batched, sync-free restatements of the reference's caller-side loss helpers.

Reference: estimation/losses.py:32-135 (pc_loss), initialization/pointset_utils.py:34-89
(depth_to_pointcloud), initialization/quaternion_utils.py (scalar-last quaternions).
These stay on PyTorch: they are not the hot path (SURVEY.md section 8f ranks a fused kernel
for them as the next step after the renderer).
"""
from __future__ import annotations

import ctypes
from typing import Optional

import torch


def depth_to_pointcloud(depth_image: torch.Tensor, camera, mask=None) -> torch.Tensor:
    """Observed depth (H,W) -> points (N,3) in the OpenGL camera frame (x right, y up, z back).

    Uses the pixel-centre-0 principal point like the reference (pointset_utils.py:57).  Reading the
    number of points is a host sync; it runs once per observation, outside the loop.  fp32 CUDA tensors go
    through ``sdfr_depth_to_points`` (same points, same order, same bits as the torch expression on CUDA).
    """
    if depth_image.is_cuda and depth_image.dtype == torch.float32 and depth_image.dim() == 2:
        sel = None if mask is None else (depth_image * mask) != 0  # the torch expression's selection
        _, points, _ = extract_instances(depth_image[None], None if sel is None else sel[None], camera)
        return points[0]
    fx, fy, cx, cy, _ = camera.get_pinhole_camera_parameters(0.0)
    img = depth_image if mask is None else depth_image * mask
    rows, cols = torch.nonzero(img, as_tuple=True)
    z = depth_image[rows, cols]
    return torch.stack([(cols.float() - cx) * z / fx, -(rows.float() - cy) * z / fy, -z], dim=1)


def extract_instances(depth: torch.Tensor, masks: Optional[torch.Tensor], camera, far_field: Optional[float] = None,
                      capacity: int = 0):
    """The observations of K object instances in one pass of ``sdfr_depth_to_points``:
    ``(masked_depth (K,H,W), points (K,M,3), counts (K,) int64)``.

    ``depth`` (H,W) is shared by all instances, or (K,H,W) is one map each; ``masks`` (K,H,W) bool or None
    (every non-zero pixel).  The masked depth is 0 outside the mask and beyond ``far_field``, as
    ``SDFPipeline`` preprocesses a view; the caller's ``depth`` is not modified.  Row k of ``points`` holds
    instance k's cloud (``depth_to_pointcloud`` of its masked depth, bit for bit) followed by
    ``PAD_COORDINATE`` rows.  M = ``capacity``, or the largest count when ``capacity`` is 0; ``counts`` are
    the true counts even where they exceed ``capacity`` (only the first ``capacity`` points are kept).
    On CUDA (fp32) this is ``sdfr_depth_to_points``: with ``capacity`` > 0 nothing synchronises with the host;
    with 0, reading the largest count does, once.  CPU tensors take the torch statement of the same."""
    from .. import _lib
    from ..differentiable_renderer.sdf_renderer import _on_device_of, _stream

    if depth.is_cuda and depth.dtype != torch.float32:
        raise RuntimeError("extract_instances takes a float32 depth on CUDA")
    if depth.dim() not in (2, 3):
        raise ValueError(f"depth must be (H,W) or (K,H,W), got {tuple(depth.shape)}")
    H, W = int(depth.shape[-2]), int(depth.shape[-1])
    if masks is not None:
        if masks.dtype != torch.bool or masks.dim() != 3 or tuple(masks.shape[1:]) != (H, W) \
                or masks.device != depth.device:
            raise ValueError(f"masks must be a bool (K,{H},{W}) tensor on {depth.device}")
        masks = masks.contiguous()
    if depth.dim() == 2 and masks is None:
        raise ValueError("a shared depth image (H,W) needs masks (K,H,W)")
    K = int(masks.shape[0]) if masks is not None else int(depth.shape[0])
    if depth.dim() == 3 and int(depth.shape[0]) != K:
        raise ValueError(f"depth has {int(depth.shape[0])} maps for {K} masks")
    if capacity < 0:
        raise ValueError("capacity must be >= 0")
    depth = depth.contiguous()
    stride = 0 if depth.dim() == 2 else H * W
    far = float("inf") if far_field is None else float(far_field)
    if not depth.is_cuda:
        masked = depth if masks is None else torch.where(masks, depth, torch.zeros_like(depth))
        masked = torch.where(masked > far, torch.zeros_like(masked), masked)
        clouds = [depth_to_pointcloud(d, camera) for d in masked]
        counts = torch.tensor([int(c.shape[0]) for c in clouds], dtype=torch.int64)
        M = capacity or max([int(c.shape[0]) for c in clouds], default=0)
        points = torch.full((K, M, 3), PAD_COORDINATE, dtype=torch.float32)
        for k, c in enumerate(clouds):
            points[k, :min(int(c.shape[0]), M)] = c[:M]
        return masked.contiguous(), points, counts
    fx, fy, cx, cy, _ = camera.get_pinhole_camera_parameters(0.0)
    lib = _lib.lib()
    with _on_device_of(depth):
        dev = depth.device
        masked = torch.empty((K, H, W), dtype=torch.float32, device=dev)
        counts = torch.empty((K,), dtype=torch.int64, device=dev)
        n = ctypes.c_longlong(0)
        _lib.check(lib.sdfr_depth_to_points_scratch(K, W, H, ctypes.byref(n)), "sdfr_depth_to_points_scratch")
        scratch = torch.empty((max(n.value, 1),), dtype=torch.uint8, device=dev)

        def run(masked_out, points, cap):
            _lib.check(lib.sdfr_depth_to_points(
                depth.data_ptr(), stride, None if masks is None else masks.data_ptr(), K, W, H, far, fx, fy, cx, cy,
                None if masked_out is None else masked_out.data_ptr(), None if points is None else points.data_ptr(),
                cap, counts.data_ptr(), scratch.data_ptr(), _stream()), "sdfr_depth_to_points")

        if capacity:
            points = torch.empty((K, capacity, 3), dtype=torch.float32, device=dev)
            run(masked, points, capacity)
        else:
            run(masked, None, 0)  # the counts first: they size the clouds
            M = int(counts.max()) if K else 0
            points = torch.empty((K, M, 3), dtype=torch.float32, device=dev)
            if M:
                run(None, points, M)
    return masked, points, counts


def subsample_points(points: torch.Tensor, max_points: int) -> torch.Tensor:
    """At most ``max_points`` of the (N,3) points, a fixed random subset (seed 0); 0 = keep all."""
    if max_points and points.shape[0] > max_points:
        sel = torch.randperm(points.shape[0], device=points.device,
                             generator=torch.Generator(points.device).manual_seed(0))[:max_points]
        points = points[sel]
    return points.contiguous()


PAD_COORDINATE = 1.0e6  # metres: outside every SDF volume, contributes exactly 0 (losses.py:84-101)


def depth_to_pointclouds(depth_images: torch.Tensor, camera, max_points: int = 0):
    """Observed depth maps (K,H,W) of K object instances -> (points (K,M,3), counts (K,)).

    Instance k owns the first counts[k] points of row k (``depth_to_pointcloud`` + ``subsample_points``
    of its own map); the rest of the row is padding far outside any SDF volume, where the reference's
    ``pc_loss`` is exactly 0 (estimation/losses.py:84-101), so a mean over the instance's own points is
    ``sum / counts[k]``.  M = the largest count (at least 1).  Once per observation, outside the loop: fp32
    CUDA tensors take one ``extract_instances`` call (one host sync, a second with ``max_points`` for the
    per-instance sub-sampling), others one host sync per instance.
    """
    if depth_images.dim() != 3:
        raise RuntimeError(f"depth_images must be (K,H,W), got {tuple(depth_images.shape)}")
    if depth_images.is_cuda and depth_images.dtype == torch.float32:
        _, points, counts = extract_instances(depth_images, None, camera)
        if max_points and points.shape[1] > max_points:
            clouds = [points[k, :n] for k, n in enumerate(counts.tolist())]
        elif points.shape[1] == 0:
            return torch.full((points.shape[0], 1, 3), PAD_COORDINATE, dtype=torch.float32,
                              device=depth_images.device), counts
        else:
            return points, counts
    else:
        clouds = [depth_to_pointcloud(d, camera) for d in depth_images]
    clouds = [subsample_points(c, max_points) for c in clouds]
    counts = torch.tensor([c.shape[0] for c in clouds], dtype=torch.int64)
    M = max(int(counts.max()) if len(clouds) else 0, 1)
    out = torch.full((len(clouds), M, 3), PAD_COORDINATE, dtype=torch.float32, device=depth_images.device)
    for k, c in enumerate(clouds):
        out[k, : c.shape[0]] = c
    return out, counts.to(depth_images.device)


# --------------------------------------------------------------------------------------------
# CUDA path: the same loss as ONE kernel pair (sdfr_point_loss_forward / _backward)
# --------------------------------------------------------------------------------------------
class _PointLoss(torch.autograd.Function):
    """mean_m |pc_loss(points, ...)[b, m]| per hypothesis, on the GPU through the C ABI."""

    @staticmethod
    def forward(ctx, points, position, orientation, scale, sdf):
        from .. import _lib
        from ..differentiable_renderer.sdf_renderer import _check_input, _on_device_of, _stream

        for t, n in ((points, "points"), (position, "position"), (orientation, "orientation"),
                     (scale, "scale"), (sdf, "sdf")):
            _check_input(t, n)
        B = position.shape[0]
        if position.shape != (B, 3) or orientation.shape != (B, 4) or scale.numel() != B:
            raise RuntimeError("position (B,3), orientation (B,4), scale (B,) expected")
        if points.dim() == 2 and points.shape[1] == 3:
            M, pstride = points.shape[0], 0
        elif points.dim() == 3 and points.shape[0] == B and points.shape[2] == 3:
            M, pstride = points.shape[1], points.shape[1] * 3
        else:
            raise RuntimeError(f"points must be (M,3) or ({B},M,3), got {tuple(points.shape)}")
        R = sdf.shape[-1]
        if sdf.dim() != 4 or sdf.shape[0] not in (1, B) or not (sdf.shape[1] == sdf.shape[2] == R):
            raise RuntimeError(f"sdf must be (1|{B},R,R,R), got {tuple(sdf.shape)}")
        stride = 0 if sdf.shape[0] == 1 else R ** 3
        with _on_device_of(sdf):
            loss_sum = torch.empty(B, dtype=torch.float32, device=sdf.device)
            _lib.check(_lib.lib().sdfr_point_loss_forward(
                points.data_ptr(), pstride, M, sdf.data_ptr(), R, stride, _lib.LAYOUT_DENSE,
                position.data_ptr(), orientation.data_ptr(), scale.data_ptr(), B,
                loss_sum.data_ptr(), _lib.ZERO_GRADS, _stream()), "sdfr_point_loss_forward")
        ctx.save_for_backward(points, position, orientation, scale, sdf)
        ctx.meta = (B, M, pstride, R, stride)
        return loss_sum / max(M, 1)

    @staticmethod
    def backward(ctx, grad_loss):
        from .. import _lib
        from ..differentiable_renderer.sdf_renderer import _on_device_of, _ptr, _stream

        points, position, orientation, scale, sdf = ctx.saved_tensors
        B, M, pstride, R, stride = ctx.meta
        needs = ctx.needs_input_grad
        if needs[0]:
            raise RuntimeError("the point loss is not differentiable w.r.t. the observed points")
        flags = _lib.ZERO_GRADS
        for need, bit in zip(needs[1:], (_lib.GRAD_POSITION, _lib.GRAD_ORIENTATION,
                                         _lib.GRAD_INV_SCALE, _lib.GRAD_SDF)):
            if need:
                flags |= bit
        g_p = torch.empty_like(position) if needs[1] else None
        g_q = torch.empty_like(orientation) if needs[2] else None
        g_s = torch.empty_like(scale) if needs[3] else None
        g_sdf = torch.empty_like(sdf) if needs[4] else None
        if any(needs[1:]):
            upstream = (grad_loss.to(torch.float32) / max(M, 1)).contiguous()
            with _on_device_of(sdf):
                _lib.check(_lib.lib().sdfr_point_loss_backward(
                    points.data_ptr(), pstride, M, sdf.data_ptr(), R, stride, _lib.LAYOUT_DENSE,
                    position.data_ptr(), orientation.data_ptr(), scale.data_ptr(), B,
                    upstream.data_ptr(), _ptr(g_sdf), stride, _ptr(g_p), _ptr(g_q), _ptr(g_s), flags,
                    _stream()), "sdfr_point_loss_backward")
        return None, g_p, g_q, g_s, g_sdf


def point_loss(points: torch.Tensor, position: torch.Tensor, orientation: torch.Tensor,
               scale: torch.Tensor, sdf: torch.Tensor) -> torch.Tensor:
    """Per-hypothesis ``mean_m |pc_loss[b, m]|`` (estimation/simple_setup.py:134-144) through the fused
    kernels of ``libsdfrender.so`` (all observed points, no sub-sampling, no intermediate (B,M)
    tensors).  points (M,3) or (B,M,3); sdf (B|1,R,R,R).  CUDA tensors only: there is no CPU path in
    the product (the torch restatement of the reference's ``pc_loss`` lives in ``oracle/pc_loss.py`` as
    test infrastructure)."""
    if not points.is_cuda:
        raise RuntimeError("point_loss needs CUDA tensors: sdfest_b200 has no CPU fallback")
    return _PointLoss.apply(points.contiguous(), position.contiguous(), orientation.contiguous(),
                            scale.contiguous(), sdf.contiguous())
