"""Batched render-and-compare: the loop body of SDFPipeline.__call__ for B hypotheses at once.

Reference: estimation/simple_setup.py:400-470 optimises ONE hypothesis with a Python loop of
decode -> render -> losses -> backward -> Adam, ~dozens of tiny kernels and two host syncs per
iteration.  Here B pose/scale(/latent) hypotheses advance together: one fused render-and-compare
launch pair (libsdfrender.so), batched torch ops for the caller-side pieces, no host
synchronisation inside the loop, and -- across GPUs -- hypotheses sharded per rank with one tiny
all_gather of the per-hypothesis losses (the reference has no distributed code at all).
"""
from __future__ import annotations

import ctypes
from typing import Callable, Optional

import torch
import torch.distributed as dist

from .. import _lib
from ..differentiable_renderer import Camera, render_and_compare
from ..differentiable_renderer.sdf_renderer import (_camera_params, _grid_operand, _ptr,
                                                    _skewed_elems, _stream)
from . import losses, views
from .decoder import FusedTailDecoder
from .fused import decode_render_compare


def shard_range(n_total: int, rank: int, world: int):
    """Contiguous shard [lo, hi) of n_total hypotheses owned by `rank` (remainder to low ranks)."""
    if world <= 0 or not (0 <= rank < world):
        raise ValueError("bad rank/world")
    q, r = divmod(n_total, world)
    lo = rank * q + min(rank, r)
    return lo, lo + q + (1 if rank < r else 0)


def exchange_shard_sizes(n_local: int, device, group=None):
    """Every rank's shard size (one small all_gather and a host read: do it once, not per step)."""
    world = dist.get_world_size(group)
    mine = torch.tensor([n_local], device=device)
    everyone = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(everyone, mine, group=group)
    return [int(s.item()) for s in everyone]


def gather_losses(local: torch.Tensor, group=None, sizes=None) -> torch.Tensor:
    """All ranks' per-hypothesis losses, concatenated in rank order (equal shard sizes use
    all_gather_into_tensor -- NCCL over NVLink on GPUs, gloo on CPU in the tests).  ``sizes``: the
    shard sizes of all ranks when the caller already knows them (``shard_range`` /
    ``exchange_shard_sizes``); without it they are exchanged first, which costs a second
    collective and a host synchronisation per call (0.37 ms per iteration in the 8-GPU sweep)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return local
    world = dist.get_world_size(group)
    if sizes is None:
        sizes = exchange_shard_sizes(local.numel(), local.device, group)
    elif len(sizes) != world or sizes[dist.get_rank(group)] != local.numel():
        raise ValueError("sizes must list every rank's shard size, this rank's included")
    if len(set(sizes)) == 1:
        out = local.new_empty(world * local.numel())
        dist.all_gather_into_tensor(out, local.contiguous(), group=group)
        return out
    pad = max(sizes)
    buf = local.new_zeros(pad)
    buf[: local.numel()] = local
    out = [local.new_empty(pad) for _ in range(world)]
    dist.all_gather(out, buf, group=group)
    return torch.cat([o[:n] for o, n in zip(out, sizes)])


def global_best(local_losses: torch.Tensor, lo: int, group=None):
    """(global index, loss) of the best hypothesis over all ranks; NaN losses never win."""
    all_losses = gather_losses(torch.nan_to_num(local_losses, nan=float("inf")), group)
    idx = int(torch.argmin(all_losses).item())
    return idx, float(all_losses[idx].item())


class HypothesisOptimizer:
    """Adam on B hypotheses of (position, orientation, scale[, latent]) against one observation.

    Learning rates and loss weights default to the reference's (simple_setup.py:400-405,
    estimation/configs/default.yaml:14-16).  ``decoder`` maps latents (B,L) to grids
    (B,1,R,R,R) (e.g. ``SDFVAE.decode``); without it ``sdf`` holds fixed grids (B|1,R,R,R).

    Object instances: ``depth_obs`` (H,W) is one observation shared by all hypotheses; (K,H,W) with
    ``instance`` (B,) compares hypothesis b with the depth map *and the observed points* of instance
    ``instance[b]`` (default ``arange(B)``: one map per hypothesis), each instance's point loss
    averaged over its own points -- the reference's loop run for K objects x B/K hypotheses at once.

    Views: with ``camera_positions`` (V,3) and ``camera_orientations`` (V,4) (camera-to-world, as
    SDFPipeline.__call__ takes them) ``depth_obs`` is (V,H,W), one image per view of the SAME object;
    the pose is optimised in the world frame, moved into every camera frame (``estimation/views.py``,
    simple_setup.py:423-431) and the per-view losses are summed (:432-446); the inlier ratio is
    evaluated on the last view, as the reference's loop variables leave it (:463).  On the fused path
    the rigid maps and their adjoint are two tiny kernels (``sdfr_view_poses``,
    ``sdfr_views_pull_back``) around V batched render / compare / point-loss launches that accumulate
    the normalised SDF gradients of all views into ONE gradient grid per hypothesis.

    ``point_constraint`` = (source (3,), target (3,), weight) adds ``weight * |R(orientation) source -
    target|`` on the un-normalised orientation (simple_setup.py:164-175, losses.py:138-153):
    ``sdfr_point_constraint`` on the fused path.

    Result selection: with ``inlier_threshold`` (the reference's ``relative_inlier_threshold``, 0.03)
    every iteration also evaluates the inlier ratio of simple_setup.py:177-188 -- on the depth rendered
    before the update, as :463 does -- into ``inlier_ratio`` (B,) and keeps the parameters after the
    update with the best ratio so far in ``best_position / best_orientation / best_scale /
    best_latent`` (``best_inlier_ratio``, ``best_iteration``): ``result("best_inlier_ratio")``.
    The reference keeps references to the live tensors there (:207-210), so what it returns is always
    the last iterate (``result("last_iteration")``); the copies are what the code evidently intends.

    Serving many observations with ONE captured graph: ``point_capacity`` (fused path; a shared observation,
    views or object instances) stores each observed cloud in a buffer of that fixed size (padding outside every volume,
    where the point loss is exactly 0; the mean is taken over the true count), so that ``reset(...)`` can load
    the next observation and initial estimate into the same device buffers and ``step()`` keeps replaying
    the graph captured for the first one (``SDFPipeline`` does this).

    ``optimizer``: ``"fused"`` runs the whole iteration as direct C-ABI launches -- decoder tail,
    ``sdfr_compare_fused``, ``sdfr_point_loss_fused``, tail adjoint, and ONE
    ``sdfr_hypothesis_step`` kernel for the gradient chain rule, Adam on all four groups, the
    quaternion renormalisation and the loss (autograd only carries the tail's gradient through the
    decoder trunk); ``"torch"`` composes the package's autograd operators with
    ``torch.optim.Adam`` (~60 more 1-2 us launches per iteration).  ``"auto"`` (default) picks
    ``"fused"`` for CUDA tensors with fixed grids or a ``FusedTailDecoder``.
    """

    def __init__(self, camera: Camera, threshold: float, depth_obs: torch.Tensor,
                 position: torch.Tensor, orientation: torch.Tensor, scale: torch.Tensor,
                 sdf: Optional[torch.Tensor] = None, latent: Optional[torch.Tensor] = None,
                 decoder: Optional[Callable] = None, depth_weight: float = 1.0,
                 pc_weight: float = 3.0, max_points: int = 0, group=None, optimizer: str = "auto",
                 lrs=(1e-3, 1e-2, 1e-3, 1e-2), betas=(0.9, 0.999), eps: float = 1e-8,
                 overlap: bool = True, instance: Optional[torch.Tensor] = None,
                 inlier_threshold: Optional[float] = None,
                 camera_positions: Optional[torch.Tensor] = None,
                 camera_orientations: Optional[torch.Tensor] = None,
                 point_constraint=None, point_capacity: int = 0):
        if (decoder is None) == (sdf is None):
            raise ValueError("give either fixed `sdf` grids or a `decoder` with `latent`")
        if optimizer not in ("auto", "fused", "torch"):
            raise ValueError("optimizer must be 'auto', 'fused' or 'torch'")
        if (camera_positions is None) != (camera_orientations is None):
            raise ValueError("give camera_positions and camera_orientations together")
        multiview = camera_positions is not None
        can_fuse = position.is_cuda and (decoder is None or isinstance(decoder, FusedTailDecoder)) \
            and (latent is None or int(latent.shape[1]) <= 64)  # sdfr_hypothesis_step: kStepMaxLatent
        # (source (3,), target (3,), weight): simple_setup.py:164-175, 224, 299
        self.point_constraint = None
        if point_constraint is not None:
            source, target, weight = point_constraint
            self.point_constraint = (torch.as_tensor(source, dtype=torch.float32, device=position.device),
                                     torch.as_tensor(target, dtype=torch.float32, device=position.device),
                                     float(weight))
        if optimizer == "fused" and not can_fuse:
            raise ValueError("optimizer='fused' needs CUDA tensors and fixed grids or a FusedTailDecoder "
                             "(latent size <= 64)")
        self.optimizer_impl = "fused" if (optimizer != "torch" and can_fuse) else "torch"
        self.overlap = bool(overlap)
        # corner weights of the SDF gradient (SURVEY Q2): the module default at construction time
        from ..differentiable_renderer.sdf_renderer import get_sdf_grad_mode
        self.sdf_grad_mode = get_sdf_grad_mode()
        self.lrs, self.betas, self.eps = tuple(float(x) for x in lrs), tuple(betas), float(eps)
        self.camera, self.threshold, self.group = camera, float(threshold), group
        self.depth_weight, self.pc_weight = depth_weight, pc_weight
        self.position = position.detach().clone().requires_grad_(True)
        self.orientation = orientation.detach().clone().requires_grad_(True)
        self.scale = scale.detach().clone().requires_grad_(True)
        self.decoder, self.sdf = decoder, sdf
        groups = [{"params": [self.position], "lr": self.lrs[0]},
                  {"params": [self.orientation], "lr": self.lrs[1]},
                  {"params": [self.scale], "lr": self.lrs[2]}]
        self.latent = None
        if decoder is not None:
            self.latent = latent.detach().clone().requires_grad_(True)
            groups.append({"params": [self.latent], "lr": self.lrs[3]})
        self.optimizer = None
        if self.optimizer_impl == "torch":
            self.optimizer = torch.optim.Adam(groups, betas=self.betas, eps=self.eps,
                                              capturable=self.position.is_cuda)
        B = self.position.shape[0]
        self.point_capacity, self.max_points = int(point_capacity), int(max_points)
        if point_capacity and self.optimizer_impl != "fused":
            raise ValueError("point_capacity needs the fused path")
        self.last_losses = None
        self.inlier_threshold = None if inlier_threshold is None else float(inlier_threshold)
        if self.inlier_threshold is not None:
            dev0 = self.position.device
            self._inl = torch.zeros(2, B, dtype=torch.float32, device=dev0)  # n_inlier, n_valid
            self.inlier_ratio = torch.zeros(B, dtype=torch.float32, device=dev0)
            self.best_inlier_ratio = torch.full((B,), -1.0, dtype=torch.float32, device=dev0)
            self.best_iteration = torch.full((B,), -1, dtype=torch.int32, device=dev0)
            self.best_position = self.position.detach().clone()
            self.best_orientation = self.orientation.detach().clone()
            self.best_scale = self.scale.detach().clone()
            self.best_latent = None if self.latent is None else self.latent.detach().clone()
            self._iteration = torch.zeros(B, dtype=torch.int32, device=dev0)  # optimizer="torch" (device-side: survives graph replay)
        # valid pixels depend on the observation alone (simple_setup.py:186): counted once where the fused iteration
        # counts inliers only (thresholds <= 1, no views); else sdfr_inlier_count recounts both every iteration
        self._valid_once = self.optimizer_impl == "fused" and self.inlier_threshold is not None \
            and self.inlier_threshold <= 1.0 and not multiview
        self.depth_obs = self._views = self.instance = self._n_points = None
        self.point_counts = None  # (B,) points hypothesis b owns, when the clouds differ
        self._set_observation(depth_obs, camera_positions, camera_orientations, instance)
        self._graph = None
        self._shard_sizes = None  # exchanged on the first gather of run()
        if self.optimizer_impl == "fused":
            with torch.cuda.device(self.position.device):
                self._init_fused()

    def _set_observation(self, depth_obs: torch.Tensor, camera_positions: Optional[torch.Tensor] = None,
                         camera_orientations: Optional[torch.Tensor] = None,
                         instance: Optional[torch.Tensor] = None) -> None:
        """The observation into the buffers every iteration reads: depth images and camera poses, each view's
        observed points (one shared observation is one view), sub-sampled once -- the only host syncs --, the
        weight pc_weight / (true number of points) per hypothesis in device memory, and the valid pixels where
        they are counted once.  Construction allocates the buffers (private copies: never the caller's tensors);
        reset() overwrites them in place, so a captured graph keeps reading them, and raises before it writes any.

        Object instances: ``depth_obs`` (K,H,W) and ``instance`` (B,): hypothesis b is compared with the depth map and
        the points of instance[b] (default: one map per hypothesis); K and the mapping are fixed at construction."""
        B, cap, first = int(self.position.shape[0]), self.point_capacity, self.depth_obs is None
        views = camera_positions is not None or self._views is not None
        if not first:
            instance = self.instance
        if first:
            if views:
                if instance is not None:
                    raise ValueError("views and object instances cannot be combined")
                V = int(camera_positions.shape[0])
                if tuple(camera_positions.shape) != (V, 3) or tuple(camera_orientations.shape) != (V, 4) \
                        or depth_obs.dim() != 3 or depth_obs.shape[0] != V:
                    raise ValueError("camera_positions (V,3), camera_orientations (V,4) and depth_obs (V,H,W) expected")
            elif depth_obs.dim() == 2:
                if instance is not None:
                    raise ValueError("`instance` needs one observed depth map per object instance (K,H,W)")
            else:
                if instance is None:
                    instance = torch.arange(B, device=depth_obs.device)
                instance = instance.to(device=depth_obs.device, dtype=torch.int64)
                if instance.shape != (B,) or depth_obs.dim() != 3:
                    raise ValueError("depth_obs (K,H,W) and instance (B,) expected")
                if int(instance.min()) < 0 or int(instance.max()) >= depth_obs.shape[0]:
                    raise ValueError("instance index out of range")
            W, H = int(self.camera.width), int(self.camera.height)
            if self.optimizer_impl == "fused" and tuple(depth_obs.shape[-2:]) != (H, W):
                raise RuntimeError(f"depth_obs must have shape (V,{H},{W})" if views
                                   else f"depth_obs must have shape ({H},{W}) or ({B},{H},{W})")
        else:
            shape = tuple(self.depth_obs.shape) if instance is None else (self._n_instances, *self.depth_obs.shape[1:])
            if tuple(depth_obs.shape) != shape:
                raise ValueError(f"depth_obs must keep its shape {shape}")
            if self.pc_weight and not cap:
                raise RuntimeError("a new observation needs point_capacity (the cloud sizes are baked in)")
        if instance is not None:
            clouds, counts = losses.depth_to_pointclouds(depth_obs, self.camera, self.max_points)
            if cap and int(counts.max()) > cap:
                raise ValueError(f"{int(counts.max())} observed points exceed point_capacity {cap}")
            # hypothesis b weighs its own points with pc_weight / counts[b]
            n = counts.index_select(0, instance).to(torch.float32)
            up_p = torch.where(n > 0, self.pc_weight / n.clamp(min=1.0), torch.zeros_like(n))
            if first:
                self.instance, self._n_instances = instance, int(depth_obs.shape[0])
                self.depth_obs = depth_obs.index_select(0, instance).contiguous()
                self.point_counts = counts.index_select(0, instance)
                self._up_p = up_p.contiguous()
                # with point_capacity: fixed-size clouds, padded outside every volume (point loss exactly 0 there)
                self.points = clouds.index_select(0, instance).contiguous() if not cap else \
                    torch.empty((B, cap, 3), dtype=torch.float32, device=clouds.device)
            else:
                self.depth_obs.copy_(depth_obs.index_select(0, instance))
                self.point_counts.copy_(counts.index_select(0, instance))
                self._up_p.copy_(up_p)
            if cap:
                self.points.fill_(losses.PAD_COORDINATE)
                self.points[:, :clouds.shape[1]].copy_(clouds.index_select(0, instance))
        else:
            V = int(depth_obs.shape[0]) if views else 1
            poses = [None if p is None else p.detach().reshape(V, k)
                     for p, k in ((camera_positions, 3), (camera_orientations, 4))]
            clouds = []
            if first or self.pc_weight:
                clouds = [losses.subsample_points(losses.depth_to_pointcloud(d, self.camera), self.max_points)
                          for d in (depth_obs if views else depth_obs[None])]
            for c in clouds:
                if cap and int(c.shape[0]) > cap:
                    raise ValueError(f"{int(c.shape[0])} observed points exceed point_capacity {cap}")
            if first:
                dev = self.position.device
                self.depth_obs = torch.empty_like(depth_obs, memory_format=torch.contiguous_format)
                # with point_capacity: fixed-size clouds, padded outside every volume (point loss exactly 0 there)
                self._view_points = [torch.empty((cap, 3), dtype=torch.float32, device=c.device) if cap else c
                                     for c in clouds]
                self._view_counts = [0] * V
                self._view_up_p = [torch.empty((B,), dtype=torch.float32, device=dev) for _ in range(V)]
                self.points = self._view_points[0]
                if views:
                    self._views = tuple(torch.empty((V, k), dtype=torch.float32, device=depth_obs.device)
                                        for k in (3, 4))
                else:
                    self._up_p = self._view_up_p[0]
            self.depth_obs.copy_(depth_obs)
            for v, c in enumerate(clouds):
                n = int(c.shape[0])
                if cap:
                    self._view_points[v].fill_(losses.PAD_COORDINATE)
                    self._view_points[v][:n].copy_(c)
                self._view_counts[v] = n
                self._view_up_p[v].fill_(self.pc_weight / n if n else 0.0)
            if not views:
                self._n_points = self._view_counts[0]  # true number of points of the shared cloud
            for buf, p in zip(self._views or (), poses):
                if p is not None:
                    buf.copy_(p)
        if self._valid_once:
            self._inl[1].copy_((self.depth_obs != 0).flatten(-2).sum(-1))

    def reset(self, position: torch.Tensor, orientation: torch.Tensor, scale: torch.Tensor,
              latent: Optional[torch.Tensor] = None, depth_obs: Optional[torch.Tensor] = None,
              camera_positions: Optional[torch.Tensor] = None,
              camera_orientations: Optional[torch.Tensor] = None) -> None:
        """Start over from a new initial estimate -- and, with ``depth_obs``, a new observation -- in the SAME
        device buffers: optimiser state, result selection and losses are cleared, and a captured graph stays
        valid (``step()`` keeps replaying it).  Fused path only; a new observation needs ``point_capacity``
        (or ``pc_weight`` 0).  With views: ``depth_obs`` (V,H,W) and, optionally, new camera poses.  With object
        instances: ``depth_obs`` (K,H,W), the same K and ``instance`` mapping as at construction.  The point
        constraint, if any, stays the one given at construction.  Raises ValueError when a new cloud does not
        fit the capacity."""
        if self.optimizer_impl != "fused":
            raise RuntimeError("reset() is for optimizer='fused'")
        if not self._V and (camera_positions is not None or camera_orientations is not None):
            raise ValueError("camera poses can only be reset on an optimiser constructed with views")
        if self.latent is not None and latent is None:
            raise ValueError("latent expected")
        with torch.no_grad(), torch.cuda.device(self.position.device):
            if depth_obs is not None or camera_positions is not None or camera_orientations is not None:
                # new camera poses alone: the clouds are reloaded from the current observation
                self._set_observation(self.depth_obs if depth_obs is None else depth_obs, camera_positions,
                                      camera_orientations)
            self.position.copy_(position.reshape(self.position.shape))
            self.orientation.copy_(orientation.reshape(self.orientation.shape))
            self.scale.copy_(scale.reshape(self.scale.shape))
            if self.latent is not None:
                self.latent.copy_(latent.reshape(self.latent.shape))
            for t in (self._m, self._v, self._t, self._small, self._loss):
                t.zero_()
            if self._g_raw is not None:
                self._g_raw.zero_()
                self._loss_extra.zero_()
            if self.inlier_threshold is not None:
                self._inl[0].zero_()
                if not self._valid_once:  # else: the valid pixels of the observation, counted by _set_observation
                    self._inl[1].zero_()
                self.inlier_ratio.zero_()
                self.best_inlier_ratio.fill_(-1.0)
                self.best_iteration.fill_(-1)
                self._iteration.zero_()
            self._hyp_step(_lib.STEP_NO_UPDATE)  # unit quaternions and 1/scale of the new estimate
        self.last_losses = None

    # ------------------------------------------------------------------------------------
    # optimizer="fused": one iteration = a handful of C-ABI launches, no autograd outside the trunk
    # ------------------------------------------------------------------------------------
    def _init_fused(self) -> None:
        B, dev = self.position.shape[0], self.position.device
        for t, shape in ((self.position, (B, 3)), (self.orientation, (B, 4))):
            if tuple(t.shape) != shape:
                raise RuntimeError(f"position (B,3) and orientation (B,4) expected, got {tuple(t.shape)}")
        if self.scale.numel() != B:
            raise RuntimeError("scale must have one element per hypothesis")
        for t in (self.position, self.orientation, self.scale):
            t.requires_grad_(False)  # updated in place by sdfr_hypothesis_step
        L = 0 if self.latent is None else int(self.latent.shape[1])
        self._L = L
        W, H = int(self.camera.width), int(self.camera.height)
        V = 0 if self._views is None else int(self.depth_obs.shape[0])
        self._V = V
        self._obs_stride = 0 if self.point_counts is None else H * W  # (B,H,W): one image per hypothesis
        # every small per-hypothesis buffer in one allocation: consumed AND cleared by the step kernel
        # (with views: [V,B,...] each, consumed and cleared by sdfr_views_pull_back)
        NB = max(V, 1) * B
        small = torch.zeros(20 * NB, dtype=torch.float32, device=dev)
        cuts = (("loss_sum", 1), ("n_overlap", 1), ("gr_p", 3), ("gr_q", 4), ("gr_is", 1),
                ("pl", 1), ("g2_p", 3), ("g2_q", 4), ("g2_s", 1))
        off, self._buf = 0, {}
        for name, k in cuts:
            self._buf[name] = small[off:off + k * NB]
            off += k * NB
        self._small = small
        # gradient w.r.t. the un-normalised orientation and a loss term taken as is: the point constraint
        # and (loss only) the view loop's sum; consumed and cleared by the step kernel
        self._g_raw = self._loss_extra = None
        if self.point_constraint is not None or V:
            extra = torch.zeros(5 * B, dtype=torch.float32, device=dev)
            self._g_raw, self._loss_extra = extra[:4 * B], extra[4 * B:]
        if self.point_constraint is not None:
            src, tgt, _ = self.point_constraint
            self._pc_src = (ctypes.c_float * 3)(*[float(x) for x in src.tolist()])
            self._pc_tgt = (ctypes.c_float * 3)(*[float(x) for x in tgt.tolist()])
        self._unit_q = torch.empty((B, 4), dtype=torch.float32, device=dev)
        self._inv_scale = torch.empty((B,), dtype=torch.float32, device=dev)
        self._loss = torch.zeros((B,), dtype=torch.float32, device=dev)
        self._m = torch.zeros((B, 8 + L), dtype=torch.float32, device=dev)
        self._v = torch.zeros((B, 8 + L), dtype=torch.float32, device=dev)
        self._t = torch.zeros((B,), dtype=torch.int32, device=dev)
        self._lr = (ctypes.c_float * 4)(*self.lrs)
        self._depth = torch.empty((B, H, W), dtype=torch.float32, device=dev)
        M = int(self.points.shape[-2]) if self.pc_weight else 0
        if V:
            # per view: camera-frame poses, the pulled-back gradients, and each view's own cloud weighted
            # with pc_weight / (its number of points) in the loss and the gradients
            M = 0  # the single-view point buffers of the step kernel stay unused
            self._pose_c = (torch.empty((V, B, 3), dtype=torch.float32, device=dev),
                            torch.empty((V, B, 4), dtype=torch.float32, device=dev),
                            torch.empty((V, B), dtype=torch.float32, device=dev))
            pb = torch.zeros(8 * B, dtype=torch.float32, device=dev)
            self._pb = (pb[:3 * B], pb[3 * B:7 * B], pb[7 * B:])
            self._view_M = [int(p.shape[0]) if self.pc_weight else 0 for p in self._view_points]
        self._M = M
        # fixed-size and per-instance clouds: the weight pc_weight / (true count) lives in device memory (_up_p:
        # upstream and, with SDFR_LOSS_WEIGHTED, the loss), so reset() can change it under a captured graph;
        # a plain shared cloud passes it to the step kernel as a scalar
        weighted = bool(self.point_capacity) or self.point_counts is not None
        self._point_flags = _lib.LOSS_WEIGHTED if weighted else 0
        self._point_weight = 1.0 if weighted else ((self.pc_weight / M) if M else 0.0)
        self._points_stride = 0 if self.point_counts is None else 3 * M
        self._up_d = torch.full((B,), float(self.depth_weight), dtype=torch.float32, device=dev)
        if self.decoder is None:
            sdf = self.sdf.contiguous()
            R = int(sdf.shape[-1])
            stride = 0 if sdf.shape[0] == 1 else R ** 3
            self._R = R
            self._grid_op = _grid_operand(sdf, R, stride, B, W * H)  # (tensor, stride, layout), made once
            self._g_sdf = self._g_sdf_pc = None
        else:
            R = int(self.decoder.volume_size)
            self._R = R
            SK = _skewed_elems(R)
            self._grid_op = (torch.empty((B, SK), dtype=torch.float32, device=dev), SK, _lib.LAYOUT_SKEWED)
            # both gradient grids in one allocation: one clear per iteration
            # (views: the normalised gradients of every view and cloud accumulate into the first one)
            self._g_both = torch.empty((2 if M else 1, B, R ** 3), dtype=torch.float32, device=dev)
            self._g_sdf = self._g_both[0]
            self._g_sdf_pc = self._g_both[1] if M else None
        from ..differentiable_renderer.sdf_renderer import get_empty_space_policy
        n_grids = 1 if self._grid_op[1] == 0 else B
        self._bounds = None if get_empty_space_policy() == "off" else \
            torch.empty((max(V, 1), n_grids, 8), dtype=torch.int32, device=dev)
        # fixed grids: their slab minima are read once; every iteration's bounds (they depend on the
        # pose through the hit-threshold bound) are then 3 R comparisons per grid instead of a grid scan
        self._minima = None
        if self._bounds is not None and self.decoder is None:
            grids, gstride, layout = self._grid_op
            self._minima = torch.empty((n_grids, 3, R), dtype=torch.float32, device=dev)
            _lib.check(_lib.lib().sdfr_grid_slab_minima(grids.data_ptr(), R, gstride, layout, n_grids,
                                                        self._minima.data_ptr(), _stream()), "sdfr_grid_slab_minima")
        # second stream: the point loss runs beside the render (both only read the grids), the
        # gradient-grid clears beside the decoder trunk; forks and joins are captured by capture()
        self._side = torch.cuda.Stream(dev) if self.overlap else None
        self._hyp_step(_lib.STEP_NO_UPDATE)  # unit quaternions and 1/scale for the first render

    def _grid_bounds(self, position_ptr: int, inv_scale_ptr: int, out: torch.Tensor) -> int:
        """Empty-space bounds of this iteration's grids for the given poses into ``out``; its pointer."""
        lib, B = _lib.lib(), self.position.shape[0]
        grids, gstride, layout = self._grid_op
        if self._minima is not None:
            _lib.check(lib.sdfr_bounds_from_minima(
                self._minima.data_ptr(), self._R, int(self._minima.shape[0]), position_ptr, inv_scale_ptr, B,
                self.threshold, out.data_ptr(), _stream()), "sdfr_bounds_from_minima")
        else:
            _lib.check(lib.sdfr_grid_bounds(grids.data_ptr(), self._R, gstride, layout, position_ptr, inv_scale_ptr,
                                            B, self.threshold, out.data_ptr(), _stream()), "sdfr_grid_bounds")
        return out.data_ptr()

    def _hyp_step(self, flags: int, g_latent: Optional[torch.Tensor] = None,
                  g_orientation_raw: Optional[torch.Tensor] = None,
                  loss_extra: Optional[torch.Tensor] = None) -> None:
        b, B = self._buf, self.position.shape[0]
        M = self._M
        if self._V:
            # the per-view sums were folded into (g_position, g_orientation, g_scale, loss_extra) by
            # sdfr_views_pull_back: they enter as the already weighted second gradient set
            raw = (None,) * 5
            g2 = tuple(t.data_ptr() for t in self._pb)
            pl = None
        else:
            raw = (b["loss_sum"].data_ptr(), b["n_overlap"].data_ptr(), b["gr_p"].data_ptr(),
                   b["gr_q"].data_ptr(), b["gr_is"].data_ptr())
            g2 = (b["g2_p"].data_ptr(), b["g2_q"].data_ptr(), b["g2_s"].data_ptr()) if M else (None,) * 3
            pl = b["pl"].data_ptr() if M else None
        _lib.check(_lib.lib().sdfr_hypothesis_step(
            self.position.data_ptr(), self.orientation.data_ptr(), self.scale.data_ptr(),
            _ptr(self.latent), self._L, B, *raw, float(self.depth_weight),
            pl, self._point_weight, *g2, _ptr(g_latent), _ptr(g_orientation_raw), _ptr(loss_extra),
            self._m.data_ptr(),
            self._v.data_ptr(), self._t.data_ptr(), self._lr, self.betas[0], self.betas[1], self.eps,
            self._unit_q.data_ptr(), self._inv_scale.data_ptr(), self._loss.data_ptr(), flags,
            _stream()), "sdfr_hypothesis_step")

    def _latent_leaf(self) -> torch.Tensor:
        """A FRESH autograd leaf over the latent's storage for this iteration's trunk graph.  Autograd caches a
        leaf's AccumulateGrad node together with the stream it was created on; a node left over from an eager
        iteration on the default stream (kept alive by a not-yet-collected graph) makes the engine synchronise
        the default stream with the capturing one, which is illegal inside a capture
        (cudaErrorStreamCaptureImplicit; seen under compute-sanitizer, where the garbage collector's timing
        differs).  A new leaf per iteration has no history."""
        return self.latent.detach().requires_grad_(True)

    def _constraint_launch(self) -> None:
        """sdfr_point_constraint on the un-normalised orientation: += into g_raw / loss_extra."""
        if self.point_constraint is None:
            return
        _lib.check(_lib.lib().sdfr_point_constraint(
            self.orientation.data_ptr(), self.position.shape[0], self._pc_src, self._pc_tgt,
            self.point_constraint[2], self._g_raw.data_ptr(), self._loss_extra.data_ptr(), _stream()),
            "sdfr_point_constraint")

    def _tail_forward(self, with_bounds: bool):
        """The decoder trunk on a fresh latent leaf (autograd graph: latent -> x only), then the tail into this
        iteration's grids; ``with_bounds``: the tail also compares every value with the hypothesis' hit-threshold
        bound as it stores it, so the empty-space bounds cost no extra read of the grids.  Returns (leaf, x, w)."""
        dec, B, R = self.decoder, self.position.shape[0], self._R
        grids, gstride, layout = self._grid_op
        leaf = self._latent_leaf()
        x = dec.trunk(leaf).contiguous()
        w, bias = dec.tail_parameters()
        args = (x.data_ptr(), int(x.shape[1]), int(x.shape[2]), w.data_ptr(), _ptr(bias), _ptr(dec.base), B, R,
                grids.data_ptr(), gstride, layout)
        if with_bounds:
            _lib.check(_lib.lib().sdfr_decoder_tail_forward_bounds(
                *args, self.position.data_ptr(), self._inv_scale.data_ptr(), self.threshold,
                self._bounds.data_ptr(), _stream()), "sdfr_decoder_tail_forward_bounds")
        else:
            _lib.check(_lib.lib().sdfr_decoder_tail_forward(*args, _stream()), "sdfr_decoder_tail_forward")
        return leaf, x, w

    def _tail_backward(self, leaf: torch.Tensor, x: torch.Tensor, w: torch.Tensor, n_overlap=None, upstream=None,
                       g_sdf_pc=None, g_sdf_pc_stride: int = 0) -> torch.Tensor:
        """Tail adjoint of the gradient grid(s) -- with ``n_overlap`` and ``upstream`` it also applies the deferred
        depth-loss normalisation -- then autograd through the trunk: the latent gradient."""
        B, R = self.position.shape[0], self._R
        g_x = torch.empty_like(x)
        _lib.check(_lib.lib().sdfr_decoder_tail_backward(
            self._g_sdf.data_ptr(), R ** 3, n_overlap, upstream, g_sdf_pc, g_sdf_pc_stride, w.data_ptr(),
            int(x.shape[1]), int(x.shape[2]), B, R, g_x.data_ptr(), _stream()), "sdfr_decoder_tail_backward")
        (g_latent,) = torch.autograd.grad(x, leaf, g_x)
        return g_latent.contiguous()

    def _track_best(self, flags: int) -> None:
        """sdfr_track_best: inlier ratio of this iteration's counts, and the best estimate so far."""
        _lib.check(_lib.lib().sdfr_track_best(
            self._inl[0].data_ptr(), self._inl[1].data_ptr(), self.position.data_ptr(),
            self.orientation.data_ptr(), self.scale.data_ptr(), _ptr(self.latent), self._L, self.position.shape[0],
            self._t.data_ptr(), self.inlier_ratio.data_ptr(), self.best_inlier_ratio.data_ptr(),
            self.best_iteration.data_ptr(), self.best_position.data_ptr(),
            self.best_orientation.data_ptr(), self.best_scale.data_ptr(), _ptr(self.best_latent),
            flags, _stream()), "sdfr_track_best")

    def _fused_views_iteration(self) -> torch.Tensor:
        """One iteration over V views of the same object (simple_setup.py:408-463) as C-ABI launches:
        decoder tail -> camera-frame poses -> per view {bounds, render + compare, its backward with the
        1/n_overlap normalisation, point loss} -> pull-back to the world frame -> tail adjoint -> step."""
        lib, b = _lib.lib(), self._buf
        B, R, V = self.position.shape[0], self._R, self._V
        W, H, cx, cy, fx, fy = _camera_params(self.camera)
        grids, gstride, layout = self._grid_op
        flags = _lib.GRAD_POSITION | _lib.GRAD_ORIENTATION | _lib.GRAD_INV_SCALE
        if self.decoder is not None:
            self._g_both.zero_()
            leaf, x, w = self._tail_forward(with_bounds=False)
            flags |= _lib.GRAD_SDF
        render_flags = flags | (_lib.SDF_GRAD_EXACT if self.sdf_grad_mode == "exact" else 0)
        cam_p, cam_q = self._views
        pos_c, ori_c, isc_c = self._pose_c
        _lib.check(lib.sdfr_view_poses(
            self.position.data_ptr(), self._unit_q.data_ptr(), self._inv_scale.data_ptr(), cam_p.data_ptr(),
            cam_q.data_ptr(), V, B, pos_c.data_ptr(), ori_c.data_ptr(), isc_c.data_ptr(), _stream()),
            "sdfr_view_poses")
        g_sdf = _ptr(self._g_sdf)

        def view(t, v, k):  # slice v of a [V, B*k] buffer
            return t.data_ptr() + 4 * v * B * k

        for v in range(V):
            p_v, q_v, is_v = pos_c[v].data_ptr(), ori_c[v].data_ptr(), isc_c[v].data_ptr()
            obs = self.depth_obs[v].data_ptr()
            bounds = None
            if self._bounds is not None:
                bounds = self._grid_bounds(p_v, is_v, self._bounds[v])
            _lib.check(lib.sdfr_compare_forward(
                grids.data_ptr(), R, gstride, layout, p_v, q_v, is_v, B, W, H, cx, cy, fx, fy, self.threshold,
                obs, 0, self._depth.data_ptr(), view(b["loss_sum"], v, 1), view(b["n_overlap"], v, 1), 0,
                bounds, _stream()), "sdfr_compare_forward")
            # upstream = depth_weight: the gradients arrive weighted and normalised by this view's overlap
            _lib.check(lib.sdfr_compare_backward(
                self._depth.data_ptr(), obs, 0, view(b["n_overlap"], v, 1), self._up_d.data_ptr(),
                grids.data_ptr(), R, gstride, layout, p_v, q_v, is_v, B, W, H, cx, cy, fx, fy, g_sdf, R ** 3,
                view(b["gr_p"], v, 3), view(b["gr_q"], v, 4), view(b["gr_is"], v, 1), render_flags, bounds,
                _stream()), "sdfr_compare_backward")
            if self._view_M[v]:
                _lib.check(lib.sdfr_point_loss_fused(
                    self._view_points[v].data_ptr(), 0, self._view_M[v], grids.data_ptr(), R, gstride, layout,
                    p_v, q_v, self.scale.data_ptr(), B, self._view_up_p[v].data_ptr(), view(b["pl"], v, 1),
                    g_sdf, R ** 3, view(b["g2_p"], v, 3), view(b["g2_q"], v, 4), view(b["g2_s"], v, 1),
                    flags | _lib.LOSS_WEIGHTED, _stream()), "sdfr_point_loss_fused")
        if self.inlier_threshold is not None:  # on the last view's estimate (:463)
            _lib.check(lib.sdfr_inlier_count(
                self._depth.data_ptr(), self.depth_obs[V - 1].data_ptr(), 0, B, W, H, self.inlier_threshold,
                self._inl[0].data_ptr(), self._inl[1].data_ptr(), 0, _stream()), "sdfr_inlier_count")
        g_p, g_q, g_s = self._pb
        _lib.check(lib.sdfr_views_pull_back(
            cam_q.data_ptr(), self.scale.data_ptr(), V, B, b["gr_p"].data_ptr(), b["gr_q"].data_ptr(),
            b["gr_is"].data_ptr(), b["g2_p"].data_ptr(), b["g2_q"].data_ptr(), b["g2_s"].data_ptr(),
            b["loss_sum"].data_ptr(), b["n_overlap"].data_ptr(), float(self.depth_weight), b["pl"].data_ptr(),
            g_p.data_ptr(), g_q.data_ptr(), g_s.data_ptr(), self._loss_extra.data_ptr(),
            _lib.STEP_CLEAR_INPUTS, _stream()), "sdfr_views_pull_back")
        self._constraint_launch()
        g_latent = None if self.decoder is None else self._tail_backward(leaf, x, w)
        self._hyp_step(_lib.STEP_CLEAR_INPUTS, g_latent, self._g_raw, self._loss_extra)
        if self.inlier_threshold is not None:
            self._track_best(_lib.STEP_CLEAR_INPUTS)
        self.last_losses = self._loss
        return self.last_losses

    def _fused_iteration(self) -> torch.Tensor:
        if self._V:
            return self._fused_views_iteration()
        lib, b = _lib.lib(), self._buf
        B, R, M = self.position.shape[0], self._R, self._M
        W, H, cx, cy, fx, fy = _camera_params(self.camera)
        grids, gstride, layout = self._grid_op
        dec, tail_bounds = self.decoder, None
        main, side = torch.cuda.current_stream(), self._side

        def on_side(fn):
            """Run fn on the second stream after everything enqueued so far (or inline)."""
            if side is None:
                fn()
                return
            side.wait_stream(main)
            with torch.cuda.stream(side):
                fn()

        def clear_grids():
            self._g_both.zero_()

        if dec is not None:
            on_side(clear_grids)
            leaf, x, w = self._tail_forward(with_bounds=self._bounds is not None)
            if self._bounds is not None:
                tail_bounds = self._bounds.data_ptr()
            if side is not None:
                main.wait_stream(side)
        flags = _lib.GRAD_POSITION | _lib.GRAD_ORIENTATION | _lib.GRAD_INV_SCALE
        if dec is not None:
            flags |= _lib.GRAD_SDF
        render_flags = flags | (_lib.SDF_GRAD_EXACT if self.sdf_grad_mode == "exact" else 0)
        # empty-space bounds of this iteration's grids and poses (the hit-threshold bound depends on
        # position and scale): rays that cannot hit anything are not marched, all others unchanged
        bounds = tail_bounds
        self._constraint_launch()
        if self._bounds is not None and bounds is None:
            bounds = self._grid_bounds(self.position.data_ptr(), self._inv_scale.data_ptr(), self._bounds)

        def point_loss():
            _lib.check(lib.sdfr_point_loss_fused(
                self.points.data_ptr(), self._points_stride, M, grids.data_ptr(), R, gstride, layout,
                self.position.data_ptr(), self._unit_q.data_ptr(), self.scale.data_ptr(), B,
                self._up_p.data_ptr(), b["pl"].data_ptr(), _ptr(self._g_sdf_pc), R ** 3,
                b["g2_p"].data_ptr(), b["g2_q"].data_ptr(), b["g2_s"].data_ptr(),
                flags | self._point_flags, _stream()), "sdfr_point_loss_fused")

        if M:
            on_side(point_loss)
        # inliers of the result selection: counted in the same traversal (thresholds <= 1: a missed
        # pixel has relative error exactly 1), else by a separate pass over the written estimate
        inl_fused = self.inlier_threshold is not None and self.inlier_threshold <= 1.0
        if inl_fused:
            _lib.check(lib.sdfr_compare_fused_inliers(
                grids.data_ptr(), R, gstride, layout, self.position.data_ptr(), self._unit_q.data_ptr(),
                self._inv_scale.data_ptr(), B, W, H, cx, cy, fx, fy, self.threshold,
                self.depth_obs.data_ptr(), self._obs_stride, self._depth.data_ptr(),
                b["loss_sum"].data_ptr(), b["n_overlap"].data_ptr(), self.inlier_threshold,
                self._inl[0].data_ptr(), _ptr(self._g_sdf), R ** 3,
                b["gr_p"].data_ptr(), b["gr_q"].data_ptr(), b["gr_is"].data_ptr(), render_flags, bounds,
                _stream()), "sdfr_compare_fused_inliers")
        else:
            _lib.check(lib.sdfr_compare_fused(
                grids.data_ptr(), R, gstride, layout, self.position.data_ptr(), self._unit_q.data_ptr(),
                self._inv_scale.data_ptr(), B, W, H, cx, cy, fx, fy, self.threshold,
                self.depth_obs.data_ptr(), self._obs_stride, self._depth.data_ptr(),
                b["loss_sum"].data_ptr(), b["n_overlap"].data_ptr(), _ptr(self._g_sdf), R ** 3,
                b["gr_p"].data_ptr(), b["gr_q"].data_ptr(), b["gr_is"].data_ptr(), render_flags, bounds,
                _stream()), "sdfr_compare_fused")
        if M and side is not None:
            main.wait_stream(side)
        if self.inlier_threshold is not None and not inl_fused:
            # one streaming pass over the estimate, beside the decoder's backward
            def count_inliers():
                _lib.check(lib.sdfr_inlier_count(
                    self._depth.data_ptr(), self.depth_obs.data_ptr(), self._obs_stride, B, W, H,
                    self.inlier_threshold, self._inl[0].data_ptr(), self._inl[1].data_ptr(), 0,
                    _stream()), "sdfr_inlier_count")
            on_side(count_inliers)
        g_latent = None
        if dec is not None:
            g_latent = self._tail_backward(leaf, x, w, b["n_overlap"].data_ptr(), self._up_d.data_ptr(),
                                           _ptr(self._g_sdf_pc), R ** 3)
        self._hyp_step(_lib.STEP_CLEAR_INPUTS, g_latent, self._g_raw, self._loss_extra)
        if self.inlier_threshold is not None:
            if side is not None and not inl_fused:
                main.wait_stream(side)
            self._track_best(_lib.STEP_CLEAR_INPUTS | (_lib.TRACK_KEEP_VALID if inl_fused else 0))
        self.last_losses = self._loss
        return self.last_losses

    # ------------------------------------------------------------------------------------
    # optimizer="torch": the package's autograd operators and torch.optim.Adam
    # ------------------------------------------------------------------------------------
    def _torch_loss(self, q: torch.Tensor):
        """(loss, rendered depth, the observation the inlier ratio compares it with, no-overlap mask) of the
        current parameters; ``q`` is the unit orientation."""
        if self._views is not None:
            # V views of the same object (simple_setup.py:420-462): the pose is moved into every camera frame,
            # every view is rendered, compared and scored against its own observed points, the losses are
            # summed; autograd carries the gradients back through the rigid maps
            grids = self._grids()
            grids4 = grids if grids.dim() == 4 else grids[None]
            position_c, orientation_c = views.to_camera_frames(self.position, q, *self._views)
            inv_scale = (1.0 / self.scale).contiguous()
            loss, depth, no_overlap = 0.0, None, None
            for v in range(self.depth_obs.shape[0]):
                p_v, q_v = position_c[v].contiguous(), orientation_c[v].contiguous()
                loss_depth, depth, _ = render_and_compare(grids, p_v, q_v, inv_scale, self.depth_obs[v],
                                                          self.threshold, self.camera)
                loss = loss + self.depth_weight * torch.nan_to_num(loss_depth, nan=0.0)
                no_overlap = torch.isnan(loss_depth) if no_overlap is None else (no_overlap | torch.isnan(loss_depth))
                if self.pc_weight and self._view_points[v].shape[0] > 0:
                    loss = loss + self.pc_weight * losses.point_loss(self._view_points[v], p_v, q_v,
                                                                     self.scale, grids4)
            return loss, depth, self.depth_obs[-1], no_overlap  # the last view's inlier ratio (:463)
        if isinstance(self.decoder, FusedTailDecoder) and self.position.is_cuda \
                and self.point_counts is None:  # the chained operator takes one shared cloud
            # decoder tail, render-and-compare and point loss chained through the C ABI (estimation/fused.py):
            # no dense grid, no separate layout / scaling / add passes
            dec = self.decoder
            w, b = dec.tail_parameters()
            loss, depth, _, loss_depth = decode_render_compare(
                dec.trunk(self.latent), w, b, self.position, q.contiguous(), self.scale,
                self.depth_obs, self.points if self.pc_weight and self.points.shape[0] > 0 else None,
                dec.volume_size, self.threshold, self.camera, base=dec.base,
                depth_weight=self.depth_weight, pc_weight=self.pc_weight)
            return loss, depth, self.depth_obs, torch.isnan(loss_depth)
        grids = self._grids()
        loss_depth, depth, _ = render_and_compare(grids, self.position, q.contiguous(),
                                              (1.0 / self.scale).contiguous(), self.depth_obs,
                                              self.threshold, self.camera)
        no_overlap = torch.isnan(loss_depth)
        loss = self.depth_weight * torch.nan_to_num(loss_depth, nan=0.0)
        if self.pc_weight and self.points.shape[-2] > 0:
            # NB: the reference passes the un-normalised quaternion and lets pc_loss normalise it
            # (simple_setup.py:436-443, losses.py:56); q is already unit here, same value
            loss_pc = losses.point_loss(self.points, self.position, q, self.scale,
                                        grids if grids.dim() == 4 else grids[None])
            if self.point_counts is not None:  # mean over the instance's own points, not the padding
                n = self.point_counts.to(loss_pc.dtype)
                loss_pc = loss_pc * torch.where(n > 0, self.points.shape[1] / n.clamp(min=1.0),
                                                torch.zeros_like(n))
            loss = loss + self.pc_weight * loss_pc
        return loss, depth, self.depth_obs, no_overlap

    def _torch_step(self) -> torch.Tensor:
        self.optimizer.zero_grad(set_to_none=True)
        q = self.orientation / torch.linalg.norm(self.orientation, dim=1, keepdim=True)
        loss, depth, obs, no_overlap = self._torch_loss(q)
        if self.point_constraint is not None:
            # on the un-normalised orientation (simple_setup.py:164-175)
            source, target, weight = self.point_constraint
            loss = loss + weight * views.point_constraint_loss(self.orientation, source, target)
        loss.sum().backward()
        self.optimizer.step()
        with torch.no_grad():
            self.orientation /= torch.linalg.norm(self.orientation, dim=1, keepdim=True)
        if self.inlier_threshold is not None:
            self._track_best_torch(depth, obs)
        self.last_losses = self._reported(loss, no_overlap)
        return self.last_losses

    def _track_best_torch(self, depth: torch.Tensor, obs: Optional[torch.Tensor] = None) -> None:
        """simple_setup.py:177-211 with torch operators (optimizer="torch"; also the CPU statement
        the kernels are tested against): ratio of the depth rendered before the update, snapshot of the
        parameters after it."""
        with torch.no_grad():
            if obs is None:
                obs = self.depth_obs
            obs = obs if obs.dim() == 3 else obs[None]
            rel = (obs - depth.detach()).abs() / obs
            n_inlier = (rel < self.inlier_threshold).flatten(1).sum(1).to(torch.float32)
            n_valid = (obs != 0).flatten(1).sum(1).to(torch.float32).expand_as(n_inlier)
            ratio = n_inlier / n_valid
            self._iteration += 1
            better = (self.best_iteration < 0) | (ratio > self.best_inlier_ratio)
            self.inlier_ratio.copy_(ratio)
            self.best_inlier_ratio.copy_(torch.where(better, ratio, self.best_inlier_ratio))
            self.best_iteration.copy_(torch.where(better, self._iteration, self.best_iteration))
            for best, cur in ((self.best_position, self.position), (self.best_orientation, self.orientation),
                              (self.best_scale, self.scale), (self.best_latent, self.latent)):
                if best is not None:
                    best.copy_(torch.where(better.view(-1, *[1] * (cur.dim() - 1)), cur.detach(), best))

    def result(self, strategy: str = "last_iteration"):
        """(position, orientation, scale, latent) per hypothesis as SDFPipeline.__call__ returns them
        (simple_setup.py:583-592): ``"last_iteration"`` or ``"best_inlier_ratio"``."""
        if strategy == "last_iteration":
            return (self.position.detach(), self.orientation.detach(), self.scale.detach(),
                    None if self.latent is None else self.latent.detach())
        if strategy == "best_inlier_ratio":
            if self.inlier_threshold is None:
                raise ValueError("best_inlier_ratio needs inlier_threshold (the reference's default is 0.03)")
            return self.best_position, self.best_orientation, self.best_scale, self.best_latent
        raise ValueError(f"Result selection strategy {strategy} is not supported.")

    def _grids(self):
        if self.decoder is None:
            return self.sdf
        g = self.decoder(self.latent)
        return g[:, 0].contiguous() if g.dim() == 5 else g.contiguous()

    def capture(self, warmup: int = 3) -> None:
        """Capture one whole iteration (decode, render-and-compare, point loss, backward, Adam,
        renormalisation) in a CUDA graph; step() replays it afterwards.  The reference loop
        cannot be captured: it synchronises with the host twice per iteration
        (simple_setup.py:131, pointset_utils.py:60) and its renderer launches on the legacy
        default stream (sdf_renderer_cuda.cu:495)."""
        if not self.position.is_cuda:
            raise RuntimeError("CUDA graphs need CUDA tensors")
        with torch.cuda.device(self.position.device):
            self._capture(warmup)

    def _capture(self, warmup: int) -> None:
        side = torch.cuda.Stream(self.position.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self._eager_step()
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        if self.optimizer is not None:
            self.optimizer.zero_grad(set_to_none=True)
        with torch.cuda.graph(graph):
            self._static_loss = self._eager_step()
        self._graph = graph

    def step(self) -> torch.Tensor:
        """One iteration (simple_setup.py:408-470); returns the detached per-hypothesis loss."""
        if self._graph is not None:
            self._graph.replay()
            self.last_losses = self._static_loss
            return self.last_losses
        return self._eager_step()

    def _eager_step(self) -> torch.Tensor:
        if self.optimizer_impl == "fused":
            # the C ABI launches on the CURRENT device's stream: make the tensors' device current
            # (OptionalCUDAGuard of sdf_renderer.cpp:58, 82)
            with torch.cuda.device(self.position.device):
                return self._fused_iteration()
        return self._torch_step()

    @staticmethod
    def _reported(loss: torch.Tensor, no_overlap: Optional[torch.Tensor]) -> torch.Tensor:
        """The loss a caller sees: NaN where the rendered and the observed depth do not overlap -- the
        reference's mean over an empty selection (simple_setup.py:131).  The optimised loss uses 0
        there (zero gradients instead of the reference's NaN gradients), but a hypothesis that left the
        frustum must never rank best: ``global_best`` and ``SDFPipeline`` map NaN to +inf."""
        loss = loss.detach()
        if no_overlap is None:
            return loss
        return torch.where(no_overlap, torch.full_like(loss, float("nan")), loss)

    def run(self, iterations: int, gather_every: int = 0):
        """`iterations` steps; with gather_every=k the losses of all ranks are all-gathered every
        k-th iteration (and always after the last one).  Returns the gathered losses."""
        out = None
        for it in range(1, iterations + 1):
            local = self.step()
            if (gather_every and it % gather_every == 0) or it == iterations:
                if self._shard_sizes is None and dist.is_available() and dist.is_initialized() \
                        and dist.get_world_size(self.group) > 1:
                    self._shard_sizes = exchange_shard_sizes(local.numel(), local.device, self.group)
                out = gather_losses(local, self.group, self._shard_sizes)
        return out
