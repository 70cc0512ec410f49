"""`SDFPipeline`: the reference's estimation pipeline call, on the batched B200 loop.

Reference: sdfest/estimation/simple_setup.py -- ``SDFPipeline.__init__`` (:36-89), ``_parse_config``
(:91-110), ``__call__`` (:213-600), ``_preprocess_depth`` (:671-716), ``_nn_init`` (:718-844).
Same call signature, argument meaning, return value and errors for the parts on the render-and-compare
path; what surrounds that path in the reference and is out of this repository's scope (SURVEY.md
section 8: model files and their download, yoco configs, matplotlib visualisation, animation and log
writers, SO3 priors) is not rebuilt: the networks are handed in as modules, and the arguments that
drive those subsystems raise ``NotImplementedError`` instead of being silently ignored.

The loop itself is ``HypothesisOptimizer`` with one hypothesis: on CUDA tensors that is the fused
iteration (decoder trunk + fused tail, ``sdfr_compare_fused_inliers``, ``sdfr_point_loss_fused``, tail
adjoint, ``sdfr_hypothesis_step``, ``sdfr_track_best``; with several views or camera poses
``sdfr_view_poses`` / per-view render, compare and point loss / ``sdfr_views_pull_back``; with a point
constraint ``sdfr_point_constraint``), replayed from a CUDA graph.  A decoder that does not end in
interpolate-to-volume + 1x1x1 convolution runs through ``vae.decode`` and the autograd-composed
operators.  ``n_hypotheses`` > 1 (an extension) perturbs the initial pose and returns the best
hypothesis: highest best inlier ratio under ``best_inlier_ratio``, else lowest final loss.
``estimate_instances`` (an extension) runs that loop for every detection of a frame at once: the reference
runs ``__call__`` once per detection (estimation/scripts/real_data.py).
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from ..differentiable_renderer import Camera
from ..differentiable_renderer.sdf_renderer import get_empty_space_policy, get_sdf_grad_mode
from . import losses, views
from .decoder import FusedTailDecoder
from .hypotheses import HypothesisOptimizer


class NoDepthError(Exception):
    """Raised when there is no valid depth measurement after masking (simple_setup.py:30-33, :780)."""


class SDFPipeline:
    """``SDFPipeline(config, vae, init_network)(depth_images, masks, color_images, ...)``.

    config keys read (defaults as the reference's, estimation/configs/default.yaml): ``camera`` (dict of
    Camera arguments), ``threshold``, ``max_iterations`` (50), ``depth_weight`` (1.0), ``pc_weight``
    (3.0), ``mean_shape`` (False), ``init_view`` ("first"), ``result_selection_strategy``
    ("last_iteration" | "best_inlier_ratio"), ``relative_inlier_threshold`` (0.03), ``far_field``,
    ``init`` = {``backbone_type``, ``normalize_pose``, ``head``: {``orientation_repr``}}; extensions:
    ``cuda_graph`` (True), ``fused_decoder`` (True), ``n_hypotheses`` (1), ``max_points`` (0 = all),
    ``reuse_graph`` (True): keep the captured iteration of a call and replay it for later calls of the same
    shape (same number of views, shape optimisation on, same point constraint or none) -- the next observations,
    camera poses and initial estimate are loaded into the same device buffers (``HypothesisOptimizer.reset``),
    which removes the three eager warm-up iterations and the capture (~9 ms) from every call after the first;
    ``profile`` (False): record ``last_timings``.
    ``vae``: a module with ``decode(latent) -> (B,1,R,R,R)`` and a ``decoder`` attribute (the reference's
    ``SDFVAE``); ``init_network``: ``points (1,M,3) | depth (1,H,W) -> (latent, position, scale,
    orientation representation)`` (the reference's ``SDFPoseNet``), batched over rows for
    ``estimate_instances`` (every detection of a frame in one call).
    """

    def __init__(self, config: dict, vae: torch.nn.Module, init_network: torch.nn.Module):
        self.config = config
        self.device = config.get("device", "cuda")
        self.init_config = config.get("init", {})
        self.result_selection_strategy = config.get("result_selection_strategy", "last_iteration")
        if self.result_selection_strategy not in ("last_iteration", "best_inlier_ratio"):
            raise ValueError(f"Result selection strategy {self.result_selection_strategy} is not"
                             "supported.")
        self._relative_inlier_threshold = config.get("relative_inlier_threshold", 0.03)
        self._far_field = config.get("far_field")
        self.cam = Camera(**config["camera"])
        self.vae, self.init_network = vae.eval(), init_network.eval()
        for p in list(self.vae.parameters()) + list(self.init_network.parameters()):
            p.requires_grad_(False)  # both networks are frozen in the pipeline (simple_setup.py:65, 81)
        self._fused_decoder = None
        self.last_optimizer = None  # the HypothesisOptimizer of the last call (losses, inlier ratios)
        # config["profile"]: wall time of the call's phases (with device synchronisation between them: it
        # costs a few hundred microseconds per call, so it is off by default), the reference's
        # log_runtime breakdown (estimation/scripts/real_data.py:286-319) for this pipeline
        self.last_timings = None
        self._graph_cache = {}  # (hypotheses, latent size, decoder) -> captured HypothesisOptimizer

    # ------------------------------------------------------------------------------------------
    def _preprocess_depth(self, depth_images: torch.Tensor, masks: torch.Tensor) -> None:
        """In place, as the reference: zero outside the mask and beyond the far field (:671-692)."""
        depth_images[~masks] = 0
        if self._far_field is not None:
            depth_images[depth_images > self._far_field] = 0

    def _nn_init(self, depth_images, camera_positions, camera_orientations) -> Tuple:
        """Initial (latent (1,L), position (1,3), scale (1,), orientation (1,4)) in the world frame from
        the initialisation network on the first view (:718-844, ``init_view`` "first")."""
        head = self.init_config.get("head", {})
        repr_ = head.get("orientation_repr", "quaternion")
        if self.config.get("init_view", "first") != "first":
            raise NotImplementedError('Only the "first" init strategy is supported ("best" ranks the '
                                      "views by their SO3-grid posterior)")
        depth_image, cam_q, cam_p = depth_images[0], camera_orientations[0], camera_positions[0]
        centroid = None
        if self.init_config.get("backbone_type", "VanillaPointNet") == "VanillaPointNet":
            inp = losses.depth_to_pointcloud(depth_image, self.cam)
            if len(inp) == 0:
                raise NoDepthError
            if self.init_config.get("normalize_pose", True):
                centroid = inp.mean(dim=-2)  # pointset_utils.normalize_points (:12-31)
                inp = inp - centroid
        else:
            inp = depth_image
        latent, position, scale, orientation_repr = self.init_network(inp.unsqueeze(0))
        latent, position, scale = latent.clone(), position.clone(), scale.clone()
        if self.config.get("mean_shape", False):
            latent = torch.zeros_like(latent)
        if centroid is not None:
            position = position + centroid
        if repr_ == "quaternion":
            orientation_camera = orientation_repr
        elif repr_ == "discretized":  # the network's own SO3 grid (the reference's SDFPoseHead._grid)
            index = torch.softmax(orientation_repr, -1).argmax().item()
            orientation_camera = torch.tensor(self.init_network._head._grid.index_to_quat(index),
                                              dtype=torch.float, device=position.device).unsqueeze(0)
        else:
            raise NotImplementedError("Orientation representation is not supported")
        # outputs are in the camera frame: to the world frame (:820-826)
        position_world = views.quaternion_apply(cam_q, position) + cam_p
        orientation_world = views.quaternion_multiply(cam_q, orientation_camera)
        return latent, position_world, scale.reshape(-1), orientation_world

    def _decoder(self, on_cuda: bool):
        if on_cuda and self.config.get("fused_decoder", True):
            if self._fused_decoder is None:
                dec = self.vae.decoder
                try:
                    self._fused_decoder = dec if isinstance(dec, FusedTailDecoder) else FusedTailDecoder(dec)
                except ValueError:  # no interpolate + 1x1x1 tail to fuse: the plain decoder
                    self._fused_decoder = False
            if self._fused_decoder is not False:
                return self._fused_decoder
        return self.vae.decode

    # ------------------------------------------------------------------------------------------
    def __call__(self, depth_images: torch.Tensor, masks: torch.Tensor,
                 color_images: Optional[torch.Tensor] = None, visualize: bool = False,
                 camera_positions: Optional[torch.Tensor] = None,
                 camera_orientations: Optional[torch.Tensor] = None, log_path: Optional[str] = None,
                 shape_optimization: bool = True, animation_path: Optional[str] = None,
                 point_constraint=None, prior_orientation_distribution=None,
                 training_orientation_distribution=None) -> tuple:
        """Infer pose, size and latent shape from depth images and masks (:213-296).

        depth_images (N,H,W) or (H,W) -- modified in place by the mask, like the reference; masks the
        same shape, bool; camera_positions (N,3) / camera_orientations (N,4) camera-to-world, default
        origin / identity.  Returns (position (1,3), orientation (1,4), scale (1,), latent (1,L)).
        """
        if visualize or log_path is not None or animation_path is not None:
            raise NotImplementedError("visualisation, logging and animation writers are outside this "
                                      "package's scope (SURVEY.md section 8)")
        if prior_orientation_distribution is not None or training_orientation_distribution is not None:
            raise NotImplementedError("orientation priors act on the SO3 grid of the initialisation "
                                      "network, which is outside this package's scope")
        if depth_images.dim() == 2:  # add the view dimension (:306-313)
            depth_images, masks = depth_images.unsqueeze(0), masks.unsqueeze(0)
            if camera_positions is not None:
                camera_positions = camera_positions.unsqueeze(0)
            if camera_orientations is not None:
                camera_orientations = camera_orientations.unsqueeze(0)
        n_imgs, dev = depth_images.shape[0], depth_images.device
        marks, mark = self._phase_marks(dev)
        mark("start")
        world_is_camera = camera_positions is None and camera_orientations is None and n_imgs == 1
        if camera_positions is None:
            camera_positions = torch.zeros(n_imgs, 3, device=dev)
        if camera_orientations is None:
            camera_orientations = torch.zeros(n_imgs, 4, device=dev)
            camera_orientations[:, 3] = 1.0
        with torch.no_grad():
            self._preprocess_depth(depth_images, masks)
            latent, position, scale, orientation = self._nn_init(depth_images, camera_positions,
                                                                 camera_orientations)
        mark("preprocess_and_init_network")
        n_hyp = int(self.config.get("n_hypotheses", 1))
        if n_hyp > 1:  # extension: perturbed copies of the initial estimate, hypothesis 0 unperturbed
            g = torch.Generator(device="cpu").manual_seed(0)
            noise = lambda *s: torch.randn(*s, generator=g).to(dev)  # noqa: E731
            position = position.repeat(n_hyp, 1) + 0.02 * noise(n_hyp, 3) * (torch.arange(n_hyp, device=dev) > 0)[:, None]
            orientation = torch.nn.functional.normalize(
                orientation.repeat(n_hyp, 1) + 0.1 * noise(n_hyp, 4) * (torch.arange(n_hyp, device=dev) > 0)[:, None], dim=1)
            scale, latent = scale.repeat(n_hyp), latent.repeat(n_hyp, 1)

        if world_is_camera:
            obs, extra = depth_images[0].contiguous(), {}
        else:
            obs = depth_images.contiguous()
            extra = dict(camera_positions=camera_positions, camera_orientations=camera_orientations)
        # the view loop bakes in the number of views
        opt = self._optimize(obs, position, orientation, scale, latent, shape_optimization, n_hyp,
                             0 if world_is_camera else n_imgs, None, point_constraint, mark, **extra)
        position, orientation, scale, latent_out = opt.result(self.result_selection_strategy)
        if latent_out is None:
            latent_out = latent
        if n_hyp > 1:
            if self.result_selection_strategy == "best_inlier_ratio":
                best = int(torch.argmax(torch.nan_to_num(opt.best_inlier_ratio, nan=-1.0)))
            else:
                best = int(torch.argmin(torch.nan_to_num(opt.last_losses, nan=float("inf"))))
            position, orientation = position[best:best + 1], orientation[best:best + 1]
            scale, latent_out = scale[best:best + 1], latent_out[best:best + 1]
        # the optimiser's buffers are reused by the next call (`reuse_graph`): hand out copies
        position, orientation, scale, latent_out = (t.detach().clone() for t in (position, orientation, scale, latent_out))
        mark("result")
        if marks:
            self.last_timings = {b[0] + "_ms": (b[1] - a[1]) * 1e3 for a, b in zip(marks[:-1], marks[1:])}
        return position, orientation, scale, latent_out

    def estimate_instances(self, depth_image: torch.Tensor, masks: torch.Tensor,
                           color_image: Optional[torch.Tensor] = None, shape_optimization: bool = True) -> tuple:
        """Pose, size and latent shape of every detection of one frame in one call: ``depth_image`` (H,W) and
        ``masks`` (K,H,W) bool, one per detection; one view, in the camera frame.  Returns (position (K,3),
        orientation (K,4), scale (K,), latent (K,L)); row k is what ``__call__(depth_image, masks[k])`` returns.

        Unlike ``__call__``, the caller's depth image is NOT modified: the K masked depths (mask and far field
        applied, as ``__call__`` does in place) and their clouds come from one ``extract_instances`` call.
        Raises ``NoDepthError`` naming the detections without any depth after masking, before any network runs.
        The initialisation network runs once on all K detections; the loop optimises K x ``n_hypotheses``
        hypotheses together, each against its own detection, and keeps per detection the hypothesis
        ``result_selection_strategy`` ranks best.  With ``reuse_graph`` a later frame with as many detections
        replays the captured iteration of the first.
        """
        if depth_image.dim() != 2 or masks.dim() != 3 or tuple(masks.shape[1:]) != tuple(depth_image.shape):
            raise ValueError("depth_image (H,W) and masks (K,H,W) expected")
        K, dev = int(masks.shape[0]), depth_image.device
        marks, mark = self._phase_marks(dev)
        mark("start")
        with torch.no_grad():
            masked, points, counts = losses.extract_instances(depth_image, masks.to(torch.bool), self.cam,
                                                              self._far_field)
            n_points = counts.tolist()
            empty = [k for k, n in enumerate(n_points) if n == 0]
            if empty:
                raise NoDepthError(f"no valid depth after masking for detections {empty}")
            latent, position, scale, orientation = self._nn_init_instances(masked, points, counts)
        mark("preprocess_and_init_network")
        n_hyp = int(self.config.get("n_hypotheses", 1))
        if n_hyp > 1:  # every detection gets the perturbation rows __call__ uses, hypothesis 0 unperturbed
            g = torch.Generator(device="cpu").manual_seed(0)
            noise = lambda *s: torch.randn(*s, generator=g).to(dev)  # noqa: E731
            d_position = 0.02 * noise(n_hyp, 3) * (torch.arange(n_hyp, device=dev) > 0)[:, None]
            d_orientation = 0.1 * noise(n_hyp, 4) * (torch.arange(n_hyp, device=dev) > 0)[:, None]
            position = position.repeat_interleave(n_hyp, 0) + d_position.repeat(K, 1)
            orientation = torch.nn.functional.normalize(
                orientation.repeat_interleave(n_hyp, 0) + d_orientation.repeat(K, 1), dim=1)
            scale, latent = scale.repeat_interleave(n_hyp), latent.repeat_interleave(n_hyp, 0)
        instance = torch.arange(K, device=dev).repeat_interleave(n_hyp)
        opt = self._optimize(masked, position, orientation, scale, latent, shape_optimization, n_hyp,
                             ("instances", K), max(n_points), None, mark, instance=instance)
        position, orientation, scale, latent_out = opt.result(self.result_selection_strategy)
        if latent_out is None:
            latent_out = latent
        if n_hyp > 1:
            if self.result_selection_strategy == "best_inlier_ratio":
                best = torch.argmax(torch.nan_to_num(opt.best_inlier_ratio, nan=-1.0).view(K, n_hyp), dim=1)
            else:
                best = torch.argmin(torch.nan_to_num(opt.last_losses, nan=float("inf")).view(K, n_hyp), dim=1)
            rows = torch.arange(K, device=best.device) * n_hyp + best
            position, orientation, scale, latent_out = (t.index_select(0, rows.to(t.device))
                                                        for t in (position, orientation, scale, latent_out))
        # the optimiser's buffers are reused by the next call (`reuse_graph`): hand out copies
        position, orientation, scale, latent_out = (t.detach().clone() for t in (position, orientation, scale, latent_out))
        mark("result")
        if marks:
            self.last_timings = {b[0] + "_ms": (b[1] - a[1]) * 1e3 for a, b in zip(marks[:-1], marks[1:])}
        return position, orientation, scale, latent_out

    def _nn_init_instances(self, masked, points, counts) -> Tuple:
        """Initial (latent (K,L), position (K,3), scale (K,), orientation (K,4)) in the camera frame from ONE call
        of the initialisation network on all K detections (``_nn_init`` row by row).  A point-set backbone gets
        every cloud centred on its own centroid and padded to the largest one by repeating its own points
        cyclically: a max-pooled point network gives what it gives on the unpadded cloud."""
        head = self.init_config.get("head", {})
        repr_ = head.get("orientation_repr", "quaternion")
        if self.config.get("init_view", "first") != "first":
            raise NotImplementedError('Only the "first" init strategy is supported ("best" ranks the '
                                      "views by their SO3-grid posterior)")
        centroid = None
        if self.init_config.get("backbone_type", "VanillaPointNet") == "VanillaPointNet":
            K, M = int(points.shape[0]), int(points.shape[1])
            rows = torch.arange(M, device=points.device)
            own = (rows[None, :] % counts[:, None])[..., None].expand(K, M, 3)
            inp = torch.gather(points, 1, own)
            if self.init_config.get("normalize_pose", True):
                valid = (rows[None, :] < counts[:, None])[..., None]
                centroid = torch.where(valid, points, 0.0).sum(1) / counts[:, None].to(points.dtype)
                inp = inp - centroid[:, None]
        else:
            inp = masked
        latent, position, scale, orientation_repr = self.init_network(inp)
        latent, position, scale = latent.clone(), position.clone(), scale.clone()
        if self.config.get("mean_shape", False):
            latent = torch.zeros_like(latent)
        if centroid is not None:
            position = position + centroid
        if repr_ == "quaternion":
            orientation = orientation_repr
        elif repr_ == "discretized":  # the network's own SO3 grid, the argmax of every row
            index = torch.softmax(orientation_repr, -1).argmax(-1).tolist()
            orientation = torch.tensor([self.init_network._head._grid.index_to_quat(i) for i in index],
                                       dtype=torch.float, device=position.device).reshape(-1, 4)
        else:
            raise NotImplementedError("Orientation representation is not supported")
        return latent, position, scale.reshape(-1), orientation

    def _phase_marks(self, dev):
        """(marks, mark): ``mark(name)`` records the wall time of a phase boundary when ``profile`` is on."""
        marks = []

        def mark(name):
            if self.config.get("profile", False):
                import time

                if dev.type == "cuda":
                    torch.cuda.synchronize(dev)
                marks.append((name, time.perf_counter()))

        return marks, mark

    def _optimize(self, obs, position, orientation, scale, latent, shape_optimization, n_hyp, shape_key, n_obs,
                  point_constraint, mark, **extra) -> HypothesisOptimizer:
        """The loop of one call from the initial estimate: a HypothesisOptimizer on ``obs`` (``extra``: camera poses
        or object instances), captured and replayed, or -- ``reuse_graph`` -- the captured one of an earlier call
        of the same shape, reset to this call's observation.  ``shape_key``: what else the captured iteration bakes
        in (number of views, number of instances); ``n_obs``: the largest observed cloud when the caller knows it."""
        kw = dict(depth_weight=self.config.get("depth_weight", 1.0), pc_weight=self.config.get("pc_weight", 3.0),
                  max_points=int(self.config.get("max_points", 0)),
                  inlier_threshold=self._relative_inlier_threshold, point_constraint=point_constraint)
        if shape_optimization:
            kw.update(latent=latent, decoder=self._decoder(position.is_cuda))
        else:
            with torch.no_grad():
                kw.update(sdf=self.vae.decode(latent)[:, 0].contiguous())
        kw.update(extra)
        dev = obs.device
        n_it = int(self.config.get("max_iterations", 50))
        use_graph = self.config.get("cuda_graph", True) and n_it > 8
        # one captured iteration serves every call of the same shape (see `reuse_graph` above)
        reusable = (use_graph and self.config.get("reuse_graph", True) and position.is_cuda
                    and shape_optimization
                    and isinstance(kw.get("decoder"), FusedTailDecoder) and latent.shape[1] <= 64)
        opt, done = None, 0
        if reusable:
            # everything the captured iteration bakes in: sizes, the decoder object, and the loop's constants
            key = (n_hyp, int(latent.shape[1]), id(kw["decoder"]), str(dev), float(self.config["threshold"]),
                   float(kw["depth_weight"]), float(kw["pc_weight"]), int(kw["max_points"]),
                   float(kw["inlier_threshold"]), self.cam.width, self.cam.height, self.cam.fx, self.cam.fy,
                   self.cam.cx, self.cam.cy, self.cam.pixel_center, get_sdf_grad_mode(), get_empty_space_policy(),
                   # shape_key: what the loop bakes in besides; the point constraint's source / target / weight
                   # are launch arguments (host values) of the captured sdfr_point_constraint
                   shape_key,
                   None if point_constraint is None else tuple(
                       (float(v) for v in torch.as_tensor(point_constraint[0]).flatten().tolist()
                        + torch.as_tensor(point_constraint[1]).flatten().tolist() + [float(point_constraint[2])])))
            # the largest cloud of the call (one per view or instance) decides whether the cached buffers fit
            if not kw["pc_weight"]:
                n_obs = 0
            elif n_obs is None:
                n_obs = int((obs != 0).flatten(-2).sum(-1).max())
            n_pts = min(n_obs, kw["max_points"]) if kw["max_points"] else n_obs
            cached = self._graph_cache.get(key)
            if cached is not None and n_pts <= cached.point_capacity <= 2 * n_pts + 8192:
                cached.reset(position, orientation, scale, latent, obs, extra.get("camera_positions"),
                             extra.get("camera_orientations"))
                opt, done = cached, -1  # every iteration of this call is a replay
            else:
                kw["point_capacity"] = max(4096, -(-n_pts // 4096) * 4096 + 4096)  # room for the next clouds
        if opt is None:
            opt = HypothesisOptimizer(self.cam, self.config["threshold"], obs, position, orientation, scale, **kw)
        self.last_optimizer = opt
        mark("optimizer_setup")
        if done == 0 and opt.optimizer_impl == "fused" and use_graph:
            opt.capture(warmup=3)  # three eager iterations, then replays of the recorded one
            done = 3
            if reusable:
                self._graph_cache[key] = opt
        done = max(done, 0)
        mark("warmup_and_capture")
        for _ in range(n_it - done):
            opt.step()
        mark("iterations")
        return opt
