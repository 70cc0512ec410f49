"""Every detection of a frame in one call: ``sdfr_depth_to_points`` (the observed clouds of K object instances),
``losses.extract_instances``, ``HypothesisOptimizer`` with object instances, ``point_capacity`` and ``reset()``,
and ``SDFPipeline.estimate_instances``."""
import ctypes

import pytest
import torch
from torch import nn

from sdfest_b200 import _lib
from sdfest_b200.differentiable_renderer import Camera
from sdfest_b200.estimation import hypotheses, losses
from sdfest_b200.estimation.pipeline import NoDepthError, SDFPipeline

from test_pipeline_host import CONFIG, H, W, TinyVAE


def _torch_cloud(depth, camera):
    """The torch expression of losses.depth_to_pointcloud (pointset_utils.py:34-89)."""
    fx, fy, cx, cy, _ = camera.get_pinhole_camera_parameters(0.0)
    rows, cols = torch.nonzero(depth, as_tuple=True)
    z = depth[rows, cols]
    return torch.stack([(cols.float() - cx) * z / fx, -(rows.float() - cy) * z / fy, -z], dim=1)


def _torch_masked(depth, masks, far_field=None):
    """SDFPipeline._preprocess_depth of every instance, on copies."""
    out = (depth if depth.dim() == 3 else depth.expand(masks.shape[0], -1, -1)).clone()
    if masks is not None:
        out[~masks] = 0
    if far_field is not None:
        out[out > far_field] = 0
    return out


# ------------------------------------------------------------------------------------------------
# C ABI: argument validation (no GPU)
# ------------------------------------------------------------------------------------------------
def test_depth_to_points_argument_errors_need_no_gpu():
    from sdfest_b200 import build

    build.build()
    lib = _lib.lib()
    n = ctypes.c_longlong(-1)
    assert lib.sdfr_depth_to_points_scratch(3, 640, 480, ctypes.byref(n)) == 0
    assert n.value == 3 * 300 * 4  # one int per (instance, tile of 1024 pixels)
    assert lib.sdfr_depth_to_points_scratch(0, 640, 480, ctypes.byref(n)) == 0 and n.value == 0
    assert lib.sdfr_depth_to_points_scratch(3, 640, 480, None) == -1
    assert lib.sdfr_depth_to_points_scratch(-1, 640, 480, ctypes.byref(n)) == -2
    assert lib.sdfr_depth_to_points_scratch(1, 1 << 16, 1 << 15, ctypes.byref(n)) == -2  # > 2^30 pixels
    cam = (1e9, 500.0, 500.0, 320.0, 240.0)  # far_field, fx, fy, cx, cy

    def call(k=2, w=640, h=480, depth=None, stride=0, points=None, capacity=0, counts=None, scratch=None):
        return lib.sdfr_depth_to_points(depth, stride, None, k, w, h, *cam, None, points, capacity, counts, scratch,
                                        None)

    assert call(k=0) == 0  # nothing to do, nothing launched
    assert call() == -1  # NULL depth / counts / scratch
    assert b"NULL" in lib.sdfr_last_error()
    assert call(depth=16, counts=16, scratch=16, capacity=8) == -1  # points NULL with a capacity
    assert call(k=-1) == -2
    assert call(capacity=-1) == -2
    assert call(stride=-1) == -2
    assert call(w=0) == -2 and call(h=0) == -2
    assert call(w=1 << 16, h=1 << 15) == -2  # the image-size cap of sdfr_inlier_count


# ------------------------------------------------------------------------------------------------
# CPU: extract_instances (torch statement) and SDFPipeline.estimate_instances with host stand-ins
# ------------------------------------------------------------------------------------------------
def _frame():
    """One depth image (far-field outlier at (0,0)) and three detections of different sizes."""
    depth = torch.full((H, W), 0.8)
    depth[:, 8:] = 0.9
    depth[0, 0] = 5.0
    masks = torch.zeros(3, H, W, dtype=torch.bool)
    masks[0, 3:9, 4:11] = True
    masks[0, 0, 0] = True
    masks[1, 1:4, 12:15] = True
    masks[2, 7:12, 0:16] = True
    return depth, masks


def test_extract_instances_on_the_cpu():
    depth, masks = _frame()
    cam = Camera(**CONFIG["camera"])
    given = depth.clone()
    masked, points, counts = losses.extract_instances(given, masks, cam, far_field=2.0)
    assert torch.equal(given, depth)  # the caller's image is not modified
    want = _torch_masked(depth, masks, 2.0)
    assert torch.equal(masked, want)
    assert counts.tolist() == [42, 9, 80]
    assert points.shape == (3, 80, 3)
    for k in range(3):
        n = int(counts[k])
        assert torch.equal(points[k, :n], _torch_cloud(want[k], cam))
        assert bool((points[k, n:] == losses.PAD_COORDINATE).all())
    _, capped, n_capped = losses.extract_instances(depth, masks, cam, capacity=20)
    assert capped.shape == (3, 20, 3) and n_capped.tolist() == [43, 9, 80]  # true counts
    assert torch.equal(capped[2], _torch_cloud(_torch_masked(depth, masks)[2], cam)[:20])
    with pytest.raises(ValueError):
        losses.extract_instances(depth, None, cam)  # a shared image needs masks
    with pytest.raises(ValueError):
        losses.extract_instances(depth, masks.float(), cam)


class MaxPoolInit(nn.Module):
    """A point-set initialisation stand-in: per-point MLP (eval-mode batch norm), set-wise max, linear heads --
    the shape of gpu_configs.py::PointNetBackbone.  Records what it was given."""

    def __init__(self, latent_size=2):
        super().__init__()
        g = torch.Generator().manual_seed(3)
        self.mlp = nn.Sequential(nn.Linear(3, 16), nn.BatchNorm1d(16), nn.ReLU(), nn.Linear(16, 32), nn.ReLU())
        self.head = nn.Linear(32, latent_size + 3 + 1 + 4)
        with torch.no_grad():
            for p in self.parameters():
                p.copy_(0.3 * torch.randn(p.shape, generator=g))
            self.mlp[1].running_mean.copy_(0.1 * torch.randn(16, generator=g))
            self.mlp[1].running_var.copy_(1.0 + torch.rand(16, generator=g))
        self.latent_size = latent_size
        self.seen = []

    def forward(self, x):
        self.seen.append(x.detach().clone())
        B, M, _ = x.shape
        f = self.mlp(x.reshape(B * M, 3)).reshape(B, M, -1).amax(1)
        out = self.head(f)
        L = self.latent_size
        q = torch.nn.functional.normalize(out[:, L + 4:] * 0.1 + torch.tensor([0.0, 0.0, 0.0, 1.0]), dim=1)
        return out[:, :L], 0.01 * out[:, L:L + 3], 0.3 + 0.01 * out[:, L + 3], q


def _fake_render_and_compare(sdf, position, orientation, inv_scale, depth_obs, threshold, camera):
    """A differentiable stand-in for the CUDA renderer that compares hypothesis b with ITS observation."""
    B = position.shape[0]
    obs = depth_obs if depth_obs.dim() == 3 else depth_obs[None].expand(B, -1, -1)
    target = obs.sum((1, 2)) / (obs > 0).sum((1, 2))
    loss = (position[:, 2] + target) ** 2 + 0.1 * (orientation[:, 3] - 1) ** 2 + 0.01 * inv_scale + 0.0 * sdf.sum()
    return loss, obs * 1.02, torch.ones(B)


@pytest.fixture
def host_loop(monkeypatch):
    from oracle.pc_loss import point_loss

    monkeypatch.setattr(hypotheses, "render_and_compare", _fake_render_and_compare)
    monkeypatch.setattr(losses, "point_loss", point_loss)  # the product's point loss is CUDA-only


@pytest.mark.parametrize("n_hypotheses", [1, 2])
def test_estimate_instances_on_the_host(host_loop, n_hypotheses):
    depth, masks = _frame()
    init = MaxPoolInit()
    cfg = dict(CONFIG, far_field=2.0, n_hypotheses=n_hypotheses, profile=True)
    pipe = SDFPipeline(cfg, TinyVAE(), init)
    given = depth.clone()
    position, orientation, scale, latent = pipe.estimate_instances(given, masks)
    assert torch.equal(given, depth)  # unlike __call__, the caller's depth is untouched
    assert position.shape == (3, 3) and orientation.shape == (3, 4) and scale.shape == (3,) and latent.shape == (3, 2)
    assert set(pipe.last_timings) == {"preprocess_and_init_network_ms", "optimizer_setup_ms",
                                      "warmup_and_capture_ms", "iterations_ms", "result_ms"}
    # one batched call of the init network: clouds centred on their own points, padded cyclically to the largest
    assert len(init.seen) == 1
    seen = init.seen[0]
    counts = [42, 9, 80]
    assert seen.shape == (3, 80, 3)
    masked = _torch_masked(depth, masks, 2.0)
    for k, n in enumerate(counts):
        own = _torch_cloud(masked[k], pipe.cam)
        torch.testing.assert_close(seen[k, :n], own - own.mean(0), rtol=0, atol=1e-6)
        assert float(seen[k, :n].mean(0).abs().max()) < 1e-6
        assert torch.equal(seen[k], seen[k, torch.arange(80) % n])
    # row k is what __call__ gives for detection k alone
    for k in range(3):
        want = pipe(depth.clone(), masks[k], None)
        for got, w in zip((position, orientation, scale, latent), want):
            torch.testing.assert_close(got[k:k + 1], w, rtol=0, atol=1e-5)


def test_estimate_instances_errors(host_loop):
    depth, masks = _frame()
    init = MaxPoolInit()
    pipe = SDFPipeline(dict(CONFIG, far_field=2.0), TinyVAE(), init)
    masks[1] = False
    masks[2, :, :] = False
    masks[2, 0, 0] = True  # only the far-field outlier: nothing left after masking
    with pytest.raises(NoDepthError, match=r"\[1, 2\]"):
        pipe.estimate_instances(depth, masks)
    assert init.seen == []  # raised before any network ran
    with pytest.raises(ValueError):
        pipe.estimate_instances(depth[None], masks)


def test_batched_padded_pointnet_init_equals_per_instance_calls():
    """A max-pooled point network gives for the padded, centred (K,M,3) batch what it gives every cloud alone."""
    depth, masks = _frame()
    pipe = SDFPipeline(CONFIG, TinyVAE(), MaxPoolInit())
    masked, points, counts = losses.extract_instances(depth, masks, pipe.cam)
    batched = pipe._nn_init_instances(masked, points, counts)
    eye_q, zero_p = torch.tensor([[0.0, 0.0, 0.0, 1.0]]), torch.zeros(1, 3)
    for k in range(3):
        alone = pipe._nn_init(masked[k:k + 1], zero_p, eye_q)
        for b, a in zip(batched, alone):
            torch.testing.assert_close(b[k:k + 1], a.reshape(b[k:k + 1].shape), rtol=0, atol=1e-6)


# ------------------------------------------------------------------------------------------------
# GPU: the kernel against the torch expression
# ------------------------------------------------------------------------------------------------
def _random_scene(dev, K, H_, W_, seed, empty=None, full=None):
    g = torch.Generator().manual_seed(seed)
    depth = 0.3 + 2.0 * torch.rand(H_, W_, generator=g)
    depth[torch.rand(H_, W_, generator=g) < 0.2] = 0.0  # pixels without a measurement
    masks = torch.rand(K, H_, W_, generator=g) < torch.rand(K, 1, 1, generator=g)
    if empty is not None:
        masks[empty] = False
    if full is not None:
        masks[full] = True
    return depth.to(dev), masks.to(dev)


def _check_against_torch(depth, masks, cam, far_field=None, capacity=0):
    masked, points, counts = losses.extract_instances(depth, masks, cam, far_field, capacity)
    want = _torch_masked(depth, masks, far_field)
    assert torch.equal(masked, want)
    K = want.shape[0]
    for k in range(K):
        own = _torch_cloud(want[k], cam)
        n = own.shape[0]
        assert int(counts[k]) == n
        m = min(n, points.shape[1])
        assert torch.equal(points[k, :m], own[:m])
        assert bool((points[k, m:] == losses.PAD_COORDINATE).all())
    return counts


@pytest.mark.gpu
def test_depth_to_points_is_the_torch_expression(cuda_device):
    dev = cuda_device
    cam = Camera(640, 480, 525.0, 523.5, 319.3, 241.7, pixel_center=0.5)
    # shared depth, random masks with one empty and one full-image instance
    depth, masks = _random_scene(dev, 6, 480, 640, 0, empty=2, full=4)
    counts = _check_against_torch(depth, masks, cam)
    assert int(counts[2]) == 0 and int(counts[4]) == int((depth != 0).sum())
    # far field
    _check_against_torch(depth, masks, cam, far_field=1.2)
    # one depth map per instance, no masks
    per = torch.stack([torch.where(m, depth, torch.zeros_like(depth)) for m in masks])
    _check_against_torch(per, None, cam)
    # odd sizes, K = 1 and K = 40
    cam_odd = Camera(317, 239, 300.0, 301.0, 158.2, 119.9, pixel_center=0.5)
    for K, seed in ((1, 1), (40, 2)):
        depth, masks = _random_scene(dev, K, 239, 317, seed)
        _check_against_torch(depth, masks, cam_odd, far_field=2.0)
    # a capacity below some counts: true counts, clipped rows
    depth, masks = _random_scene(dev, 5, 239, 317, 3, full=0)
    counts = _check_against_torch(depth, masks, cam_odd, capacity=5000)
    assert int(counts[0]) > 5000


@pytest.mark.gpu
def test_depth_to_points_writes_nothing_past_the_capacity(cuda_device):
    dev = cuda_device
    cam = Camera(317, 239, 300.0, 301.0, 158.2, 119.9, pixel_center=0.5)
    depth, masks = _random_scene(dev, 3, 239, 317, 4, full=1)
    K, cap, guard = 3, 1000, 4096
    buf = torch.full((K * cap * 3 + guard,), -7.0, device=dev)
    masked = torch.full((K * 239 * 317 + guard,), -7.0, device=dev)
    counts = torch.full((K + 8,), -7, dtype=torch.int64, device=dev)
    n = ctypes.c_longlong(0)
    lib = _lib.lib()
    assert lib.sdfr_depth_to_points_scratch(K, 317, 239, ctypes.byref(n)) == 0
    scratch = torch.empty(n.value, dtype=torch.uint8, device=dev)
    fx, fy, cx, cy, _ = cam.get_pinhole_camera_parameters(0.0)
    _lib.check(lib.sdfr_depth_to_points(depth.data_ptr(), 0, masks.contiguous().data_ptr(), K, 317, 239, float("inf"),
                                        fx, fy, cx, cy, masked.data_ptr(), buf.data_ptr(), cap, counts.data_ptr(),
                                        scratch.data_ptr(), torch.cuda.current_stream().cuda_stream),
               "sdfr_depth_to_points")
    torch.cuda.synchronize()
    assert bool((buf[K * cap * 3:] == -7.0).all()) and bool((masked[K * 239 * 317:] == -7.0).all())
    assert bool((counts[K:] == -7).all())
    want = _torch_masked(depth, masks)
    assert int(counts[1]) == int((depth != 0).sum()) > cap
    points = buf[:K * cap * 3].view(K, cap, 3)
    for k in range(K):
        own = _torch_cloud(want[k], cam)
        assert int(counts[k]) == own.shape[0]
        m = min(own.shape[0], cap)
        assert torch.equal(points[k, :m], own[:m]) and bool((points[k, m:] == losses.PAD_COORDINATE).all())


@pytest.mark.gpu
def test_depth_to_points_replays_in_a_captured_graph(cuda_device):
    dev = cuda_device
    cam = Camera(317, 239, 300.0, 301.0, 158.2, 119.9, pixel_center=0.5)
    depth, masks = _random_scene(dev, 4, 239, 317, 5)
    static_depth, static_masks = depth.clone(), masks.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        losses.extract_instances(static_depth, static_masks, cam, 2.0, capacity=40000)  # warm-up
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = losses.extract_instances(static_depth, static_masks, cam, 2.0, capacity=40000)
    for seed in (6, 7):
        d, m = _random_scene(dev, 4, 239, 317, seed)
        static_depth.copy_(d)
        static_masks.copy_(m)
        graph.replay()
        torch.cuda.synchronize()
        want = losses.extract_instances(d, m, cam, 2.0, capacity=40000)
        for x, y in zip(out, want):
            assert torch.equal(x, y)
        assert int(out[2][0]) == _torch_cloud(_torch_masked(d, m, 2.0)[0], cam).shape[0]


@pytest.mark.gpu
def test_depth_to_pointclouds_on_cuda_matches_the_cpu(cuda_device):
    dev = cuda_device
    cam = Camera(317, 239, 300.0, 301.0, 158.2, 119.9, pixel_center=0.5)
    depth, masks = _random_scene(dev, 5, 239, 317, 8, empty=3)
    per = torch.stack([torch.where(m, depth, torch.zeros_like(depth)) for m in masks])
    got, n_got = losses.depth_to_pointclouds(per, cam)
    want, n_want = losses.depth_to_pointclouds(per.cpu(), cam)
    assert n_got.is_cuda and n_got.dtype == torch.int64 and torch.equal(n_got.cpu(), n_want)
    assert got.shape == want.shape
    got = got.cpu()
    # the same points in the same order; CUDA multiplies by the reciprocal of fx, the CPU divides: 1 ulp
    ulp = torch.nextafter(want.abs(), torch.full_like(want, float("inf"))) - want.abs()
    assert bool(((got - want).abs() <= ulp).all())
    # max_points: each instance's slice sub-sampled as before (same seed, same result)
    capped, n_capped = losses.depth_to_pointclouds(per, cam, max_points=500)
    for k in range(5):
        own = losses.subsample_points(_torch_cloud(per[k], cam), 500)
        assert int(n_capped[k]) == own.shape[0] and torch.equal(capped[k, :own.shape[0]], own)
    # depth_to_pointcloud: the kernel, the torch expression's bits
    assert torch.equal(losses.depth_to_pointcloud(per[0], cam), _torch_cloud(per[0], cam))
    assert torch.equal(losses.depth_to_pointcloud(depth, cam, mask=masks[1]), _torch_cloud(depth * masks[1], cam))


# ------------------------------------------------------------------------------------------------
# GPU: HypothesisOptimizer with object instances, point_capacity and reset()
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_instance_reset_reproduces_a_fresh_optimizer(cuda_device):
    from sdfest_b200 import synthetic as syn
    from sdfest_b200.estimation import HypothesisOptimizer
    from test_pipeline_gpu import CAMERA, THR, _observations

    dev = cuda_device
    dec, obs = _observations(dev)
    cam = Camera(**CAMERA)
    frames = [torch.stack(obs), torch.stack([obs[1], obs[2], obs[0]])]
    instance = torch.tensor([0, 0, 1, 1, 2, 2], device=dev)
    B = 6
    hyp = [syn.make_hypotheses(B, seed=s, device=dev, base_position=(0.0, -0.01, -0.55)) for s in (0, 1)]
    cap = max(int((o > 0).sum()) for o in obs) + 1024
    for kw in (dict(sdf=syn.sdf_mug(64, dev)[None].contiguous()), dict(decoder=dec)):
        def make(h, o, **extra):
            k = dict(kw)
            if "decoder" in k:
                k["latent"] = torch.zeros(B, 8, device=dev)
            return HypothesisOptimizer(cam, THR, o, h["position"], h["orientation"], 1.0 / h["inv_scale"],
                                       inlier_threshold=0.03, optimizer="fused", instance=instance, **k, **extra)

        a = make(hyp[0], frames[0], point_capacity=cap)
        assert a.points.shape == (B, cap, 3)
        a.capture(warmup=2)
        for _ in range(3):
            a.step()
        a.reset(hyp[1]["position"], hyp[1]["orientation"], 1.0 / hyp[1]["inv_scale"],
                torch.zeros(B, 8, device=dev) if "decoder" in kw else None, frames[1])
        b = make(hyp[1], frames[1])
        assert torch.equal(a.point_counts, b.point_counts)
        for _ in range(4):
            la, lb = a.step().clone(), b.step().clone()
            torch.testing.assert_close(la, lb, rtol=2e-3, atol=2e-5, equal_nan=True)
        assert float((a.position - b.position).abs().max()) < 1e-4
        torch.testing.assert_close(a.best_inlier_ratio, b.best_inlier_ratio, rtol=0, atol=2e-3)
        assert torch.equal(a.best_iteration, b.best_iteration)
        loaded = [t.clone() for t in (a.depth_obs, a.points, a.position)]
        too_big = frames[1].clone()
        too_big[1] = 0.7  # every pixel observed
        with pytest.raises(ValueError):
            a.reset(hyp[1]["position"], hyp[1]["orientation"], 1.0 / hyp[1]["inv_scale"],
                    torch.zeros(B, 8, device=dev) if "decoder" in kw else None, too_big)
        for t, want in zip((a.depth_obs, a.points, a.position), loaded):
            assert torch.equal(t, want)  # a rejected reset leaves the optimiser untouched
        with pytest.raises(ValueError):
            a.reset(hyp[1]["position"], hyp[1]["orientation"], 1.0 / hyp[1]["inv_scale"],
                    torch.zeros(B, 8, device=dev) if "decoder" in kw else None, frames[1][:2])  # K is fixed


# ------------------------------------------------------------------------------------------------
# GPU: SDFPipeline.estimate_instances against one __call__ per detection
# ------------------------------------------------------------------------------------------------
class PointSetInit(nn.Module):
    """Deterministic per input: a function of the set-wise maximum of the centred cloud (so padding by repeating
    the cloud's own points changes nothing), batched over rows."""

    def __init__(self, dev):
        super().__init__()
        self.dev = dev
        self.dummy = nn.Parameter(torch.zeros(1))
        self.base = (0.2 * torch.randn(1, 8, generator=torch.Generator().manual_seed(0))).to(dev)

    def forward(self, x):
        f = x.amax(1)  # (B,3)
        lat = self.base + 0.5 * f[:, :1]
        off = torch.tensor([[0.004, -0.003, -0.03]], device=self.dev) + 0.05 * f
        q = torch.nn.functional.normalize(
            torch.tensor([[0.03, -0.02, 0.01, 1.0]], device=self.dev) + 0.1 * torch.cat([f, 0 * f[:, :1]], 1), dim=1)
        return lat, off, torch.full((x.shape[0],), 0.148, device=self.dev), q


def _frame_of_three(dev, dec, shift):
    from sdfest_b200.differentiable_renderer import render_depth_composite
    from test_pipeline_gpu import CAMERA, THR

    cam = Camera(**CAMERA)
    grids = []
    for k in range(3):
        with torch.no_grad():
            z = 0.3 * torch.randn(1, 8, generator=torch.Generator().manual_seed(10 + k)).to(dev)
            grids.append(dec(z)[:, 0])
    grids = torch.cat(grids).contiguous()
    pos = torch.tensor([[-0.22 + shift, -0.02, -0.7], [0.0, 0.03 + shift, -0.6], [0.2, -0.01, -0.75 + shift]],
                       device=dev)
    quat = torch.tensor([[0.0, 0.0, 0.0, 1.0]] * 3, device=dev)
    inv_s = torch.tensor([1 / 0.15, 1 / 0.14, 1 / 0.15], device=dev)
    with torch.no_grad():
        depth, winner = render_depth_composite(grids, pos, quat, inv_s, THR, cam)
    masks = torch.stack([winner == k for k in range(3)])
    assert all(int(m.sum()) > 1000 for m in masks)
    return depth.contiguous(), masks


@pytest.mark.gpu
@pytest.mark.parametrize("n_hypotheses", [1, 2])
def test_estimate_instances_matches_one_call_per_detection(cuda_device, n_hypotheses):
    from test_pipeline_gpu import CAMERA, THR, VAE, _observations

    dev = cuda_device
    dec, _ = _observations(dev)
    cfg = {"device": str(dev), "camera": dict(CAMERA), "threshold": THR, "max_iterations": 25,
           "init": {"backbone_type": "VanillaPointNet", "normalize_pose": True, "head": {"orientation_repr": "quaternion"}},
           "result_selection_strategy": "best_inlier_ratio", "n_hypotheses": n_hypotheses}
    vae = VAE(dec)
    inst = SDFPipeline(cfg, vae, PointSetInit(dev))
    single = SDFPipeline(cfg, vae, PointSetInit(dev))
    fresh = SDFPipeline(dict(cfg, reuse_graph=False), vae, PointSetInit(dev))
    first_opt = None
    for shift in (0.0, 0.01):
        depth, masks = _frame_of_three(dev, dec, shift)
        given = depth.clone()
        got = inst.estimate_instances(given, masks)
        assert torch.equal(given, depth)
        if first_opt is None:
            first_opt = inst.last_optimizer
            assert first_opt.point_capacity > 0 and first_opt.position.shape == (3 * n_hypotheses, 3)
        else:
            assert inst.last_optimizer is first_opt  # no new optimiser, no new capture
            other = fresh.estimate_instances(depth, masks)
            assert fresh.last_optimizer.point_capacity == 0
            for x, y, tol in zip(got, other, (2e-4, 2e-3, 2e-4, 2e-3)):
                assert tuple(x.shape) == tuple(y.shape)
                assert float((x - y).abs().max()) <= tol, (x, y)
        assert [tuple(t.shape) for t in got] == [(3, 3), (3, 4), (3,), (3, 8)]
        for k in range(3):
            want = single(depth.clone(), masks[k], None)
            for x, y, tol in zip(got, want, (2e-4, 2e-3, 2e-4, 2e-3)):
                assert float((x[k:k + 1] - y).abs().max()) <= tol, (k, x[k], y)
