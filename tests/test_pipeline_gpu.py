"""SDFPipeline on the GPU with stand-in networks: the captured iteration of the first call is replayed for
later calls with other observations and initial estimates (``reuse_graph``), and gives what a freshly built
optimiser gives.  (The comparison with the reference's own pipeline is tests/test_dropin_reference.py.)"""
import pytest
import torch
from torch import nn

pytestmark = pytest.mark.gpu
W, H, R, THR = 320, 240, 64, 0.005
CAMERA = dict(width=W, height=H, fx=160.0, fy=160.0, cx=160.0, cy=120.0, pixel_center=0.5)


class VAE(nn.Module):
    def __init__(self, decoder):
        super().__init__()
        self.decoder = decoder

    def decode(self, z):
        return self.decoder(z)


class Init(nn.Module):
    """A fixed estimate relative to the centred input cloud, a different one per call."""

    def __init__(self, dev):
        super().__init__()
        self.dev, self.calls = dev, 0
        self.dummy = nn.Parameter(torch.zeros(1))

    def forward(self, x):
        k = self.calls
        self.calls += 1
        g = torch.Generator().manual_seed(k % 3)
        lat = (0.2 * torch.randn(1, 8, generator=g)).to(self.dev)
        off = torch.tensor([[0.004, -0.003, -0.03]], device=self.dev) * (1 + 0.2 * (k % 3))
        q = torch.nn.functional.normalize(torch.tensor([[0.03, -0.02, 0.01, 1.0]], device=self.dev) * 1.0, dim=1)
        return lat, off, torch.tensor([0.148], device=self.dev), q


def _observations(dev):
    from sdfest_b200 import synthetic as syn
    from sdfest_b200.differentiable_renderer import Camera, render_depth_batched

    dec = syn.residual_decoder(R, dev, syn.sdf_mug(R, dev))
    cam = Camera(**CAMERA)
    obs = []
    for k, (z, s) in enumerate(((-0.55, 0.15), (-0.8, 0.15), (-0.45, 0.14))):
        with torch.no_grad():
            grid = dec(0.3 * torch.randn(1, 8, generator=torch.Generator().manual_seed(10 + k)).to(dev))[:, 0].contiguous()
        obs.append(render_depth_batched(grid, torch.tensor([[0.01 * k, -0.01, z]], device=dev),
                                        torch.tensor([[0.0, 0.0, 0.0, 1.0]], device=dev),
                                        torch.tensor([1.0 / s], device=dev), THR, cam)[0])
    return dec, obs


def test_graph_of_the_first_call_serves_later_observations(cuda_device):
    from sdfest_b200.estimation import SDFPipeline

    dev = cuda_device
    dec, obs = _observations(dev)
    counts = [int((o > 0).sum()) for o in obs]
    assert min(counts) > 1000 and max(counts) > 1.5 * min(counts)  # clouds of clearly different sizes
    cfg = {"device": str(dev), "camera": dict(CAMERA), "threshold": THR, "max_iterations": 25,
           "init": {"backbone_type": "VanillaPointNet", "normalize_pose": True, "head": {"orientation_repr": "quaternion"}},
           "result_selection_strategy": "best_inlier_ratio"}
    vae = VAE(dec)
    reuse, fresh = SDFPipeline(cfg, vae, Init(dev)), SDFPipeline(dict(cfg, reuse_graph=False), vae, Init(dev))
    outs, first_opt = [], None
    for k in (0, 1, 2, 0):
        a = reuse(obs[k].clone(), obs[k] > 0, None)
        b = fresh(obs[k].clone(), obs[k] > 0, None)
        if first_opt is None:
            first_opt = reuse.last_optimizer
            assert first_opt.point_capacity >= counts[0]
        else:
            assert reuse.last_optimizer is first_opt  # no new optimiser, no new capture
            assert fresh.last_optimizer is not first_opt and fresh.last_optimizer.point_capacity == 0
        assert first_opt._n_points == counts[k]
        for x, y, tol in zip(a, b, (2e-4, 2e-3, 2e-4, 2e-3)):
            assert tuple(x.shape) == tuple(y.shape)
            assert float((x - y).abs().max()) <= tol, (k, x, y)
        assert abs(float(reuse.last_optimizer.best_inlier_ratio[0]) - float(fresh.last_optimizer.best_inlier_ratio[0])) < 5e-3
        outs.append([t.clone() for t in a])
        kept = a
    # results handed out earlier are copies: the next call did not overwrite them
    reuse(obs[1].clone(), obs[1] > 0, None)
    for x, y in zip(kept, outs[-1]):
        assert torch.equal(x, y)
    # a cloud that does not fit the capacity: a new optimiser is built (and cached) instead
    big = torch.where(obs[2] > 0, obs[2], torch.full_like(obs[2], 0.9))  # every pixel observed
    reuse(big, torch.ones_like(big, dtype=torch.bool), None)
    assert reuse.last_optimizer is not first_opt and reuse.last_optimizer.point_capacity >= W * H


def test_reset_reproduces_a_fresh_optimizer(cuda_device):
    """HypothesisOptimizer.reset: the same parameters, state and losses as a newly built optimiser, for fixed
    grids (slab minima kept) and with a decoder, eager and under a captured graph."""
    from sdfest_b200 import synthetic as syn
    from sdfest_b200.differentiable_renderer import Camera
    from sdfest_b200.estimation import HypothesisOptimizer

    dev = cuda_device
    dec, obs = _observations(dev)
    cam = Camera(**CAMERA)
    B = 3
    hyp = [syn.make_hypotheses(B, seed=s, device=dev, base_position=(0.0, -0.01, -0.55)) for s in (0, 1)]
    for kw in (dict(sdf=syn.sdf_mug(R, dev)[None].contiguous()), dict(decoder=dec)):
        def make(h, o, **extra):
            k = dict(kw)
            if "decoder" in k:
                k["latent"] = torch.zeros(B, 8, device=dev)
            return HypothesisOptimizer(cam, THR, o, h["position"], h["orientation"], 1.0 / h["inv_scale"],
                                       inlier_threshold=0.03, optimizer="fused", **k, **extra)

        a = make(hyp[0], obs[0], point_capacity=32768)
        a.capture(warmup=2)
        for _ in range(3):
            a.step()
        a.reset(hyp[1]["position"], hyp[1]["orientation"], 1.0 / hyp[1]["inv_scale"],
                torch.zeros(B, 8, device=dev) if "decoder" in kw else None, obs[1])
        b = make(hyp[1], obs[1])
        for _ in range(4):
            la, lb = a.step().clone(), b.step().clone()
            torch.testing.assert_close(la, lb, rtol=2e-3, atol=2e-5, equal_nan=True)
        assert float((a.position - b.position).abs().max()) < 1e-4
        torch.testing.assert_close(a.best_inlier_ratio, b.best_inlier_ratio, rtol=0, atol=2e-3)
        assert torch.equal(a.best_iteration, b.best_iteration)
        loaded = [t.clone() for t in (a.depth_obs, a.points, a.position)]
        with pytest.raises(ValueError):
            a.reset(hyp[1]["position"], hyp[1]["orientation"], 1.0 / hyp[1]["inv_scale"],
                    torch.zeros(B, 8, device=dev) if "decoder" in kw else None, torch.full_like(obs[1], 0.7))
        assert torch.equal(a.depth_obs, obs[1])  # a rejected reset leaves the optimiser untouched
        for t, want in zip((a.depth_obs, a.points, a.position), loaded):
            assert torch.equal(t, want)
    with pytest.raises(RuntimeError):
        make(hyp[0], obs[0]).reset(hyp[1]["position"], hyp[1]["orientation"], 1.0 / hyp[1]["inv_scale"],
                                   torch.zeros(B, 8, device=dev), obs[1])  # no capacity: cloud size is baked in


def test_graph_of_the_first_call_serves_later_views(cuda_device):
    """The view loop (two views with camera poses, with and without a point constraint): the iteration captured
    by the first call is replayed for later calls with other observations, camera poses and initial estimates,
    and gives what a pipeline that builds a new optimiser per call gives."""
    from sdfest_b200.estimation import SDFPipeline

    dev = cuda_device
    dec, obs = _observations(dev)
    cfg = {"device": str(dev), "camera": dict(CAMERA), "threshold": THR, "max_iterations": 20,
           "init": {"backbone_type": "VanillaPointNet", "normalize_pose": True, "head": {"orientation_repr": "quaternion"}},
           "result_selection_strategy": "best_inlier_ratio"}
    vae = VAE(dec)

    def cameras(k):  # the second camera a few centimetres / degrees away from the first, differently per call
        p = torch.tensor([[0.0, 0.0, 0.0], [0.02 + 0.01 * k, -0.01, 0.005 * k]], device=dev)
        q = torch.nn.functional.normalize(torch.tensor([[0.0, 0.0, 0.0, 1.0], [0.01 * (k + 1), -0.015, 0.005, 1.0]],
                                                       device=dev), dim=1)
        return p, q

    for constraint in (None, (torch.tensor([0.0, 0.0, 1.0]), torch.tensor([0.0, 0.0, 1.0]), 0.05)):
        reuse, fresh = SDFPipeline(cfg, vae, Init(dev)), SDFPipeline(dict(cfg, reuse_graph=False), vae, Init(dev))
        first_opt = None
        for k in (0, 1, 2, 1):
            views = torch.stack([obs[k], obs[(k + 1) % 3]])
            p, q = cameras(k)
            a = reuse(views.clone(), views > 0, None, camera_positions=p, camera_orientations=q,
                      point_constraint=constraint)
            b = fresh(views.clone(), views > 0, None, camera_positions=p, camera_orientations=q,
                      point_constraint=constraint)
            if first_opt is None:
                first_opt = reuse.last_optimizer
                assert first_opt._V == 2 and first_opt.point_capacity > 0
            else:
                assert reuse.last_optimizer is first_opt  # no new optimiser, no new capture
                assert fresh.last_optimizer is not first_opt
            assert first_opt._view_counts == [int((v > 0).sum()) for v in views]
            for x, y, tol in zip(a, b, (2e-4, 2e-3, 2e-4, 2e-3)):
                assert tuple(x.shape) == tuple(y.shape)
                assert float((x - y).abs().max()) <= tol, (k, x, y)
        if constraint is not None:  # another constraint is another captured launch: a new optimiser
            other = (constraint[0], torch.tensor([0.0, 1.0, 0.0]), 0.05)
            reuse(views.clone(), views > 0, None, camera_positions=p, camera_orientations=q, point_constraint=other)
            assert reuse.last_optimizer is not first_opt
