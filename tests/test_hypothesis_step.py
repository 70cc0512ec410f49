"""sdfr_hypothesis_step (ABI v7) and sdfr_point_loss_fused: the optimiser side of the loop.

CPU: the numpy oracle (oracle/hypothesis_step.py) is pinned against torch autograd through the
reference's chain (simple_setup.py:411, :431, :447-452) followed by torch.optim.Adam.step() and the
renormalisation (:462).  GPU: the kernel against that oracle; the fused optimiser against the
torch-composed one.
"""
import ctypes

import numpy as np
import pytest
import torch

from oracle import hypothesis_step as hs

LRS = (1e-3, 1e-2, 1e-3, 1e-2)


def _random_case(B, L, seed, with_points=True):
    rng = np.random.default_rng(seed)
    c = dict(
        position=rng.normal(0, 0.3, (B, 3)), orientation=rng.normal(0, 1, (B, 4)),
        scale=rng.uniform(0.1, 0.3, B), latent=rng.normal(0, 1, (B, L)) if L else None,
        loss_sum=rng.uniform(0, 50, B), n_overlap=rng.integers(0, 3, B) * rng.integers(1, 5000, B),
        gr_p=rng.normal(0, 300, (B, 3)), gr_q=rng.normal(0, 300, (B, 4)), gr_is=rng.normal(0, 30, B),
        g_latent=rng.normal(0, 1e-3, (B, L)) if L else None)
    c["orientation"] /= np.linalg.norm(c["orientation"], axis=1, keepdims=True) * rng.uniform(0.9, 1.1, (B, 1))
    if with_points:
        c.update(point_sum=rng.uniform(0, 10, B), g2_p=rng.normal(0, 1, (B, 3)),
                 g2_q=rng.normal(0, 1, (B, 4)), g2_s=rng.normal(0, 1, B))
    else:
        c.update(point_sum=None, g2_p=None, g2_q=None, g2_s=None)
    return {k: (None if v is None else np.asarray(v, np.float64)) for k, v in c.items()}


def _torch_reference(case, steps, depth_weight, point_weight):
    """The reference's own operators: autograd through q = o/|o|, 1/scale and the weighted loss
    with SURROGATE linear losses that have the given gradients, then torch.optim.Adam."""
    t = lambda a: None if a is None else torch.tensor(a, dtype=torch.float64)  # noqa: E731
    pos, ori, scale = (t(case[k]).requires_grad_(True) for k in ("position", "orientation", "scale"))
    groups = [{"params": [pos], "lr": LRS[0]}, {"params": [ori], "lr": LRS[1]}, {"params": [scale], "lr": LRS[2]}]
    lat = None
    if case["latent"] is not None:
        lat = t(case["latent"]).requires_grad_(True)
        groups.append({"params": [lat], "lr": LRS[3]})
    opt = torch.optim.Adam(groups)
    n = t(case["n_overlap"])
    coef = torch.where(n > 0, depth_weight / torch.where(n > 0, n, torch.ones_like(n)), torch.zeros_like(n))
    for _ in range(steps):
        opt.zero_grad()
        q = ori / torch.sqrt(torch.sum(ori ** 2, dim=1, keepdim=True))
        inv = 1 / scale
        loss = (coef * ((t(case["gr_p"]) * pos).sum(1) + (t(case["gr_q"]) * q).sum(1) + t(case["gr_is"]) * inv)).sum()
        if case["g2_p"] is not None:
            loss = loss + ((t(case["g2_p"]) * pos).sum(1) + (t(case["g2_q"]) * q).sum(1) + t(case["g2_s"]) * scale).sum()
        if lat is not None:
            loss = loss + (t(case["g_latent"]) * lat).sum()
        loss.backward()
        opt.step()
        with torch.no_grad():
            ori /= torch.sqrt(torch.sum(ori ** 2, dim=1, keepdim=True))
    return [None if x is None else x.detach().numpy() for x in (pos, ori, scale, lat)]


def _oracle_run(case, steps, depth_weight, point_weight, L):
    B = case["position"].shape[0]
    st = dict(position=case["position"], orientation=case["orientation"], scale=case["scale"],
              latent=case["latent"], m=np.zeros((B, 8 + L)), v=np.zeros((B, 8 + L)), t=0)
    out = None
    for _ in range(steps):
        out = hs.hypothesis_step(st, case["loss_sum"], case["n_overlap"], case["gr_p"], case["gr_q"],
                                 case["gr_is"], depth_weight, case["point_sum"], point_weight,
                                 case["g2_p"], case["g2_q"], case["g2_s"], case["g_latent"], LRS)
        st = out[0]
    return out


@pytest.mark.parametrize("L,with_points", [(0, True), (8, True), (5, False)])
def test_oracle_matches_torch_adam(L, with_points):
    case = _random_case(7, L, seed=L + 3, with_points=with_points)
    ref = _torch_reference(case, 6, 1.0, 0.01)
    st, unit, inv, loss = _oracle_run(case, 6, 1.0, 0.01, L)
    for a, b in zip(ref, (st["position"], st["orientation"], st["scale"], st["latent"])):
        if a is not None:
            np.testing.assert_allclose(b, a, rtol=1e-12, atol=1e-13)
    np.testing.assert_allclose(np.linalg.norm(unit, axis=1), 1.0, atol=1e-14)
    np.testing.assert_allclose(inv, 1.0 / st["scale"])
    n = case["n_overlap"]
    # no overlap: NaN like the reference's mean over an empty selection (simple_setup.py:131)
    exp = np.where(n > 0, case["loss_sum"] / np.where(n > 0, n, 1), np.nan)
    if with_points:
        exp = exp + 0.01 * case["point_sum"]
    assert np.isnan(exp).any() and not np.isnan(exp).all()
    np.testing.assert_allclose(loss, exp, equal_nan=True)


# ------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------
def _dev(case, dev):
    return {k: (None if v is None else torch.tensor(v, dtype=torch.float32, device=dev).contiguous())
            for k, v in case.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("B,L,with_points", [(1, 0, True), (64, 8, True), (300, 5, False)])
def test_step_kernel_matches_oracle(cuda_device, B, L, with_points):
    from sdfest_b200 import _lib

    lib = _lib.lib()
    case = _random_case(B, L, seed=11 + B, with_points=with_points)
    case32 = {k: (None if v is None else v.astype(np.float32).astype(np.float64)) for k, v in case.items()}
    d = _dev(case, cuda_device)
    m = torch.zeros((B, 8 + L), device=cuda_device)
    v = torch.zeros((B, 8 + L), device=cuda_device)
    t = torch.zeros(B, dtype=torch.int32, device=cuda_device)
    unit = torch.empty((B, 4), device=cuda_device)
    inv = torch.empty(B, device=cuda_device)
    loss = torch.empty(B, device=cuda_device)
    lr = (ctypes.c_float * 4)(*LRS)
    p = lambda x: None if x is None else x.data_ptr()  # noqa: E731
    steps = 5
    for _ in range(steps):
        _lib.check(lib.sdfr_hypothesis_step(
            p(d["position"]), p(d["orientation"]), p(d["scale"]), p(d["latent"]), L, B,
            p(d["loss_sum"]), p(d["n_overlap"]), p(d["gr_p"]), p(d["gr_q"]), p(d["gr_is"]), 1.0,
            p(d["point_sum"]), 0.01, p(d["g2_p"]), p(d["g2_q"]), p(d["g2_s"]), p(d["g_latent"]), None, None,
            p(m), p(v), p(t), lr, 0.9, 0.999, 1e-8, p(unit), p(inv), p(loss), 0, None), "step")
    torch.cuda.synchronize()
    st, unit_o, inv_o, loss_o = _oracle_run(case32, steps, 1.0, 0.01, L)
    assert int(t.min()) == steps and int(t.max()) == steps
    for name, got in (("position", d["position"]), ("orientation", d["orientation"]),
                      ("scale", d["scale"]), ("latent", d["latent"])):
        if got is not None:
            np.testing.assert_allclose(got.cpu().numpy(), st[name], rtol=2e-5, atol=2e-6, err_msg=name)
    np.testing.assert_allclose(unit.cpu().numpy(), unit_o, rtol=2e-5, atol=2e-6)
    np.testing.assert_allclose(inv.cpu().numpy(), inv_o, rtol=2e-5)
    np.testing.assert_allclose(loss.cpu().numpy(), loss_o, rtol=1e-5, atol=1e-6, equal_nan=True)
    np.testing.assert_allclose(m.cpu().numpy(), st["m"], rtol=1e-4, atol=1e-6)

    # NO_UPDATE leaves parameters and state alone; CLEAR_INPUTS zeroes what was consumed
    before = [x.clone() for x in (d["position"], d["orientation"], d["scale"], m, v)]
    _lib.check(lib.sdfr_hypothesis_step(
        p(d["position"]), p(d["orientation"]), p(d["scale"]), p(d["latent"]), L, B,
        p(d["loss_sum"]), p(d["n_overlap"]), p(d["gr_p"]), p(d["gr_q"]), p(d["gr_is"]), 1.0,
        p(d["point_sum"]), 0.01, p(d["g2_p"]), p(d["g2_q"]), p(d["g2_s"]), p(d["g_latent"]), None, None,
        p(m), p(v), p(t), lr, 0.9, 0.999, 1e-8, p(unit), p(inv), p(loss),
        _lib.STEP_NO_UPDATE | _lib.STEP_CLEAR_INPUTS, None), "step")
    torch.cuda.synchronize()
    for a, b in zip(before, (d["position"], d["orientation"], d["scale"], m, v)):
        assert torch.equal(a, b)
    assert int(t.max()) == steps
    for k in ("loss_sum", "n_overlap", "gr_p", "gr_q", "gr_is", "point_sum", "g2_p", "g2_q", "g2_s"):
        if d[k] is not None:
            assert float(d[k].abs().max()) == 0.0, k


@pytest.mark.gpu
def test_step_kernel_argument_errors(cuda_device):
    from sdfest_b200 import _lib

    lib = _lib.lib()
    x = torch.zeros(8, device=cuda_device)
    lr = (ctypes.c_float * 4)(*LRS)
    a = x.data_ptr()
    assert lib.sdfr_hypothesis_step(None, a, a, None, 0, 1, None, None, None, None, None, 1.0, None, 0.0,
                                    None, None, None, None, None, None, a, a, a, lr, 0.9, 0.999, 1e-8, None, None,
                                    None, 0, None) == -1
    assert lib.sdfr_hypothesis_step(a, a, a, None, 65, 1, None, None, None, None, None, 1.0, None, 0.0,
                                    None, None, None, None, None, None, a, a, a, lr, 0.9, 0.999, 1e-8, None, None,
                                    None, 0, None) == -2
    assert lib.sdfr_hypothesis_step(a, a, a, None, 0, 1, None, None, None, None, None, 1.0, None, 0.0,
                                    None, None, None, None, None, None, a, a, a, lr, 0.9, 0.999, 1e-8, None, None,
                                    None, 0x1, None) == -3
    assert lib.sdfr_hypothesis_step(a, a, a, None, 0, 0, None, None, None, None, None, 1.0, None, 0.0,
                                    None, None, None, None, None, None, None, None, None, None, 0.9, 0.999, 1e-8,
                                    None, None, None, 0, None) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["dense", "skewed"])
def test_point_loss_fused_matches_forward_and_backward(cuda_device, layout):
    from sdfest_b200 import _lib, synthetic as syn
    from sdfest_b200.differentiable_renderer.sdf_renderer import _skewed_elems

    lib, dev = _lib.lib(), cuda_device
    B, R, M = 5, 32, 4000
    hyp = syn.make_hypotheses(B, seed=3, device=dev)
    grids = syn.hypothesis_grids(hyp["shape_param"], R, dev).contiguous()
    scale = (1.0 / hyp["inv_scale"]).contiguous()
    g = torch.Generator(device="cpu").manual_seed(0)
    pts = (torch.randn(M, 3, generator=g) * 0.12).to(dev) + hyp["position"][0]
    pts = pts.contiguous()
    up = torch.full((B,), 3.0 / M, device=dev)
    if layout == "skewed":
        SK = _skewed_elems(R)
        src = torch.empty((B, SK), device=dev)
        _lib.check(lib.sdfr_skew_grids(grids.data_ptr(), R, R ** 3, B, src.data_ptr(), SK, None), "skew")
        stride, lay = SK, _lib.LAYOUT_SKEWED
    else:
        src, stride, lay = grids, R ** 3, _lib.LAYOUT_DENSE
    flags = _lib.GRAD_ALL | _lib.ZERO_GRADS
    pose = (hyp["position"].data_ptr(), hyp["orientation"].data_ptr(), scale.data_ptr())

    def bufs():
        return (torch.empty(B, device=dev), torch.empty((B, R ** 3), device=dev), torch.empty((B, 3), device=dev),
                torch.empty((B, 4), device=dev), torch.empty(B, device=dev))

    l0, gs0, gp0, gq0, gsc0 = bufs()
    _lib.check(lib.sdfr_point_loss_forward(pts.data_ptr(), 0, M, src.data_ptr(), R, stride, lay, *pose, B,
                                           l0.data_ptr(), _lib.ZERO_GRADS, None), "fwd")
    _lib.check(lib.sdfr_point_loss_backward(pts.data_ptr(), 0, M, src.data_ptr(), R, stride, lay, *pose, B,
                                            up.data_ptr(), gs0.data_ptr(), R ** 3, gp0.data_ptr(),
                                            gq0.data_ptr(), gsc0.data_ptr(), flags, None), "bwd")
    l1, gs1, gp1, gq1, gsc1 = bufs()
    _lib.check(lib.sdfr_point_loss_fused(pts.data_ptr(), 0, M, src.data_ptr(), R, stride, lay, *pose, B,
                                         up.data_ptr(), l1.data_ptr(), gs1.data_ptr(), R ** 3,
                                         gp1.data_ptr(), gq1.data_ptr(), gsc1.data_ptr(), flags, None), "fused")
    torch.cuda.synchronize()
    assert float(l0.abs().min()) > 0
    for a, b in ((l0, l1), (gp0, gp1), (gq0, gq1), (gsc0, gsc1), (gs0, gs1)):
        torch.testing.assert_close(b, a, rtol=1e-4, atol=1e-6 * float(a.abs().max()))
    # loss only (no gradient flags): the forward kernel
    l2 = torch.empty(B, device=dev)
    _lib.check(lib.sdfr_point_loss_fused(pts.data_ptr(), 0, M, src.data_ptr(), R, stride, lay, *pose, B,
                                         None, l2.data_ptr(), None, 0, None, None, None, _lib.ZERO_GRADS,
                                         None), "fused loss only")
    torch.testing.assert_close(l2, l0, rtol=1e-5, atol=0)


def _make_optimizers(dev, B, with_decoder, optimizer):
    from sdfest_b200 import synthetic as syn
    from sdfest_b200.differentiable_renderer import Camera, render_depth_batched
    from sdfest_b200.estimation import HypothesisOptimizer

    W, H, thr = 160, 120, 0.005
    R = 64 if with_decoder else 32  # the mug decoder architecture ends at 64^3
    cam = Camera(W, H, W / 2, W / 2, W / 2, H / 2, pixel_center=0.5)
    hyp = syn.make_hypotheses(B, seed=0, device=dev)
    base = syn.make_hypotheses(1, seed=0, device=dev)
    obs = render_depth_batched(syn.hypothesis_grids(base["shape_param"], R, dev), base["position"],
                               base["orientation"], base["inv_scale"], thr, cam)[0].contiguous()
    torch.manual_seed(0)
    if with_decoder:
        dec = syn.residual_decoder(R, dev, syn.sdf_mug(R, dev))
        kw = dict(latent=0.1 * torch.randn(B, 8, device=dev), decoder=dec)
    else:
        kw = dict(sdf=syn.hypothesis_grids(hyp["shape_param"], R, dev))
    return HypothesisOptimizer(cam, thr, obs, hyp["position"], hyp["orientation"], 1.0 / hyp["inv_scale"],
                               optimizer=optimizer, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("with_decoder", [False, True])
def test_fused_optimizer_matches_torch_optimizer(cuda_device, with_decoder):
    B, steps = 6, 4
    a = _make_optimizers(cuda_device, B, with_decoder, "torch")
    b = _make_optimizers(cuda_device, B, with_decoder, "fused")
    assert a.optimizer_impl == "torch" and b.optimizer_impl == "fused"
    for _ in range(steps):
        la = a.step().clone()
        lb = b.step().clone()
        torch.testing.assert_close(lb, la, rtol=2e-3, atol=1e-5)
    # Adam's first steps move every parameter by ~lr regardless of the gradient's size, so
    # parameters agree to a small fraction of steps * lr unless a gradient is pure noise
    for name, lr in (("position", 1e-3), ("orientation", 1e-2), ("scale", 1e-3)):
        pa, pb = getattr(a, name).detach(), getattr(b, name).detach()
        assert float((pa - pb).abs().max()) < 0.05 * lr * steps, name
    if with_decoder:
        moved = float((a.latent.detach() - 0.0).abs().max())
        assert moved > 0
        assert float((a.latent.detach() - b.latent.detach()).abs().max()) < 0.05 * 1e-2 * steps
    torch.testing.assert_close(torch.linalg.norm(b.orientation, dim=1),
                               torch.ones(B, device=cuda_device), rtol=0, atol=1e-6)


@pytest.mark.gpu
def test_fused_optimizer_graph_replay_matches_eager(cuda_device):
    a = _make_optimizers(cuda_device, 4, True, "fused")
    b = _make_optimizers(cuda_device, 4, True, "fused")
    a.step()
    b.capture(warmup=1)  # one eager iteration, then one recorded (not executed) iteration
    for _ in range(3):
        la = a.step().clone()
        lb = b.step().clone()
    torch.cuda.synchronize()
    torch.testing.assert_close(lb, la, rtol=2e-3, atol=1e-5)
    assert float((a.position - b.position).abs().max()) < 1e-4
    assert float((a.latent.detach() - b.latent.detach()).abs().max()) < 1e-3


@pytest.mark.gpu
def test_fused_optimizer_at_full_c2_size(cuda_device):
    """BASELINE config 2 at full size (64 hypotheses x 640x480, 64^3, decoder in the loop): the fused
    iteration and the torch-composed one report the same per-hypothesis losses step by step, the loss
    of the batch goes down, quaternions stay unit length, and graph replay continues the sequence."""
    from sdfest_b200 import synthetic as syn
    from sdfest_b200.differentiable_renderer import Camera, render_depth_batched
    from sdfest_b200.estimation import HypothesisOptimizer

    dev = cuda_device
    B, W, H, R, thr = 64, 640, 480, 64, 0.005
    cam = Camera(W, H, 320.0, 320.0, 320.0, 240.0, pixel_center=0.5)
    hyp = syn.make_hypotheses(B, seed=0, device=dev)
    base = syn.make_hypotheses(1, seed=0, device=dev)
    obs = render_depth_batched(syn.hypothesis_grids(base["shape_param"], R, dev), base["position"],
                               base["orientation"], base["inv_scale"], thr, cam)[0].contiguous()

    def make(optimizer):
        dec = syn.residual_decoder(R, dev, syn.sdf_mug(R, dev))
        return HypothesisOptimizer(cam, thr, obs, hyp["position"], hyp["orientation"], 1.0 / hyp["inv_scale"],
                                   latent=torch.zeros(B, 8, device=dev), decoder=dec, optimizer=optimizer)

    a, b = make("torch"), make("fused")
    first = None
    for it in range(4):
        la, lb = a.step().clone(), b.step().clone()
        torch.testing.assert_close(lb, la, rtol=3e-3, atol=2e-5)
        first = lb if first is None else first
    b.capture(warmup=1)
    for _ in range(10):
        last = b.step()
    torch.cuda.synchronize()
    assert float(last.mean()) < 0.8 * float(first.mean())
    assert bool(torch.isfinite(last).all())
    torch.testing.assert_close(torch.linalg.norm(b.orientation, dim=1), torch.ones(B, device=dev),
                               rtol=0, atol=1e-6)
    assert float(b.latent.detach().abs().max()) > 0


def _instance_scene(dev, K, per):
    """K object instances (different poses and apparent sizes -> clouds of different sizes, one of them
    cropped to a few rows), `per` hypotheses each."""
    from sdfest_b200 import synthetic as syn
    from sdfest_b200.differentiable_renderer import Camera, render_depth_batched

    W, H, R, thr = 160, 120, 32, 0.005
    cam = Camera(W, H, W / 2, W / 2, W / 2, H / 2, pixel_center=0.5)
    truth = syn.make_hypotheses(K, seed=5, device=dev)
    truth["position"][:, 2] -= 0.08 * torch.arange(K, device=dev)  # farther away = fewer pixels
    grid = syn.sdf_mug(R, dev)[None].contiguous()
    obs = render_depth_batched(grid, truth["position"], truth["orientation"], truth["inv_scale"], thr,
                               cam).contiguous()
    obs[K - 1, : H // 2] = 0.0
    hyp = syn.make_hypotheses(K * per, seed=1, device=dev)
    instance = torch.arange(K * per, device=dev) // per
    hyp["position"] = (hyp["position"] - hyp["position"].mean(0)) + truth["position"][instance]
    return cam, thr, grid, obs, hyp, instance


@pytest.mark.gpu
@pytest.mark.parametrize("max_points", [0, 500])
def test_instance_batched_optimizer_equals_one_optimizer_per_instance(cuda_device, max_points):
    """Object instances in one batch (depth map + observed points per instance, SDFR_LOSS_WEIGHTED):
    the same numbers as running the shared-observation optimiser once per instance."""
    from sdfest_b200.estimation import HypothesisOptimizer

    K, per, steps = 3, 4, 5
    cam, thr, grid, obs, hyp, instance = _instance_scene(cuda_device, K, per)
    kw = dict(sdf=grid, optimizer="fused", max_points=max_points)
    joint = HypothesisOptimizer(cam, thr, obs, hyp["position"], hyp["orientation"], 1.0 / hyp["inv_scale"],
                                instance=instance, **kw)
    counts = joint.point_counts.view(K, per)[:, 0].tolist()
    assert len(set(counts)) == K or max_points  # the clouds really differ in size
    singles = [HypothesisOptimizer(cam, thr, obs[k], hyp["position"][k * per:(k + 1) * per],
                                   hyp["orientation"][k * per:(k + 1) * per],
                                   1.0 / hyp["inv_scale"][k * per:(k + 1) * per], **kw) for k in range(K)]
    for _ in range(steps):
        lj = joint.step().clone()
        ls = torch.cat([s.step().clone() for s in singles])
        torch.testing.assert_close(lj, ls, rtol=1e-4, atol=1e-6)
    for name, lr in (("position", 1e-3), ("orientation", 1e-2), ("scale", 1e-3)):
        pj = getattr(joint, name).detach()
        ps = torch.cat([getattr(s, name).detach() for s in singles])
        assert float((pj - ps).abs().max()) < 0.05 * lr * steps, name
    assert float(lj.min()) > 0


@pytest.mark.gpu
def test_instance_batched_fused_matches_torch_composition(cuda_device):
    from sdfest_b200.estimation import HypothesisOptimizer

    K, per, steps = 3, 2, 4
    cam, thr, grid, obs, hyp, instance = _instance_scene(cuda_device, K, per)

    def make(optimizer):
        return HypothesisOptimizer(cam, thr, obs, hyp["position"], hyp["orientation"], 1.0 / hyp["inv_scale"],
                                   sdf=grid, optimizer=optimizer, instance=instance)

    a, b = make("torch"), make("fused")
    la = a.step().clone()
    b.capture(warmup=1)  # one eager iteration, then graph replay
    torch.testing.assert_close(b.last_losses, la, rtol=2e-3, atol=1e-5)
    for _ in range(steps):
        la, lb = a.step().clone(), b.step().clone()
        torch.testing.assert_close(lb, la, rtol=2e-3, atol=1e-5)
    for name, lr in (("position", 1e-3), ("orientation", 1e-2), ("scale", 1e-3)):
        assert float((getattr(a, name).detach() - getattr(b, name).detach()).abs().max()) < 0.05 * lr * (steps + 1)
    with pytest.raises(ValueError):
        HypothesisOptimizer(cam, thr, obs[0], hyp["position"], hyp["orientation"], 1.0 / hyp["inv_scale"],
                            sdf=grid, instance=instance)
    with pytest.raises(ValueError):
        HypothesisOptimizer(cam, thr, obs, hyp["position"], hyp["orientation"], 1.0 / hyp["inv_scale"],
                            sdf=grid, instance=instance + 1)


# ------------------------------------------------------------------------------------------
# result selection: inlier ratio and best estimate (simple_setup.py:177-211)
# ------------------------------------------------------------------------------------------
def _inlier_images(B, H, W, seed):
    """Estimates and observations with every special case of the torch expression: obs == 0 with and
    without an estimate (nan / inf: never inliers), misses of the estimate, errors just below and above
    the threshold."""
    g = np.random.default_rng(seed)
    obs = (0.4 + 0.3 * g.random((B, H, W))).astype(np.float32)
    obs[g.random((B, H, W)) < 0.3] = 0.0
    est = (obs * (1 + 0.06 * (g.random((B, H, W)) - 0.5))).astype(np.float32)
    est[g.random((B, H, W)) < 0.2] = 0.0
    est[(obs == 0) & (g.random((B, H, W)) < 0.5)] = 0.5
    return obs, est


def test_track_best_torch_statement_matches_oracle():
    """The torch statement of the result selection (the optimizer="torch" path, usable on CPU) against
    the numpy oracle, over a sequence of iterations with parameters that keep moving."""
    from oracle import hypothesis_step as hs
    from sdfest_b200.differentiable_renderer import Camera
    from sdfest_b200.estimation import HypothesisOptimizer

    B, H, W, thr = 3, 12, 16, 0.03
    cam = Camera(W, H, 14.0, 14.0, 8.0, 6.0, pixel_center=0.5)
    obs, _ = _inlier_images(B, H, W, 0)
    opt = HypothesisOptimizer(cam, 0.005, torch.tensor(obs), torch.zeros(B, 3), torch.tensor([[0.0, 0, 0, 1]]).repeat(B, 1),
                              torch.ones(B), sdf=torch.zeros(1, 8, 8, 8), inlier_threshold=thr)
    best = [hs.BestEstimate() for _ in range(B)]
    for it in range(1, 7):
        _, est = _inlier_images(B, H, W, it)
        if it == 4:
            est = obs.copy()  # a perfect iteration in the middle: must stay the best
        with torch.no_grad():
            opt.position += 0.01
            opt.scale *= 1.01
        opt._track_best_torch(torch.tensor(est))
        for b in range(B):
            ni, nv = hs.inlier_counts(obs[b], est[b], thr)
            r = best[b].update(ni, nv, it, (opt.position[b].detach().numpy(), opt.scale[b].detach().numpy()))
            assert float(opt.inlier_ratio[b]) == pytest.approx(float(r), rel=1e-6)
    assert opt.best_iteration.tolist() == [4] * B
    for b in range(B):
        assert best[b].iteration == 4 and float(opt.best_inlier_ratio[b]) == 1.0
        np.testing.assert_array_equal(opt.best_position[b].numpy(), best[b].params[0])
        np.testing.assert_array_equal(opt.best_scale[b].numpy(), best[b].params[1])
    pos, quat, scale, latent = opt.result("best_inlier_ratio")
    assert torch.equal(pos, opt.best_position) and latent is None
    assert torch.equal(opt.result("last_iteration")[0], opt.position.detach())
    with pytest.raises(ValueError):
        opt.result("median")
    plain = HypothesisOptimizer(cam, 0.005, torch.tensor(obs), torch.zeros(B, 3), torch.tensor([[0.0, 0, 0, 1]]).repeat(B, 1),
                                torch.ones(B), sdf=torch.zeros(1, 8, 8, 8))
    with pytest.raises(ValueError):
        plain.result("best_inlier_ratio")


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,shared", [(48, 64, False), (37, 53, False), (48, 64, True)])
def test_inlier_count_kernel_is_exact(cuda_device, H, W, shared):
    from oracle import hypothesis_step as hs
    from sdfest_b200 import _lib

    lib, B, thr = _lib.lib(), 5, 0.03
    obs, est = _inlier_images(B, H, W, 7)
    if shared:
        obs = np.repeat(obs[:1], B, 0)
    d_obs = torch.tensor(obs[0] if shared else obs, device=cuda_device).contiguous()
    d_est = torch.tensor(est, device=cuda_device)
    counts = torch.full((2, B), 3.0, device=cuda_device)
    _lib.check(lib.sdfr_inlier_count(d_est.data_ptr(), d_obs.data_ptr(), 0 if shared else H * W, B, W, H, thr,
                                     counts[0].data_ptr(), counts[1].data_ptr(), _lib.ZERO_GRADS, None), "count")
    want = np.array([hs.inlier_counts(obs[b], est[b], thr) for b in range(B)], np.float32).T
    assert want[0].min() > 0 and (want[0] < want[1]).all()
    np.testing.assert_array_equal(counts.cpu().numpy(), want)
    # accumulates without the flag
    _lib.check(lib.sdfr_inlier_count(d_est.data_ptr(), d_obs.data_ptr(), 0 if shared else H * W, B, W, H, thr,
                                     counts[0].data_ptr(), counts[1].data_ptr(), 0, None), "count")
    np.testing.assert_array_equal(counts.cpu().numpy(), 2 * want)
    assert lib.sdfr_inlier_count(None, d_obs.data_ptr(), 0, B, W, H, thr, counts.data_ptr(), counts.data_ptr(), 0, None) == -1
    assert lib.sdfr_inlier_count(d_est.data_ptr(), d_obs.data_ptr(), 0, B, 0, H, thr, counts.data_ptr(), counts.data_ptr(), 0, None) == -2
    assert lib.sdfr_inlier_count(d_est.data_ptr(), d_obs.data_ptr(), 0, B, W, H, thr, counts.data_ptr(), counts.data_ptr(), 0x1, None) == -3


@pytest.mark.gpu
def test_track_best_kernel_matches_oracle(cuda_device):
    from oracle import hypothesis_step as hs
    from sdfest_b200 import _lib

    lib, B, L = _lib.lib(), 70, 5
    g = np.random.default_rng(3)
    dev = cuda_device
    pos, quat = torch.zeros(B, 3, device=dev), torch.zeros(B, 4, device=dev)
    scale, lat = torch.ones(B, device=dev), torch.zeros(B, L, device=dev)
    step = torch.zeros(B, dtype=torch.int32, device=dev)
    ratio, best_ratio = torch.zeros(B, device=dev), torch.full((B,), -1.0, device=dev)
    best_it = torch.full((B,), -1, dtype=torch.int32, device=dev)
    bp, bq, bs, bl = (torch.zeros_like(t) for t in (pos, quat, scale, lat))
    best = [hs.BestEstimate() for _ in range(B)]
    for it in range(1, 9):
        n_valid = g.integers(0, 3, B).astype(np.float32) * 50  # some hypotheses never see a valid pixel
        n_inl = np.floor(g.random(B) * n_valid).astype(np.float32)
        counts = torch.tensor(np.stack([n_inl, n_valid]), device=dev)
        for t in (pos, quat, scale, lat):
            t += torch.tensor(g.standard_normal(t.shape).astype(np.float32), device=dev)
        step += 1
        _lib.check(lib.sdfr_track_best(
            counts[0].data_ptr(), counts[1].data_ptr(), pos.data_ptr(), quat.data_ptr(), scale.data_ptr(),
            lat.data_ptr(), L, B, step.data_ptr(), ratio.data_ptr(), best_ratio.data_ptr(), best_it.data_ptr(),
            bp.data_ptr(), bq.data_ptr(), bs.data_ptr(), bl.data_ptr(), _lib.STEP_CLEAR_INPUTS, None), "track")
        assert float(counts.abs().max()) == 0.0
        cur = [t.cpu().numpy() for t in (pos, quat, scale, lat)]
        for b in range(B):
            r = best[b].update(n_inl[b], n_valid[b], it, [c[b] for c in cur])
            got = float(ratio[b])
            assert (np.isnan(r) and np.isnan(got)) or got == float(r)
    np.testing.assert_array_equal(best_it.cpu().numpy(), [e.iteration for e in best])
    for k, t in enumerate((bp, bq, bs, bl)):
        np.testing.assert_array_equal(t.cpu().numpy(), np.stack([e.params[k] for e in best]))
    assert lib.sdfr_track_best(None, None, None, None, None, None, 0, 1, None, None, None, None, None, None,
                               None, None, 0, None) == -1


@pytest.mark.gpu
@pytest.mark.parametrize("with_decoder", [False, True])
def test_fused_result_selection_matches_torch_composition(cuda_device, with_decoder):
    """inlier_ratio and the best estimate of the fused iteration (graph replay) against the torch path."""
    def make(optimizer):
        o = _make_optimizers(cuda_device, 6, with_decoder, optimizer)
        # same construction, with result selection switched on
        from sdfest_b200.estimation import HypothesisOptimizer
        kw = dict(latent=o.latent.detach(), decoder=o.decoder) if with_decoder else dict(sdf=o.sdf)
        return HypothesisOptimizer(o.camera, o.threshold, o.depth_obs, o.position.detach(), o.orientation.detach(),
                                   o.scale.detach(), optimizer=optimizer, inlier_threshold=0.03, **kw)

    a, b = make("torch"), make("fused")
    a.step()
    b.capture(warmup=1)
    torch.testing.assert_close(b.inlier_ratio, a.inlier_ratio, rtol=0, atol=1e-2)
    for _ in range(5):
        a.step()
        b.step()
        torch.cuda.synchronize()
        torch.testing.assert_close(b.inlier_ratio, a.inlier_ratio, rtol=0, atol=1e-2)
    assert float(b.inlier_ratio.max()) > 0.05
    assert int(b.best_iteration.min()) >= 1 and int(b._t.max()) == 6
    torch.testing.assert_close(b.best_inlier_ratio, a.best_inlier_ratio, rtol=0, atol=1e-2)
    same = (b.best_iteration == a.best_iteration)
    # a tie within a pixel or two can pick a neighbouring iteration; the snapshots of the others agree
    assert int(same.sum()) >= 3
    assert float((b.best_position[same] - a.best_position[same]).abs().max()) < 1e-3
    # the snapshot is a copy of the parameters of its iteration, not the live tensor
    moved = b.best_iteration < 6
    if bool(moved.any()):
        assert float((b.best_position[moved] - b.position[moved]).abs().max()) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("per_hypothesis_obs", [False, True])
def test_compare_fused_inliers_counts_in_the_same_traversal(cuda_device, per_hypothesis_obs):
    """sdfr_compare_fused_inliers = sdfr_compare_fused + the inlier count of sdfr_inlier_count on the
    depth it wrote (exactly), without a second pass."""
    from oracle import hypothesis_step as hs
    from sdfest_b200 import _lib

    lib, B, thr = _lib.lib(), 6, 0.03
    opt = _make_optimizers(cuda_device, B, False, "fused")
    cam, R = opt.camera, opt._R
    W, H = int(cam.width), int(cam.height)
    obs = opt.depth_obs
    if per_hypothesis_obs:
        obs = torch.stack([torch.roll(obs, k, 1) for k in range(B)]).contiguous()
        obs[1] = 0.0  # an observation without a valid pixel: ratio 0/0
    grids, gstride, layout = opt._grid_op
    dev = cuda_device
    outs = {}
    for name in ("plain", "inliers"):
        depth = torch.empty(B, H, W, device=dev)
        sums = torch.zeros(3, B, device=dev)
        gp, gq, gi = torch.zeros(B, 3, device=dev), torch.zeros(B, 4, device=dev), torch.zeros(B, device=dev)
        flags = _lib.GRAD_POSITION | _lib.GRAD_ORIENTATION | _lib.GRAD_INV_SCALE | _lib.ZERO_GRADS
        head = (grids.data_ptr(), R, gstride, layout, opt.position.data_ptr(), opt._unit_q.data_ptr(),
                opt._inv_scale.data_ptr(), B, W, H, W / 2, H / 2, W / 2, W / 2, opt.threshold, obs.data_ptr(),
                H * W if per_hypothesis_obs else 0, depth.data_ptr(), sums[0].data_ptr(), sums[1].data_ptr())
        tail = (None, 0, gp.data_ptr(), gq.data_ptr(), gi.data_ptr(), flags, None, None)  # ..., bounds, stream
        if name == "plain":
            _lib.check(lib.sdfr_compare_fused(*head, *tail), name)
        else:
            sums[2] = 7.0  # ZERO_GRADS clears the inlier counter too
            _lib.check(lib.sdfr_compare_fused_inliers(*head, thr, sums[2].data_ptr(), *tail), name)
        torch.cuda.synchronize()
        outs[name] = (depth, sums, gp, gq, gi)
    assert torch.equal(outs["plain"][0], outs["inliers"][0])
    torch.testing.assert_close(outs["plain"][1][:2], outs["inliers"][1][:2], rtol=1e-5, atol=0)
    for k in (2, 3, 4):
        torch.testing.assert_close(outs["plain"][k], outs["inliers"][k], rtol=1e-4, atol=1e-6)
    depth, sums = outs["inliers"][0], outs["inliers"][1]
    counts = torch.zeros(2, B, device=dev)
    _lib.check(lib.sdfr_inlier_count(depth.data_ptr(), obs.data_ptr(), H * W if per_hypothesis_obs else 0, B, W, H,
                                     thr, counts[0].data_ptr(), counts[1].data_ptr(), 0, None), "count")
    assert torch.equal(sums[2], counts[0])
    d, o = depth.cpu().numpy(), obs.cpu().numpy()
    want = [hs.inlier_counts(o[b] if per_hypothesis_obs else o, d[b], thr)[0] for b in range(B)]
    assert sums[2].tolist() == want and max(want) > 50
    # thresholds above 1 would have to count missed pixels: rejected
    assert lib.sdfr_compare_fused_inliers(*head, 1.5, sums[2].data_ptr(), *tail) == -2
    assert lib.sdfr_compare_fused_inliers(*head, thr, None, *tail) == -1


@pytest.mark.gpu
def test_result_selection_with_a_threshold_above_one_uses_the_separate_pass(cuda_device):
    from sdfest_b200.estimation import HypothesisOptimizer

    o = _make_optimizers(cuda_device, 4, False, "fused")

    def make(optimizer):
        return HypothesisOptimizer(o.camera, o.threshold, o.depth_obs, o.position.detach(), o.orientation.detach(),
                                   o.scale.detach(), sdf=o.sdf, optimizer=optimizer, inlier_threshold=1.5)

    a, b = make("torch"), make("fused")
    for _ in range(3):
        a.step()
        b.step()
    torch.cuda.synchronize()
    # every valid pixel is an inlier: missed ones have relative error 1 < 1.5
    torch.testing.assert_close(b.inlier_ratio, a.inlier_ratio, rtol=0, atol=1e-2)
    assert float(b.inlier_ratio.min()) > 0.9


@pytest.mark.gpu
def test_fused_optimizer_on_a_device_that_is_not_current(cuda_device):
    """Tensors on cuda:1 while cuda:0 is the current device: the fused iteration, its second stream, the
    captured graph and the autograd operators all run on the tensors' device (the library launches on the
    CURRENT device's stream and never calls cudaSetDevice, so the Python side must make it current) and
    give the results of the same optimiser built on cuda:0."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    torch.cuda.set_device(0)
    a = _make_optimizers(torch.device("cuda:0"), 4, True, "fused")
    b = _make_optimizers(torch.device("cuda:1"), 4, True, "fused")
    assert torch.cuda.current_device() == 0 and b.position.device.index == 1
    for _ in range(3):
        la, lb = a.step().clone(), b.step().clone()
    torch.testing.assert_close(lb.cpu(), la.cpu(), rtol=2e-3, atol=1e-5)
    b.capture(warmup=1)
    a.step(), a.step()
    lb = b.step().clone()
    torch.cuda.synchronize(1)
    torch.testing.assert_close(lb.cpu(), a.last_losses.cpu(), rtol=2e-3, atol=1e-5)
    assert torch.cuda.current_device() == 0
    t = _make_optimizers(torch.device("cuda:1"), 4, False, "torch")
    f = _make_optimizers(torch.device("cuda:1"), 4, False, "fused")
    torch.testing.assert_close(f.step().cpu(), t.step().cpu(), rtol=2e-3, atol=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("optimizer", ["fused", "torch"])
def test_a_hypothesis_without_overlap_never_ranks_best(cuda_device, optimizer):
    """One hypothesis far off-screen: its rendered depth never overlaps the observation.  The reference's mean
    over an empty selection is NaN (simple_setup.py:131) and so is the loss reported here -- it must not look
    like the best one (its depth and point terms are both 0) -- while its parameters and Adam state stay finite
    and the other hypotheses are unaffected."""
    from sdfest_b200 import _lib
    from sdfest_b200.estimation.hypotheses import global_best

    good = _make_optimizers(cuda_device, 4, False, optimizer)
    bad = _make_optimizers(cuda_device, 4, False, optimizer)
    with torch.no_grad():
        bad.position[2] += torch.tensor([5.0, 0.0, 0.0], device=cuda_device)  # out of the frustum
    if optimizer == "fused":
        bad._hyp_step(_lib.STEP_NO_UPDATE)
    for _ in range(3):
        lg, lb = good.step().clone(), bad.step().clone()
    assert bool(torch.isnan(lb[2])) and bool(torch.isfinite(lb[[0, 1, 3]]).all())
    torch.testing.assert_close(lb[[0, 1, 3]], lg[[0, 1, 3]], rtol=1e-5, atol=1e-7)
    for t in (bad.position, bad.orientation, bad.scale):
        assert bool(torch.isfinite(t.detach()).all())
    idx, loss = global_best(lb, 0)
    assert idx != 2 and loss == float(lb[idx]) and idx == int(torch.argmin(torch.nan_to_num(lg, nan=float("inf"))))
