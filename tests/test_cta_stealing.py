"""The forward kernels are scheduling independent.

A resident CTA of the forward / compare / fused kernels renders every logical CTA (a tile range of
one hypothesis) that it can cancel before the hardware launches it, so which CTA renders which
hypothesis changes from launch to launch.  None of that may show in the results: every pixel is
written, each hypothesis' depth is bit-identical to a launch of that hypothesis alone, the overlap
counts are exact, and nothing carries over from one CUDA-graph replay to the next.
"""
import ctypes

import pytest
import torch

from sdfest_b200 import _lib
from sdfest_b200 import synthetic as syn

W, H, THR = 640, 480, 0.005
CX, CY, FX, FY = 320.0, 240.0, 320.0, 320.0
# The loss sums and pose gradients are float sums whose grouping follows the CTA split, and a launch
# of one hypothesis splits its image into more CTAs than a batched launch does.
SUM_RTOL = 1e-5

CASES = [(B, 64, layout) for B in (1, 3, 64, 300) for layout in ("dense", "skewed")]
CASES += [(64, 32, "skewed"), (64, 24, "dense")]  # 24: run-time resolution (no compile-time pitches)


def _scene(dev, B, R, layout):
    lib = _lib.lib()
    hyp = syn.make_hypotheses(B, seed=11, device=dev)
    grids = syn.hypothesis_grids(hyp["shape_param"], R, dev)
    if layout == "skewed":
        n = ctypes.c_longlong(0)
        _lib.check(lib.sdfr_skewed_pitches(R, None, None, ctypes.byref(n)), "sdfr_skewed_pitches")
        stride = int(n.value)
        sdf = torch.empty(B, stride, device=dev)
        _lib.check(lib.sdfr_skew_grids(grids.data_ptr(), R, R ** 3, B, sdf.data_ptr(), stride,
                                       torch.cuda.current_stream().cuda_stream), "sdfr_skew_grids")
    else:
        sdf, stride = grids.reshape(B, -1).contiguous(), R ** 3
    base = syn.make_hypotheses(1, seed=11, device=dev)
    obs = torch.empty(1, H, W, device=dev)
    _lib.check(lib.sdfr_forward(syn.hypothesis_grids(base["shape_param"], R, dev).data_ptr(), R, R ** 3, 0,
                                base["position"].data_ptr(), base["orientation"].data_ptr(),
                                base["inv_scale"].data_ptr(), 1, W, H, CX, CY, FX, FY, THR, obs.data_ptr(),
                                None, torch.cuda.current_stream().cuda_stream), "sdfr_forward")
    return dict(sdf=sdf, stride=stride, R=R, layout=1 if layout == "skewed" else 0, obs=obs,
                pos=hyp["position"], quat=hyp["orientation"], inv=hyp["inv_scale"])


def _outputs(dev, B, R):
    nan = float("nan")
    return dict(depth=torch.full((B, H, W), nan, device=dev), loss=torch.full((B,), nan, device=dev),
                n=torch.full((B,), nan, device=dev), gsdf=torch.full((B, R ** 3), nan, device=dev),
                gpos=torch.zeros(B, 3, device=dev), gquat=torch.zeros(B, 4, device=dev),
                ginv=torch.zeros(B, device=dev))


def _forward(s, lo, hi, depth):
    _lib.check(_lib.lib().sdfr_forward(
        s["sdf"][lo:hi].data_ptr(), s["R"], s["stride"], s["layout"], s["pos"][lo:hi].data_ptr(),
        s["quat"][lo:hi].data_ptr(), s["inv"][lo:hi].data_ptr(), hi - lo, W, H, CX, CY, FX, FY, THR,
        depth.data_ptr(), None, torch.cuda.current_stream().cuda_stream), "sdfr_forward")


def _fused(s, lo, hi, o):
    """sdfr_compare_fused of hypotheses lo..hi-1; SDFR_ZERO_GRADS clears every accumulator first."""
    _lib.check(_lib.lib().sdfr_compare_fused(
        s["sdf"][lo:hi].data_ptr(), s["R"], s["stride"], s["layout"], s["pos"][lo:hi].data_ptr(),
        s["quat"][lo:hi].data_ptr(), s["inv"][lo:hi].data_ptr(), hi - lo, W, H, CX, CY, FX, FY, THR,
        s["obs"].data_ptr(), 0, o["depth"].data_ptr(), o["loss"].data_ptr(), o["n"].data_ptr(),
        o["gsdf"].data_ptr(), s["R"] ** 3, o["gpos"].data_ptr(), o["gquat"].data_ptr(), o["ginv"].data_ptr(),
        _lib.GRAD_ALL | _lib.ZERO_GRADS, None, torch.cuda.current_stream().cuda_stream), "sdfr_compare_fused")


def _close(a, b, what):
    scale = float(b.abs().max())
    err = float((a - b).abs().max())
    assert err <= SUM_RTOL * scale, f"{what}: max |diff| {err:.3g} against max |value| {scale:.3g}"


def _same_fused(a, b, what):
    assert not torch.isnan(a["depth"]).any(), f"{what}: unwritten depth pixels"
    assert torch.equal(a["depth"], b["depth"]), f"{what}: depth"
    assert torch.equal(a["n"], b["n"]), f"{what}: n_overlap"
    for k in ("loss", "gpos", "gquat", "ginv", "gsdf"):
        _close(a[k], b[k], f"{what}: {k}")


@pytest.mark.gpu
@pytest.mark.parametrize("B,R,layout", CASES)
def test_batched_launch_equals_one_launch_per_hypothesis(cuda_device, B, R, layout):
    s = _scene(cuda_device, B, R, layout)
    depth = torch.full((B, H, W), float("nan"), device=cuda_device)
    _forward(s, 0, B, depth)
    batched = _outputs(cuda_device, B, R)
    _fused(s, 0, B, batched)
    alone = _outputs(cuda_device, B, R)
    for b in range(B):
        one_depth = torch.full((1, H, W), float("nan"), device=cuda_device)
        _forward(s, b, b + 1, one_depth)
        assert torch.equal(depth[b], one_depth[0]), f"forward depth of hypothesis {b}"
        one = _outputs(cuda_device, 1, R)
        _fused(s, b, b + 1, one)
        for k in alone:
            alone[k][b] = one[k][0]
    torch.cuda.synchronize()
    assert not torch.isnan(depth).any(), "forward: unwritten depth pixels"
    assert torch.equal(depth, batched["depth"]), "forward and fused depth"
    _same_fused(batched, alone, "batched against one launch per hypothesis")


@pytest.mark.gpu
@pytest.mark.parametrize("B,R,layout", [(64, 64, "skewed"), (300, 64, "dense")])
def test_graph_replays_are_independent(cuda_device, B, R, layout):
    """Replaying the captured fused launch twice gives the eager launch's results each time."""
    s = _scene(cuda_device, B, R, layout)
    eager = _outputs(cuda_device, B, R)
    _fused(s, 0, B, eager)
    replayed = _outputs(cuda_device, B, R)
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(stream):
        _fused(s, 0, B, replayed)  # warm-up on the capture stream
        torch.cuda.synchronize()
        with torch.cuda.graph(graph, stream=stream):
            replayed["depth"].fill_(float("nan"))
            _fused(s, 0, B, replayed)
    for i in range(2):
        for k in ("loss", "n", "gsdf", "gpos", "gquat", "ginv"):
            replayed[k].fill_(float("nan") if k in ("loss", "n", "gsdf") else 0.0)
        graph.replay()
        torch.cuda.synchronize()
        _same_fused(replayed, eager, f"replay {i}")
