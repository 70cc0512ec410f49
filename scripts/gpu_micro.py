"""GPU micro-measurements that guide kernel work (not a bench line):
  1. C1: one 640x480 / 64^3 frame forward+backward, ours vs the reference CUDA extension;
  2. C2 kernels (64 hypotheses) in the dense and skewed layouts.
Writes JSON to gpurun_out/<tag>_micro.json."""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from sdfest_b200 import _lib  # noqa: E402
from sdfest_b200 import synthetic as syn  # noqa: E402
from sdfest_b200.differentiable_renderer import Camera, render_depth_gpu  # noqa: E402

W, H, R, THR = 640, 480, 64, 0.005
dev = torch.device("cuda:0")
cam = Camera(W, H, 320.0, 320.0, 320.0, 240.0, pixel_center=0.5)
lib = _lib.lib()
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def timed(fn, n=30, warm=5, do_flush=True):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(n):
        if do_flush:
            flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    ts.sort()
    return {"median_us": ts[len(ts) // 2], "min_us": ts[0]}


out = {}
# ---- 1. single frame --------------------------------------------------------------------
hyp = syn.make_hypotheses(1, seed=0, device=dev)
grid = syn.hypothesis_grids(hyp["shape_param"], R, dev)[0].contiguous()
p, q, s = hyp["position"][0].clone(), hyp["orientation"][0].clone(), hyp["inv_scale"].clone()
g = torch.randn(H, W, device=dev)


def ours_single():
    a = [grid.detach().requires_grad_(True), p.detach().requires_grad_(True),
         q.detach().requires_grad_(True), s.detach().requires_grad_(True)]
    d = render_depth_gpu(*a, threshold=THR, camera=cam)
    d.backward(g)


depth1 = torch.empty(1, H, W, device=dev)
gs, gp, gq, gi = torch.empty_like(grid), torch.empty(3, device=dev), torch.empty(4, device=dev), torch.empty(1, device=dev)
st = torch.cuda.current_stream().cuda_stream


def ours_single_cabi():
    lib.sdfr_forward(grid.data_ptr(), R, 0, 0, p.data_ptr(), q.data_ptr(), s.data_ptr(), 1, W, H,
                     320.0, 240.0, 320.0, 320.0, THR, depth1.data_ptr(), None, st)
    lib.sdfr_backward(g.data_ptr(), depth1.data_ptr(), grid.data_ptr(), R, 0, 0, p.data_ptr(),
                      q.data_ptr(), s.data_ptr(), 1, W, H, 320.0, 240.0, 320.0, 320.0,
                      gs.data_ptr(), 0, gp.data_ptr(), gq.data_ptr(), gi.data_ptr(),
                      _lib.GRAD_ALL | _lib.ZERO_GRADS, None, st)


out["c1_ours_autograd"] = timed(ours_single)
try:  # the same autograd call captured once and replayed (no host work per call)
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            ours_single()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    c1_graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(c1_graph):
        ours_single()
    out["c1_ours_autograd_cuda_graph"] = timed(c1_graph.replay)
except Exception as e:  # noqa: BLE001
    out["c1_ours_autograd_cuda_graph"] = {"unavailable": str(e)[:300]}
out["c1_ours_cabi"] = timed(ours_single_cabi)
out["c1_ours_cabi_warm_l2"] = timed(ours_single_cabi, do_flush=False)
try:
    from oracle import build_ref

    ext = build_ref.load_module()

    def ref_single():
        (d,) = ext.forward(grid, p, q, s, W, H, 320.0, 240.0, 320.0, 320.0, THR)
        ext.backward(g, d, grid, p, q, s, W, H, 320.0, 240.0, 320.0, 320.0)

    out["c1_reference_ext"] = timed(ref_single)
    out["c1_reference_ext_warm_l2"] = timed(ref_single, do_flush=False)
except Exception as e:  # noqa: BLE001
    out["c1_reference_ext"] = {"unavailable": str(e)}

# ---- 2. C2 kernels vs CTA count ---------------------------------------------------------------
B = 64
hyp = syn.make_hypotheses(B, seed=0, device=dev)
grids = syn.hypothesis_grids(hyp["shape_param"], R, dev)
pos, quat, inv_s = hyp["position"], hyp["orientation"], hyp["inv_scale"]
depth = torch.empty(B, H, W, device=dev)
sums = torch.zeros(2, B, device=dev)
obs = torch.empty(H, W, device=dev)
lib.sdfr_forward(grids.data_ptr(), R, 0, 0, pos.data_ptr(), quat.data_ptr(), inv_s.data_ptr(), 1, W, H,
                 320.0, 240.0, 320.0, 320.0, THR, obs.data_ptr(), None, st)
g_sdf = torch.empty_like(grids)
g_pos, g_quat, g_is = torch.empty_like(pos), torch.empty_like(quat), torch.empty_like(inv_s)
RRR = R ** 3


import ctypes

n_sk = ctypes.c_longlong(0)
lib.sdfr_skewed_pitches(R, None, None, ctypes.byref(n_sk))
SK = int(n_sk.value)
skewed = torch.empty(B, SK, device=dev)
lib.sdfr_skew_grids(grids.data_ptr(), R, RRR, B, skewed.data_ptr(), SK, st)


bounds = torch.empty(B, 8, dtype=torch.int32, device=dev)
lib.sdfr_grid_bounds(skewed.data_ptr(), R, SK, 1, pos.data_ptr(), inv_s.data_ptr(), B, THR, bounds.data_ptr(), st)
USE_BOUNDS = [True]


def bptr():
    return bounds.data_ptr() if USE_BOUNDS[0] else None


def src(layout):
    return (skewed.data_ptr(), SK, 1) if layout else (grids.data_ptr(), RRR, 0)


def fwd(layout=1):
    ptr, stride, lt = src(layout)
    lib.sdfr_compare_forward(ptr, R, stride, lt, pos.data_ptr(), quat.data_ptr(),
                             inv_s.data_ptr(), B, W, H, 320.0, 240.0, 320.0, 320.0, THR,
                             obs.data_ptr(), 0, depth.data_ptr(), sums[0].data_ptr(),
                             sums[1].data_ptr(), _lib.ZERO_GRADS, bptr(), st)


def fused(layout=1, flags=_lib.GRAD_ALL | _lib.ZERO_GRADS):
    ptr, stride, lt = src(layout)
    lib.sdfr_compare_fused(ptr, R, stride, lt, pos.data_ptr(), quat.data_ptr(),
                           inv_s.data_ptr(), B, W, H, 320.0, 240.0, 320.0, 320.0, THR,
                           obs.data_ptr(), 0, depth.data_ptr(), sums[0].data_ptr(),
                           sums[1].data_ptr(), g_sdf.data_ptr(), RRR, g_pos.data_ptr(),
                           g_quat.data_ptr(), g_is.data_ptr(), flags, bptr(), st)


def bwd(layout=1, flags=_lib.GRAD_ALL | _lib.ZERO_GRADS):
    ptr, stride, lt = src(layout)
    lib.sdfr_compare_backward(depth.data_ptr(), obs.data_ptr(), 0, sums[1].data_ptr(), None,
                              ptr, R, stride, lt, pos.data_ptr(), quat.data_ptr(),
                              inv_s.data_ptr(), B, W, H, 320.0, 240.0, 320.0, 320.0,
                              g_sdf.data_ptr(), RRR, g_pos.data_ptr(), g_quat.data_ptr(),
                              g_is.data_ptr(), flags, bptr(), st)


fwd()
out["c2_layouts"] = {
    "skew_pass": timed(lambda: lib.sdfr_skew_grids(grids.data_ptr(), R, RRR, B, skewed.data_ptr(), SK, st)),
    "fwd_dense": timed(lambda: fwd(0)), "fwd_skewed": timed(lambda: fwd(1)),
    "fused_dense": timed(lambda: fused(0)), "fused_skewed": timed(lambda: fused(1)),
    "fused_skewed_pose_only": timed(lambda: fused(1, 0x0E | _lib.ZERO_GRADS)),
    "fused_skewed_sdf_only": timed(lambda: fused(1, 0x01 | _lib.ZERO_GRADS)),
    "bwd_dense": timed(lambda: bwd(0)), "bwd_skewed": timed(lambda: bwd(1)),
    "bwd_skewed_pose_only": timed(lambda: bwd(1, 0x0E | _lib.ZERO_GRADS)),
    "bwd_skewed_sdf_only": timed(lambda: bwd(1, 0x01 | _lib.ZERO_GRADS)),
    "bwd_skewed_no_memset": timed(lambda: bwd(1, _lib.GRAD_ALL)),
}
tag = sys.argv[1] if len(sys.argv) > 1 else "micro"
os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
with open(os.path.join(ROOT, "gpurun_out", f"{tag}_micro.json"), "w") as f:
    json.dump(out, f, indent=1)
print(json.dumps(out, indent=1))
