"""C1 (ONE 640x480 / 64^3 frame) as a latency problem: where the ~20 us of a single forward launch go.

  * the launch as shipped;
  * crops of the same frame rendered with a shifted principal point (identical rays): one 32x8 tile that
    holds the frame's longest sphere trace (43 samples; found with the CPU oracle, see DESIGN.md), one
    tile of box pixels that miss the surface after a few samples, one tile outside the box -- i.e. launch +
    CTA prologue + the longest dependent chain, launch + prologue + a short chain, launch + prologue;
  * the fused render + compare + backward launch at B = 1, the unfused backward, an empty kernel.

Writes gpurun_out/<tag>_c1_latency.json.  Timing: CUDA events around ONE call, median of 40, L2 flushed.
"""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from sdfest_b200 import _lib  # noqa: E402
from sdfest_b200 import synthetic as syn  # noqa: E402

W, H, R, THR = 640, 480, 64, 0.005
dev = torch.device("cuda:0")
lib = _lib.lib()
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
st = torch.cuda.current_stream().cuda_stream


def timed(fn, n=40, warm=5, do_flush=True):
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
    return {"median_us": round(ts[len(ts) // 2], 2), "min_us": round(ts[0], 2)}


hyp = syn.make_hypotheses(1, seed=0, device=dev)
grid = syn.hypothesis_grids(hyp["shape_param"], R, dev)[0].contiguous()
p, q, s = hyp["position"][0].clone(), hyp["orientation"][0].clone(), hyp["inv_scale"].clone()
g = torch.randn(H, W, device=dev)
depth = torch.empty(1, H, W, device=dev)
gs, gp, gq, gi = torch.empty_like(grid), torch.empty(3, device=dev), torch.empty(4, device=dev), torch.empty(1, device=dev)
sums = torch.zeros(2, 1, device=dev)


def fwd(w=W, h=H, x0=0, y0=0, layout=0, src=None):
    lib.sdfr_forward((src if src is not None else grid).data_ptr(), R, 0, layout, p.data_ptr(), q.data_ptr(),
                     s.data_ptr(), 1, w, h, 320.0 - x0, 240.0 - y0, 320.0, 320.0, THR, depth.data_ptr(), None, st)


def bwd(flags=_lib.GRAD_ALL | _lib.ZERO_GRADS):
    lib.sdfr_backward(g.data_ptr(), depth.data_ptr(), grid.data_ptr(), R, 0, 0, p.data_ptr(), q.data_ptr(),
                      s.data_ptr(), 1, W, H, 320.0, 240.0, 320.0, 320.0, gs.data_ptr(), 0, gp.data_ptr(),
                      gq.data_ptr(), gi.data_ptr(), flags, None, st)


out = {}
fwd()
torch.cuda.synchronize()
full = depth.clone()
obs = torch.roll(full[0], 3, 1).contiguous()  # a shifted copy of the render as the observation


def fused(flags=_lib.GRAD_ALL | _lib.ZERO_GRADS):
    lib.sdfr_compare_fused(grid.data_ptr(), R, 0, 0, p.data_ptr(), q.data_ptr(), s.data_ptr(), 1, W, H,
                           320.0, 240.0, 320.0, 320.0, THR, obs.data_ptr(), 0, depth.data_ptr(),
                           sums[0].data_ptr(), sums[1].data_ptr(), gs.data_ptr(), 0, gp.data_ptr(),
                           gq.data_ptr(), gi.data_ptr(), flags, None, st)


empty = torch.empty(1, device=dev)
out["empty_torch_kernel"] = timed(lambda: empty.zero_())
out["zero_small_only"] = timed(lambda: lib.sdfr_backward(None, None, grid.data_ptr(), R, 0, 0, p.data_ptr(),
                                                         q.data_ptr(), s.data_ptr(), 1, 0, 0, 320.0, 240.0, 320.0,
                                                         320.0, gs.data_ptr(), 0, gp.data_ptr(), gq.data_ptr(),
                                                         gi.data_ptr(), 0x0E | _lib.ZERO_GRADS, None, st))
out["forward"] = timed(fwd)
out["forward_warm_l2"] = timed(fwd, do_flush=False)
out["backward_incl_clears"] = timed(bwd)
out["backward_no_clears"] = timed(lambda: bwd(_lib.GRAD_ALL))
out["fused_compare_incl_clears"] = timed(fused)
out["fused_compare_no_clears"] = timed(lambda: fused(_lib.GRAD_ALL))
out["forward_then_backward"] = timed(lambda: (fwd(), bwd()))
# crops (tile coordinates from the oracle's step-count image of this scene: longest trace 43 samples in tile
# (11, 37); tile (5, 30) holds box pixels that miss; tile (0, 59) is outside the projected box)
for name, (tx, ty) in {"tile_longest_trace": (11, 37), "tile_box_miss": (5, 30), "tile_outside": (0, 59)}.items():
    out["crop_" + name] = timed(lambda tx=tx, ty=ty: fwd(32, 8, 32 * tx, 8 * ty))
    torch.cuda.synchronize()
    ref = full[0, 8 * ty:8 * ty + 8, 32 * tx:32 * tx + 32]
    got = depth.flatten()[:256].view(8, 32)
    out["crop_" + name]["max_abs_diff_vs_full_frame"] = float((ref - got).abs().max())
    out["crop_" + name]["hit_pixels"] = int((got > 0).sum())
# the rows of tiles through the object, 640 x 8 and 640 x 64
out["crop_rows_8"] = timed(lambda: fwd(640, 8, 0, 8 * 37))
out["crop_rows_64"] = timed(lambda: fwd(640, 64, 0, 8 * 30))
tag = sys.argv[1] if len(sys.argv) > 1 else "c1"
os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
with open(os.path.join(ROOT, "gpurun_out", f"{tag}_c1_latency.json"), "w") as f:
    json.dump(out, f, indent=1)
print(json.dumps(out, indent=1))
