"""Every detection of one frame in one call: SDFPipeline.estimate_instances against one __call__ per detection.

    python scripts/gpu_instances.py [out.json]

Workload: K in {1, 4, 8, 16} objects (64^3 grids decoded around an analytic mug, scale 0.1 m, on a 4x4 lattice
1.1 m in front of the camera, the first K lattice places) rendered into ONE 640x480 depth map with
render_depth_composite (Redwood camera: fx = fy = 525, cx = 319.5, cy = 239.5, pixel centre 0); detection k is
the mask winner == k.  The pipeline runs its defaults (50 iterations, CUDA graph, fused decoder tail) with
best-inlier-ratio selection.  The initialisation network is a per-input stand-in (a function of the set-wise
maximum of the centred cloud): a trained network is not part of this repository, and its cost is not what is
compared here.

(a) per K: K sequential __call__(depth, mask_k) against one estimate_instances(depth, masks), each on a new
    pipeline (first call: the optimiser is built and captured) and on a warmed one (reused graph: reset + replay);
(b) per K: the observed clouds of the K detections -- the torch loop (mask, far field and torch.nonzero per
    detection, as __call__ and depth_to_pointclouds did it) against one extract_instances call
    (sdfr_depth_to_points).
Times: host clock around work that ends in a device synchronise; median of the repetitions.  The card's name
and power limit are read in the same run.  Prints the result as JSON and, given a path, also writes it there.
"""
import json
import os
import statistics
import subprocess
import sys
import time

import torch
from torch import nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from sdfest_b200 import synthetic as syn  # noqa: E402
from sdfest_b200.differentiable_renderer import Camera, render_depth_composite  # noqa: E402
from sdfest_b200.estimation import SDFPipeline, losses  # noqa: E402

dev = torch.device("cuda:0")
W, H, R, THR, FAR = 640, 480, 64, 0.005, 3.0
CAMERA = dict(width=W, height=H, fx=525.0, fy=525.0, cx=319.5, cy=239.5, pixel_center=0.0)
CONFIG = {"device": str(dev), "camera": dict(CAMERA), "threshold": THR, "far_field": FAR,
          "init": {"backbone_type": "VanillaPointNet", "normalize_pose": True, "head": {"orientation_repr": "quaternion"}},
          "result_selection_strategy": "best_inlier_ratio"}


class VAE(nn.Module):
    def __init__(self, decoder):
        super().__init__()
        self.decoder = decoder

    def decode(self, z):
        return self.decoder(z)


class PointSetInit(nn.Module):
    """Deterministic per input: latent, offset and orientation from the set-wise maximum of the centred cloud."""

    def __init__(self):
        super().__init__()
        self.dummy = nn.Parameter(torch.zeros(1))
        self.base = (0.2 * torch.randn(1, 8, generator=torch.Generator().manual_seed(0))).to(dev)

    def forward(self, x):
        f = x.amax(1)
        q = torch.nn.functional.normalize(
            torch.tensor([[0.03, -0.02, 0.01, 1.0]], device=dev) + 0.1 * torch.cat([f, 0 * f[:, :1]], 1), dim=1)
        off = torch.tensor([[0.004, -0.003, -0.03]], device=dev) + 0.05 * f
        return self.base + 0.5 * f[:, :1], off, torch.full((x.shape[0],), 0.1, device=dev), q


def frame(dec, K):
    cam = Camera(**CAMERA)
    lattice = [(x, y) for y in (0.33, 0.11, -0.11, -0.33) for x in (-0.45, -0.15, 0.15, 0.45)]
    with torch.no_grad():
        z = 0.3 * torch.randn(K, 8, generator=torch.Generator().manual_seed(10)).to(dev)
        grids = dec(z)[:, 0].contiguous()
        pos = torch.tensor([[x, y, -1.1] for x, y in lattice[:K]], device=dev)
        quat = torch.tensor([[0.0, 0.0, 0.0, 1.0]] * K, device=dev)
        depth, winner = render_depth_composite(grids, pos, quat, torch.full((K,), 10.0, device=dev), THR, cam)
    masks = torch.stack([winner == k for k in range(K)])
    return depth.contiguous(), masks


def wall(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3, out


def torch_extraction(depth, masks, cam):
    """The per-detection torch loop: __call__'s in-place masking on a copy, then the nonzero() cloud."""
    fx, fy, cx, cy, _ = cam.get_pinhole_camera_parameters(0.0)
    clouds = []
    for m in masks:
        d = depth.clone()
        d[~m] = 0
        d[d > FAR] = 0
        rows, cols = torch.nonzero(d, as_tuple=True)
        z = d[rows, cols]
        clouds.append(torch.stack([(cols.float() - cx) * z / fx, -(rows.float() - cy) * z / fy, -z], dim=1))
    M = max(c.shape[0] for c in clouds)
    out = torch.full((len(clouds), M, 3), losses.PAD_COORDINATE, device=depth.device)
    for k, c in enumerate(clouds):
        out[k, :c.shape[0]] = c
    return out


def main(out_path):
    try:
        card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        card = f"nvidia-smi unavailable ({e})"
    dec = syn.residual_decoder(R, dev, syn.sdf_mug(R, dev))
    vae = VAE(dec)
    cam = Camera(**CAMERA)
    result = {"device": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit_max_sm_clock": card,
              "workload": "one 640x480 frame, K detections of 64^3 mugs composited, 50 iterations, best_inlier_ratio",
              "rows": []}
    for K in (1, 4, 8, 16):
        depth, masks = frame(dec, K)
        counts = [int(m.sum()) for m in masks]
        row = {"K": K, "points_per_detection": counts}

        def sequential(pipe):
            return [pipe(depth.clone(), masks[k], None) for k in range(K)]

        first_seq, first_inst = [], []
        for _ in range(3):
            first_seq.append(wall(lambda: sequential(SDFPipeline(CONFIG, vae, PointSetInit())))[0])
            first_inst.append(wall(lambda: SDFPipeline(CONFIG, vae, PointSetInit()).estimate_instances(depth, masks))[0])
        seq_pipe, inst_pipe = SDFPipeline(CONFIG, vae, PointSetInit()), SDFPipeline(CONFIG, vae, PointSetInit())
        sequential(seq_pipe)
        inst_pipe.estimate_instances(depth, masks)
        reused_seq, reused_inst = [], []
        for _ in range(10):
            t, per_call = wall(lambda: sequential(seq_pipe))
            reused_seq.append(t)
            t, batched = wall(lambda: inst_pipe.estimate_instances(depth, masks))
            reused_inst.append(t)
        diff = [max(float((b[k] - c[k][0]).abs().max()) for k in range(K)) for b, c in
                zip(batched, [[pc[i] for pc in per_call] for i in range(4)])]
        row["sequential_call_ms"] = {"first_call": statistics.median(first_seq), "reused_graph": statistics.median(reused_seq)}
        row["estimate_instances_ms"] = {"first_call": statistics.median(first_inst),
                                        "reused_graph": statistics.median(reused_inst)}
        row["speedup_reused_graph"] = statistics.median(reused_seq) / statistics.median(reused_inst)
        row["max_abs_diff_position_orientation_scale_latent"] = diff
        ref = torch_extraction(depth, masks, cam)
        _, pts, _ = losses.extract_instances(depth, masks, cam, FAR)
        assert torch.equal(ref, pts), "extract_instances differs from the torch loop"
        t_torch = statistics.median(wall(lambda: torch_extraction(depth, masks, cam))[0] for _ in range(50))
        t_kernel = statistics.median(wall(lambda: losses.extract_instances(depth, masks, cam, FAR))[0] for _ in range(50))
        row["extraction_ms"] = {"torch_loop": t_torch, "extract_instances": t_kernel}
        result["rows"].append(row)
        print(json.dumps(row), flush=True)
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else None)
