#!/usr/bin/env python
"""Benchmark of the render-and-compare hot path (BASELINE.json metric / config 2).

    python bench.py [--gpus N] [--steps K] [--warmup W]          # this repo's sm_100a kernels
    python bench.py --impl reference [...]                        # CPU reference arm (oracle port)
    torchrun --nproc-per-node N bench.py --gpus N ...             # one rank per GPU, weak scaling

A STEP is one pass of the hot path over one batch of synthetic input: `--hypotheses` (64) pose /
shape hypotheses, each with its own 64^3 SDF grid, rendered at 640x480 (fx=fy=320, threshold
0.005: estimation/configs/default.yaml:1-9), compared with one observed depth map through the
masked L1 of the reference pipeline (estimation/simple_setup.py:125-131), and back-propagated to
the SDF grids, positions, quaternions and inverse scales.  metric = pixels rendered forward+backward
per second (all pixels of all hypotheses, misses included -- SURVEY.md section 8d).

One JSON line is printed by rank 0 (see README / DESIGN.md for the keys).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

W, H, FX, FY, CX, CY = 640, 480, 320.0, 320.0, 320.0, 240.0  # default.yaml:1-8 (pixel_center 0.5)
R = 64
THRESHOLD = 0.005
METRIC = "depth-render fwd+bwd Mpix/s (640x480, 64^3)"
UNIT = "Mpix/s"
L2_FLUSH_BYTES = 256 << 20


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, help="timed steps of c2 and of the reference arm (default 50)")
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--hypotheses", type=int, default=64, help="hypotheses per GPU (weak scaling)")
    p.add_argument("--cpu-sample", type=int, default=32,
                   help="hypotheses per step rendered by the cpu_baseline leg of the GPU arm (the "
                        "--impl reference arm renders all --hypotheses, the arm's own config)")
    p.add_argument("--e2e-chunk", type=int, default=8, help="hypotheses per pipelined chunk (e2e)")
    p.add_argument("--no-ref-ext", action="store_true",
                   help="skip timing the reference CUDA extension (oracle/_ref) beside ours")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--gather-every", type=int, default=10,
                   help="multi-GPU: steps per exchange -- every step's per-hypothesis losses are kept in a ring on "
                        "the device and all-gathered as one [K, hypotheses] block every K steps (1 = every step)")
    p.add_argument("--no-step-graph", action="store_true",
                   help="issue the step's launches one by one instead of replaying them as one CUDA graph")
    p.add_argument("--min-time", type=float, default=0.0,
                   help="raise --steps so that the timed region lasts at least this many seconds (0 = time "
                        "exactly --steps steps, the driver's contract)")
    p.add_argument("--workload", "--config", dest="workload", default="c2", choices=["c1", "c2", "c3", "c4", "c5"],
                   help="c2 (default) is the configuration the metric is quoted on and the only one with the "
                        "full contract line; c1 / c3 / c4 / c5 run BASELINE.json's other configurations "
                        "(scripts/gpu_configs.py, scripts/gpu_sweep.py) and print their result as one line")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="c2: write what the last timed step computed (rank 0) as DIR/<name>.npy, float32; "
                        "see dump_outputs()")
    args = p.parse_args()
    if args.steps is not None and args.impl == "ours" and args.workload != "c2":
        p.error("--steps applies to c2 and to --impl reference; c1 / c3 / c4 / c5 time their scripts' own counts")
    args.steps = 50 if args.steps is None else args.steps
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "c2"):
        p.error("--dump-outputs needs --impl ours --workload c2")
    return args


def workload_name(B):
    return (f"C2: {B} pose/shape hypotheses x {W}x{H} depth, one {R}^3 fp32 SDF grid per hypothesis, "
            "fused render + masked-L1 compare forward and backward (all four gradients)")  # unchanged name: the
    # driver compares `config` between the two arms


def config_object(B, distributed):
    """`config` of the JSON line -- identical for both arms (the driver compares them)."""
    return {"workload": workload_name(B), "hypotheses_per_gpu": B, "width": W, "height": H,
            "resolution": R, "threshold": THRESHOLD, "sdf": "analytic mug grids, one per hypothesis",
            "l2": f"flushed before every timed step ({L2_FLUSH_BYTES >> 20} MiB memset, outside the event pair)",
            "collective": ("all_gather of per-hypothesis losses (async, overlapped with the next step)"
                           if distributed else "none")}


# kernels each C-ABI entry point of the timed step launches (memset nodes are not counted); checked
# against the ncu launch list of this command (profiles/*_launches.csv)
KERNELS_PER_CALL = {
    "sdfr_skew_grids_bounds": 2,  # sdfr_bounds_init_kernel, sdfr_bounds_scan_kernel<true>
    "sdfr_compare_fused": 1,      # sdfr_forward_kernel<64, skewed, 2> (the step clears the outputs with memset nodes)
    "sdfr_scale_grads": 1,        # sdfr_scale_grads_kernel
}


def algorithmic_bytes(S, P, B, RRR, hits, n_over):
    """SURVEY 8d: 32 B per trilinear sample, depth store, observation read at hits, grid read once; fused
    backward: 32 B corner re-read + 64 B read-modify-write per overlap pixel, gradient grid written once."""
    fwd = 32 * S + 4 * P * B + 4 * RRR * B + 4 * hits
    bwd = 4 * P * B + 4 * hits + 32 * n_over + 64 * n_over + 4 * RRR * B
    fused = fwd + 32 * n_over + 64 * n_over + 4 * RRR * B
    return fwd, bwd, fused


def gather_peaks():
    """Pure-gather rates of this GPU type for the renderer's access pattern (scripts/micro/gather_peaks.cu,
    measured on the pool's B200s and committed): the L1 / L2 denominators MEASURED_PEAKS.json lacks."""
    try:
        with open(os.path.join(ROOT, "profiles", "gather_peaks.json")) as f:
            d = json.load(f)
        return {"l1_skewed_gsamples": d["coherent_l1_skewed_ldg32"]["gsamples_per_s"],
                "l2_skewed_gsamples": d["coherent_l2only_skewed_ldg32"]["gsamples_per_s"],
                "source": "profiles/gather_peaks.json (scripts/micro/gather_peaks.cu)"}
    except Exception:
        return None


def roofline_object(fused_bytes, fused_ms, S, peak, peak_src, traffic, peaks=None):
    """The contract's `roofline` keys for the dominant kernel, plus the gather-rate view of the same
    launch: the 32*S term never leaves L1/L2 (ncu: 88 % L1 hit rate, DRAM at 8 %), so the HBM fraction
    says how the kernel compares with a copy of its algorithmic bytes, and `gather` says how close it is
    to what the memory pipes can deliver for this access pattern."""
    achieved = fused_bytes / (fused_ms * 1e-3) / 1e9
    out = {
        "bound": "hbm", "kernel": "sdfr_forward_kernel<64, skewed, MODE=2> (fused render+compare+backward, incl. its memsets)",
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
        "peak_source": peak_src, "algorithmic_bytes_per_launch": fused_bytes, "launch_ms": fused_ms,
        "note": ("algorithmic bytes = SURVEY 8d formula (32 B per trilinear sample + compulsory image/grid "
                 "traffic); the 32*S gather term is served by L1/L2 (traffic is the ncu DRAM figure: ~0.15x "
                 "of the algorithmic bytes), so frac is against the HBM copy peak, not a claim of HBM "
                 "traffic; `gather` compares the same launch with pure-gather kernels"),
    }
    gs = S / (fused_ms * 1e-3) / 1e9
    g = {"achieved_gsamples_per_s": gs, "achieved_GBps": 32 * gs}
    if peaks:
        g.update({"l1_peak_gsamples_per_s": peaks["l1_skewed_gsamples"],
                  "l2_peak_gsamples_per_s": peaks["l2_skewed_gsamples"],
                  "frac_of_l1_gather_peak": gs / peaks["l1_skewed_gsamples"],
                  "frac_of_l2_gather_peak": gs / peaks["l2_skewed_gsamples"], "peak_source": peaks["source"],
                  "limiter": "dependent-gather latency + issue slots (ncu: issue 58 %, L1 wavefronts 59 %, "
                             "L2 20 %, DRAM 8 %): neither L2 nor HBM bandwidth"})
    out["gather"] = g
    return out


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel`, from the committed ncu
    capture of this same command (profiles/ncu_traffic.json); None when there is no capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f)[kernel]["dram_bytes_per_launch"]
    except Exception:
        return None


DUMP_SAMPLE = 1 << 22  # elements kept of a larger output (depth: 19.7 M, grad_sdf: 16.8 M at 64 hypotheses)
DUMP_LIMIT = 64_000_000  # bytes written by one dump


def dump_outputs(out_dir, outputs):
    """Write each array of `outputs` (name -> array) as out_dir/<name>.npy in float32, so that two builds
    can be compared output for output.  An array of more than DUMP_SAMPLE elements is written as the 1-D
    array of its elements at DUMP_SAMPLE flat indices drawn without replacement by numpy's
    default_rng(0), in ascending index order: the same positions in every run with the same arguments."""
    import numpy as np

    arrays = {}
    for name, a in outputs.items():
        a = np.ascontiguousarray(a, dtype=np.float32)
        if a.size > DUMP_SAMPLE:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))]
        arrays[name] = a
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the limit of {DUMP_LIMIT}")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------
# clocks: sampled through NVML while the timed region runs
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.002)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ---------------------------------------------------------------------------------------------
# CPU reference arm: the oracle port of the reference renderer on the host cores
# ---------------------------------------------------------------------------------------------
def cpu_step(oracle, grids, pos, quat, inv_s, obs, nthreads):
    """Forward render + masked L1 + backward for every hypothesis in the sample."""
    import numpy as np

    total = 0.0
    for b in range(grids.shape[0]):
        d = oracle.render(grids[b], pos[b], quat[b], inv_s[b], W, H, CX, CY, FX, FY, THRESHOLD,
                          nthreads=nthreads)
        loss, g, n = oracle.l1_depth_loss(d, obs)
        bw = oracle.render_backward(g.astype(np.float32), d, grids[b], pos[b], quat[b], inv_s[b],
                                    W, H, CX, CY, FX, FY, sdf_grad_mode="reference",
                                    nthreads=nthreads)
        total += loss + float(bw["g_inv_scale"])
    return total


def cpu_inputs(sample):
    from sdfest_b200 import synthetic as syn

    hyp = syn.make_hypotheses(sample, seed=0)
    grids = syn.hypothesis_grids(hyp["shape_param"], R, "cpu").numpy()
    return grids, hyp["position"].numpy(), hyp["orientation"].numpy(), hyp["inv_scale"].numpy()


def time_cpu(sample, steps, warmup):
    import oracle

    nthreads = os.cpu_count() or 1
    grids, pos, quat, inv_s = cpu_inputs(sample)
    obs = oracle.render(grids[0], pos[0], quat[0], inv_s[0], W, H, CX, CY, FX, FY, THRESHOLD,
                        nthreads=nthreads)
    for _ in range(warmup):
        cpu_step(oracle, grids, pos, quat, inv_s, obs, nthreads)
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_step(oracle, grids, pos, quat, inv_s, obs, nthreads)
    dt = time.perf_counter() - t0
    mpix = sample * W * H * steps / dt / 1e6
    return mpix, dt / steps * 1e3, nthreads


def run_reference_arm(args, rank):
    if rank != 0:
        return
    # the arm's own config: every step renders ALL hypotheses of the workload (64 x 640x480 is ~0.25 s of
    # CPU work per step on 16 threads); steps / warm-up as given (same floor of 3 warm-up steps as the GPU arm)
    steps = args.steps
    warmup = max(args.warmup, 3)
    sample = args.hypotheses
    mpix, ms, cores = time_cpu(sample, steps, warmup)
    desc = (f"all {sample} hypotheses of one step per timed step "
            f"(forward + masked L1 + backward through oracle/liboracle.so, OpenMP over image rows)")
    line = {
        "impl": "reference", "metric": METRIC, "value": mpix, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_object(args.hypotheses, int(os.environ.get("WORLD_SIZE", "1")) > 1),
        "cpu_baseline": {"value": mpix, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": mpix, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": ("the reference's CPU renderer is pure Python (simple_renderer.py, ~8 kpix/s) and "
                 "cannot travel to the GPU box; this arm times its C restatement (oracle/) on all "
                 "host cores"),
    }
    emit(line)


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else (NCCL's version banner, library
    chatter) was diverted to stderr by divert_stdout()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def divert_stdout():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def run_other_workload(args, rank, world):
    """BASELINE.json's configurations 1, 3, 4, 5 through their measurement scripts (parity for them lives in
    tests/test_bench_parity.py and tests/test_dropin_reference.py); one JSON line on rank 0."""
    import runpy

    tag = f"bench_{args.workload}"
    if args.workload == "c4":
        script, out_file, key = "gpu_sweep.py", f"{tag}_sweep_n{world}.json", None
    else:
        script, out_file, key = "gpu_configs.py", f"{tag}_configs_n{world}.json", args.workload
        for k in ("c1", "c3", "c5"):
            if k != args.workload:
                os.environ[f"SKIP_{k.upper()}"] = "1"
    sys.argv = [os.path.join(ROOT, "scripts", script), tag]
    runpy.run_path(sys.argv[0], run_name="__main__")
    if rank != 0:
        return
    with open(os.path.join(ROOT, "gpurun_out", out_file)) as f:
        res = json.load(f)
    res = res[key] if key else res
    metric = {
        # the step replayed as one CUDA graph when the capture succeeded, else the eager autograd call
        "c1": ("depth-render fwd+bwd of one frame behind the decoder",
               res.get("fused_tail_decoder_our_renderer_cuda_graph", {}).get("mpix_per_s")
               or res.get("fused_tail_decoder_our_renderer", {}).get("mpix_per_s"), "Mpix/s"),
        "c3": ("composite frame fwd+bwd", res.get("mpix_per_s"), "Mpix/s"),
        "c4": ("hypothesis sweep", res.get("hyp_iter_per_s"), "hypothesis-iterations/s"),
        "c5": ("analysis-by-synthesis loop", res.get("instance_iter_per_s"), "instance-iterations/s"),
    }[args.workload]
    metric, value, unit = metric
    emit({"metric": metric, "value": value, "unit": unit, "n_gpus": world,
          "higher_is_better": True, "data": "synthetic", "dtype": "f32", "vs_baseline": None,
          "config": {"workload": res.get("workload", args.workload)}, "result": res})


def main():
    args = parse_args()
    divert_stdout()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if args.workload != "c2":
        run_other_workload(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    from sdfest_b200 import _lib, build
    from sdfest_b200 import synthetic as syn
    from sdfest_b200.differentiable_renderer import Camera, forward_stats, render_and_compare

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    distributed = world > 1
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    build.build()
    lib = _lib.lib()

    B = args.hypotheses
    cam = Camera(W, H, FX, FY, CX, CY, pixel_center=0.5)
    hyp = syn.make_hypotheses(B, seed=rank, device=dev)
    grids = syn.hypothesis_grids(hyp["shape_param"], R, dev)
    pos, quat, inv_s = hyp["position"], hyp["orientation"], hyp["inv_scale"]
    # observed depth = render of the unperturbed hypothesis of rank 0's seed (SURVEY 8d, C2)
    from sdfest_b200.differentiable_renderer import render_depth_batched

    base = syn.make_hypotheses(1, seed=0, device=dev)
    obs = render_depth_batched(syn.hypothesis_grids(base["shape_param"], R, dev), base["position"],
                               base["orientation"], base["inv_scale"], THRESHOLD, cam)[0].contiguous()

    stats_full = forward_stats(grids, pos, quat, inv_s, THRESHOLD, cam)
    stats = forward_stats(grids, pos, quat, inv_s, THRESHOLD, cam, empty_space=True)
    S, Hh_all = stats["samples"], stats["hit_pixels"]
    P = W * H

    depth = torch.empty(B, H, W, device=dev)
    # the per-hypothesis sums and the three pose-gradient outputs in ONE allocation (one clear per step)
    small = torch.zeros(10 * B, device=dev)
    sums = small[:2 * B].view(2, B)
    g_pos, g_quat, g_is = small[2 * B:5 * B].view(B, 3), small[5 * B:9 * B].view(B, 4), small[9 * B:]
    g_sdf = torch.empty_like(grids)
    clear_stream = torch.cuda.Stream(dev)
    Kg = max(1, args.gather_every) if distributed else 1
    ring = torch.zeros(Kg, 2, B, device=dev)  # loss_sum / n_overlap of the last Kg steps
    gathered2 = torch.empty(2, world * Kg * B, device=dev) if distributed else None
    loss2 = torch.empty(2, Kg, B, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    RRR = R * R * R
    flags_b = _lib.GRAD_ALL | _lib.ZERO_GRADS

    import ctypes

    n_sk = ctypes.c_longlong(0)
    _lib.check(lib.sdfr_skewed_pitches(R, None, None, ctypes.byref(n_sk)), "sdfr_skewed_pitches")
    SK = int(n_sk.value)
    skewed = torch.empty(B, SK, device=dev)

    cur_stream = [stream]  # the raw stream the step's launches go to (the capture stream while capturing)

    def skew():
        # dense decoder-layout grids -> bank-conflict-free pitched copy (one streaming pass); part
        # of every step because the grids change every iteration when the latent is optimised
        _lib.check(lib.sdfr_skew_grids(grids.data_ptr(), R, RRR, B, skewed.data_ptr(), SK, cur_stream[0]),
                   "sdfr_skew_grids")

    bounds = torch.empty((B, 8), dtype=torch.int32, device=dev)

    def bound():
        # empty-space bounds of the skewed grids for this step's poses (sdfr_grid_bounds): rays that
        # cannot hit anything are written as 0 without marching; every other ray is marched exactly as
        # the reference marches it.  Part of every step for the same reason as the layout pass.
        _lib.check(lib.sdfr_grid_bounds(skewed.data_ptr(), R, SK, _lib.LAYOUT_SKEWED, pos.data_ptr(),
                                        inv_s.data_ptr(), B, THRESHOLD, bounds.data_ptr(), cur_stream[0]),
                   "sdfr_grid_bounds")

    def skew_bound():
        # layout pass and bounds pass as ONE read of the dense grids (sdfr_skew_grids_bounds)
        _lib.check(lib.sdfr_skew_grids_bounds(grids.data_ptr(), R, RRR, B, skewed.data_ptr(), SK, pos.data_ptr(),
                                              inv_s.data_ptr(), THRESHOLD, bounds.data_ptr(), cur_stream[0]),
                   "sdfr_skew_grids_bounds")

    def fwd():
        _lib.check(lib.sdfr_compare_forward(
            skewed.data_ptr(), R, SK, _lib.LAYOUT_SKEWED, pos.data_ptr(), quat.data_ptr(),
            inv_s.data_ptr(), B, W, H, CX, CY, FX, FY, THRESHOLD, obs.data_ptr(), 0,
            depth.data_ptr(), sums[0].data_ptr(), sums[1].data_ptr(), _lib.ZERO_GRADS, bounds.data_ptr(), cur_stream[0]),
            "sdfr_compare_forward")

    def bwd():
        _lib.check(lib.sdfr_compare_backward(
            depth.data_ptr(), obs.data_ptr(), 0, sums[1].data_ptr(), None, skewed.data_ptr(), R,
            SK, _lib.LAYOUT_SKEWED, pos.data_ptr(), quat.data_ptr(), inv_s.data_ptr(), B, W, H,
            CX, CY, FX, FY, g_sdf.data_ptr(), RRR, g_pos.data_ptr(), g_quat.data_ptr(),
            g_is.data_ptr(), flags_b, bounds.data_ptr(), cur_stream[0]), "sdfr_compare_backward")

    def fused(dense=False, use_bounds=True, zero=True):
        _lib.check(lib.sdfr_compare_fused(
            (grids if dense else skewed).data_ptr(), R, RRR if dense else SK,
            _lib.LAYOUT_DENSE if dense else _lib.LAYOUT_SKEWED, pos.data_ptr(), quat.data_ptr(),
            inv_s.data_ptr(), B, W, H, CX, CY, FX, FY, THRESHOLD, obs.data_ptr(), 0,
            depth.data_ptr(), sums[0].data_ptr(), sums[1].data_ptr(), g_sdf.data_ptr(), RRR,
            g_pos.data_ptr(), g_quat.data_ptr(), g_is.data_ptr(), flags_b if zero else _lib.GRAD_ALL,
            bounds.data_ptr() if use_bounds else None, cur_stream[0]), "sdfr_compare_fused")

    def scale():
        _lib.check(lib.sdfr_scale_grads(
            sums[1].data_ptr(), None, R, B, g_sdf.data_ptr(), RRR, g_pos.data_ptr(),
            g_quat.data_ptr(), g_is.data_ptr(), _lib.GRAD_ALL, bounds.data_ptr(), 1, cur_stream[0]), "sdfr_scale_grads")

    launches = {"kernels": 0, "steps": 0}
    pending = []  # async all_gather work handles, at most two in flight (double-buffered losses)

    step_graph = [None] * Kg  # one captured step per ring slot (they differ in the slot the sums are copied to)

    def step_kernels(slot=None):
        # layout + empty-space-bounds pass, forward render + masked-L1 compare + backward in ONE traversal, then
        # the deferred per-hypothesis normalisation of the gradients inside the bounds box.  The outputs are
        # cleared on a second stream BESIDE the layout pass (the C ABI accumulates when SDFR_ZERO_GRADS is not
        # set, include/sdfrender.h; the product loop does the same, estimation/hypotheses.py): two memset nodes
        # parallel to the first kernels of the captured graph instead of a serial 64 MiB clear in front of the render
        main = torch.cuda.current_stream()
        clear_stream.wait_stream(main)
        with torch.cuda.stream(clear_stream):
            g_sdf.zero_()
            small.zero_()
        skew_bound()
        main.wait_stream(clear_stream)
        fused(zero=False)
        scale()
        if slot is not None:
            ring[slot].copy_(sums)  # 2 x hypotheses floats, device to device

    def step_serial_clears():
        # the same step with the library clearing its outputs in front of the render (SDFR_ZERO_GRADS)
        skew_bound()
        fused()
        scale()

    ring_pos = [0]
    n_exchanges = [0]

    def exchange():
        # the only exchange of the path: per-hypothesis losses (<= 2 KB per rank and step).  Nothing in the next
        # steps depends on it (the loop only ranks hypotheses at the end), so the losses of Kg steps are gathered
        # as one block, on NCCL's own stream beside the next steps' kernels; the buffers alternate, and a buffer
        # is reused only after the gather that read it has completed (stream-side wait, no host synchronisation).
        k = n_exchanges[0] & 1
        n_exchanges[0] += 1
        if len(pending) == 2:
            pending.pop(0).wait()
        torch.div(ring[:, 0], ring[:, 1], out=loss2[k])
        pending.append(dist.all_gather_into_tensor(gathered2[k], loss2[k].view(-1), async_op=True))
        launches["kernels"] += 2  # the division and NCCL's all-gather kernel

    def step():
        slot = ring_pos[0] if distributed else None
        if step_graph[slot or 0] is not None:
            step_graph[slot or 0].replay()
        else:
            step_kernels(slot)
        launches["kernels"] += (KERNELS_PER_CALL["sdfr_skew_grids_bounds"] + KERNELS_PER_CALL["sdfr_compare_fused"]
                                + KERNELS_PER_CALL["sdfr_scale_grads"])
        if distributed:
            ring_pos[0] = (ring_pos[0] + 1) % Kg
            if ring_pos[0] == 0:
                exchange()
        launches["steps"] += 1

    def drain():
        if distributed and ring_pos[0] != 0:  # the last, partial block
            ring_pos[0] = 0
            exchange()
        while pending:
            pending.pop(0).wait()

    flush_buf = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)

    def flush_l2():
        flush_buf.zero_()

    def timed(fn, n, warm, finish=None):
        """Sum of per-call CUDA-event times (ms) over n calls, L2 flushed before every call.  `finish`
        (the drain of the overlapped all-gathers) runs after the last call and its wait is added."""
        for _ in range(warm):
            flush_l2()
            fn()
        if finish is not None:
            finish()
        torch.cuda.synchronize()
        if distributed:
            dist.barrier()
            torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
               for _ in range(n)]
        for a, b in evs:
            flush_l2()
            a.record()
            fn()
            b.record()
        tail = None
        if finish is not None:
            finish()  # the current stream waits for the last gathers
            tail = torch.cuda.Event(enable_timing=True)
            tail.record()
        torch.cuda.synchronize()
        if distributed:
            dist.barrier()
            torch.cuda.synchronize()
        total = sum(a.elapsed_time(b) for a, b in evs)
        if tail is not None:
            total += evs[-1][1].elapsed_time(tail)
        return total

    if not args.no_step_graph:
        # the step's launches recorded once and replayed: what a caller with fixed buffers does (the product
        # loop and the e2e leg below do the same); the collective of the multi-GPU run stays outside the graph
        for _ in range(2):
            step_kernels()
        torch.cuda.synchronize()
        for slot in range(Kg):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):  # NCCL's watchdog thread polls events
                cur_stream[0] = torch.cuda.current_stream().cuda_stream
                step_kernels(slot if distributed else None)
            cur_stream[0] = stream
            step_graph[slot] = g
    K, Wm = args.steps, max(args.warmup, 3)
    if args.min_time > 0:  # one probe step decides how many steps fill the requested time (same on every rank)
        probe = torch.tensor([timed(step, 3, 2, finish=drain if distributed else None) / 3], device=dev)
        if distributed:
            dist.all_reduce(probe, op=dist.ReduceOp.MAX)
        K = max(K, int(args.min_time * 1e3 / float(probe.item())) + 1)
    with ClockSampler(local_rank) as clocks:
        launches["kernels"] = launches["steps"] = 0
        total_ms = timed(step, K, Wm, finish=drain if distributed else None)
    if args.dump_outputs and rank == 0:  # before the launches below overwrite the step's outputs
        dump_outputs(args.dump_outputs, {
            "depth": depth.cpu().numpy(), "loss_sum": sums[0].cpu().numpy(), "n_overlap": sums[1].cpu().numpy(),
            "grad_sdf": g_sdf.cpu().numpy(), "grad_position": g_pos.cpu().numpy(),
            "grad_orientation": g_quat.cpu().numpy(), "grad_inv_scale": g_is.cpu().numpy()})
    kernels_timed = launches["kernels"] * K // (K + Wm)  # warm-up steps launch the same kernels
    if distributed:
        t = torch.tensor([total_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    value = world * B * P * K / (total_ms * 1e-3) / 1e6
    ms_per_step = total_ms / K

    # the same step issued launch by launch, and with the normalisation as a separate pass
    step_eager_ms = timed(step_kernels, K, 2) / K
    step_serial_clears_ms = timed(step_serial_clears, K, 2) / K
    # per-kernel launch durations for the roofline (rank 0's GPU; same flush discipline)
    skew()
    bound()
    fused_ms = timed(fused, K, 2) / K
    fused_nobounds_ms = timed(lambda: fused(False, False), K, 2) / K
    bound_ms = timed(bound, K, 2) / K
    skew_bound_ms = timed(skew_bound, K, 2) / K
    fused_dense_ms = timed(lambda: fused(True), K, 2) / K
    skew_ms = timed(skew, K, 2) / K
    scale_ms = timed(scale, K, 2) / K
    fwd_ms = timed(fwd, K, 2) / K
    bwd_ms = timed(bwd, K, 2) / K

    # ---- end-to-end through the public API with host buffers --------------------------------
    # sdfest_b200.estimation.StreamedRenderCompare: every step copies the step's inputs (B grids,
    # poses, observed depth) from pinned host memory, renders + compares + back-propagates, and
    # reads the per-hypothesis results (loss, overlap count, 8 pose gradients) back to the host;
    # chunks of hypotheses are pipelined over copy / compute / copy-back streams.  SDF-grid
    # gradients stay in HBM (the decoder's backward consumes them there).
    from sdfest_b200.estimation import StreamedRenderCompare

    h_grids = grids.cpu().pin_memory()
    h_pos, h_quat, h_inv = pos.cpu().pin_memory(), quat.cpu().pin_memory(), inv_s.cpu().pin_memory()
    h_obs = obs.cpu().pin_memory()
    streamer = StreamedRenderCompare(cam, THRESHOLD, B, R, dev, chunk=args.e2e_chunk)
    h2d, d2h = streamer.h2d_bytes, streamer.d2h_bytes

    def e2e_step(graph):
        return streamer(h_grids, h_pos, h_quat, h_inv, h_obs, graph=graph, sync=True)

    def time_e2e(graph, n):
        for _ in range(3):
            e2e_step(graph)
        torch.cuda.synchronize()
        if distributed:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(n):
            res = e2e_step(graph)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if distributed:
            t = torch.tensor([dt], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        return dt, float(res["loss"].sum())

    Ke = max(3, min(K, 30))
    e2e_eager_s, e2e_check = time_e2e(False, Ke)
    try:
        e2e_graph_s, e2e_check_g = time_e2e(True, Ke)
    except Exception as e:  # capture is an optimisation, never a requirement
        e2e_graph_s, e2e_check_g = None, str(e)[:120]
    e2e_s = min(e2e_eager_s, e2e_graph_s) if e2e_graph_s else e2e_eager_s
    e2e_value = world * B * P * Ke / e2e_s / 1e6

    # ---- end to end the way the reference's callers actually hold their data -------------------
    # (estimation/simple_setup.py:414: sdf = vae.decode(latent) ON the device): every step the host hands
    # over 8 latent floats + pose + scale per hypothesis and the observed depth map from pinned memory, the
    # device decodes the grids (decoder trunk + fused tail), renders, compares, back-propagates to pose AND
    # latent, and the host reads back loss, overlap count and gradients (estimation.StreamedDecodeRenderCompare,
    # one CUDA graph per step).  More device work per step than the grid-shipping variant above (the decoder
    # and its backward), ~55x fewer bytes over PCIe.  This is `e2e`; the grid-shipping step is `e2e_grids`.
    e2e_decoded = None
    try:
        from sdfest_b200.estimation import StreamedDecodeRenderCompare

        dec_e = syn.residual_decoder(R, dev, syn.sdf_mug(R, dev))
        sdrc = StreamedDecodeRenderCompare(dec_e, cam, THRESHOLD, B, 8, dev)
        h_lat = torch.zeros(B, 8).pin_memory()
        h_scale = (1.0 / inv_s).cpu().pin_memory()

        def e2e_decoded_step():
            return sdrc(h_lat, h_pos, h_quat, h_scale, h_obs, graph=True, sync=True)

        for _ in range(3):
            e2e_decoded_step()
        torch.cuda.synchronize()
        if distributed:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(Ke):
            r_dec = e2e_decoded_step()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if distributed:
            t = torch.tensor([dt], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        dt_serial = dt
        # the same steps with TWO in flight: a second set of device / pinned result buffers and a second captured
        # graph on a second stream, so that step k+1's host->device copies and launch overlap step k's kernels
        # and result copy; the host waits for a step's result (event) before it reuses that step's buffers --
        # every step still copies its inputs from pinned host memory and delivers its result to the host
        try:
            pipe = [sdrc, StreamedDecodeRenderCompare(dec_e, cam, THRESHOLD, B, 8, dev)]
            lanes = [torch.cuda.Stream(dev) for _ in pipe]
            done = [None, None]

            def e2e_pipelined(n):
                for i in range(n):
                    k = i & 1
                    if done[k] is not None:
                        done[k].synchronize()  # the result of step i-2 is in host memory from here on
                    with torch.cuda.stream(lanes[k]):
                        pipe[k](h_lat, h_pos, h_quat, h_scale, h_obs, graph=True, sync=False)
                        done[k] = torch.cuda.Event()
                        done[k].record(lanes[k])
                for ev in done:
                    if ev is not None:
                        ev.synchronize()

            for lane in lanes:
                lane.wait_stream(torch.cuda.current_stream())
            e2e_pipelined(4)
            torch.cuda.synchronize()
            if distributed:
                dist.barrier()
            t0 = time.perf_counter()
            e2e_pipelined(Ke)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if distributed:
                t = torch.tensor([dt], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            same = float((pipe[0].h_out - pipe[1].h_out).abs().max())  # both lanes computed the same step
            two_in_flight = {"value": world * B * P * Ke / dt / 1e6, "unit": UNIT, "ms_per_step": dt / Ke * 1e3,
                             "max_abs_difference_between_the_two_lanes": same,
                             "what": "independent steps (e.g. the hypotheses of different objects or frames): a second "
                                     "set of device / pinned result buffers and a second captured graph on a second "
                                     "stream; the host waits for a step's result before it reuses that step's buffers"}
        except Exception as e:  # noqa: BLE001
            two_in_flight = {"unavailable": str(e)[:200]}
        dt = dt_serial  # `e2e` itself: one step at a time, as the dependent Adam steps of one batch of hypotheses run
        e2e_decoded = {"value": world * B * P * Ke / dt / 1e6, "unit": UNIT, "h2d_bytes_per_step": sdrc.h2d_bytes,
                       "d2h_bytes_per_step": sdrc.d2h_bytes, "steps": Ke, "ms_per_step": dt / Ke * 1e3,
                       "two_steps_in_flight": two_in_flight,
                       "api": "estimation.StreamedDecodeRenderCompare: pinned host latents / poses / scale / observed "
                              "depth -> decoder trunk + sdfr_decoder_tail_forward + sdfr_compare_fused + tail adjoint "
                              "+ trunk backward -> loss, overlap count and gradients w.r.t. latent, position, "
                              "orientation, scale back to the host; one CUDA graph per step, copies included",
                       "d2h": "loss, n_overlap, 8 pose / scale gradients and 8 latent gradients per hypothesis",
                       "checksum": float(r_dec["loss"].sum())}
    except Exception as e:
        e2e_decoded = {"unavailable": str(e)[:200]}

    # ---- the whole loop of BASELINE config 2: 50 Adam steps on pose / scale / latent -------------
    # decoder (reference architecture, trunk + fused tail on this library's kernels) -> fused
    # render-and-compare -> point-cloud loss -> backward -> Adam, B hypotheses at once, replayed as a
    # CUDA graph (estimation.HypothesisOptimizer).  Reported beside the render metric, not instead.
    loop = None
    try:
        from sdfest_b200.estimation import HypothesisOptimizer

        dec = syn.residual_decoder(R, dev, syn.sdf_mug(R, dev))
        opt = HypothesisOptimizer(cam, THRESHOLD, obs, pos, quat, 1.0 / inv_s,
                                  latent=torch.zeros(B, 8, device=dev), decoder=dec,
                                  inlier_threshold=0.03)  # the reference evaluates it every iteration (:463)
        opt.capture()
        for _ in range(5):
            opt.step()
        torch.cuda.synchronize()
        if distributed:
            dist.barrier()
        n_it = 50
        a, b_ev = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n_it):
            opt.step()
        b_ev.record()
        torch.cuda.synchronize()
        loop_ms = a.elapsed_time(b_ev)
        if distributed:
            t = torch.tensor([loop_ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            loop_ms = float(t.item())
            final = opt.run(1)  # one more step with the all_gather of the per-hypothesis losses
            assert final.numel() == world * B
        loop = {"hyp_iter_per_s": world * B * n_it / (loop_ms * 1e-3), "ms_per_iteration": loop_ms / n_it,
                "iterations": n_it, "hypotheses_per_gpu": B, "optimizer": opt.optimizer_impl,
                "what": "50 Adam steps on position/orientation/scale/latent: decoder trunk + fused tail, "
                        "fused render-and-compare, fused point loss, tail adjoint + trunk backward, one "
                        "sdfr_hypothesis_step kernel (chain rule + Adam + renormalisation), inlier ratio + best estimate (counted inside the render traversal, sdfr_track_best); CUDA-graph replay",
                "final_mean_loss": float(opt.last_losses.mean()),
                "final_mean_inlier_ratio": float(torch.nan_to_num(opt.inlier_ratio).mean())}
        # fixed grids (BASELINE config 4's per-GPU work: pose/scale hypotheses on given shapes)
        opt = HypothesisOptimizer(cam, THRESHOLD, obs, pos, quat, 1.0 / inv_s, sdf=grids, inlier_threshold=0.03)
        opt.capture()
        for _ in range(5):
            opt.step()
        torch.cuda.synchronize()
        a, b_ev = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n_it):
            opt.step()
        b_ev.record()
        torch.cuda.synchronize()
        pose_ms = a.elapsed_time(b_ev)
        if distributed:
            t = torch.tensor([pose_ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            pose_ms = float(t.item())
        loop["pose_only"] = {"hyp_iter_per_s": world * B * n_it / (pose_ms * 1e-3),
                             "ms_per_iteration": pose_ms / n_it,
                             "what": "same loop on fixed grids: 4 launches per iteration (fused "
                                     "render-and-compare with inlier count, fused point loss, "
                                     "hypothesis step, best-estimate bookkeeping)"}
    except Exception as e:  # the loop demo never blocks the render metric
        loop = {"unavailable": str(e)[:200]}

    if rank != 0:
        if distributed:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel ------------------------------------------------------
    n_over = int(sums[1].sum().item())
    fwd_bytes, bwd_bytes, fused_bytes = algorithmic_bytes(S, P, B, RRR, Hh_all, n_over)
    peak, peak_src = measured_peaks()
    roofline = roofline_object(fused_bytes, fused_ms, S, peak, peak_src, ncu_traffic("fused"), gather_peaks())
    roofline["kernels"] = {
        "fused_incl_memsets": {"ms": fused_ms, "bytes": fused_bytes, "GBps": fused_bytes / fused_ms / 1e6},
        "fused_dense_layout_incl_memsets": {"ms": fused_dense_ms, "bytes": fused_bytes,
                                            "GBps": fused_bytes / fused_dense_ms / 1e6},
        "fused_without_empty_space_bounds": {"ms": fused_nobounds_ms},
        "grid_bounds": {"ms": bound_ms, "bytes": 4 * SK * B, "GBps": 4 * SK * B / bound_ms / 1e6},
        "skew_grids_bounds": {"ms": skew_bound_ms, "bytes": 4 * (RRR + SK) * B,
                              "GBps": 4 * (RRR + SK) * B / skew_bound_ms / 1e6},
        "skew_grids": {"ms": skew_ms, "bytes": 4 * (RRR + SK) * B, "GBps": 4 * (RRR + SK) * B / skew_ms / 1e6},
        "scale_grads": {"ms": scale_ms, "bytes": 8 * RRR * B, "GBps": 8 * RRR * B / scale_ms / 1e6},
        "unfused_forward": {"ms": fwd_ms, "bytes": fwd_bytes, "GBps": fwd_bytes / fwd_ms / 1e6,
                            "gsamples_per_s": S / fwd_ms / 1e6},
        "unfused_backward_incl_memsets": {"ms": bwd_ms, "bytes": bwd_bytes, "GBps": bwd_bytes / bwd_ms / 1e6},
    }
    roofline["work"] = {"samples_S": S, "hit_pixels": Hh_all, "overlap_pixels_Hh": n_over,
                        "box_pixels": stats["box_pixels"], "pixels": P * B,
                        "without_empty_space_bounds": {"samples_S": stats_full["samples"],
                                                       "box_pixels": stats_full["box_pixels"]}}

    e2e_grids = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                 "steps": Ke, "ms_per_step": e2e_s / Ke * 1e3,
                 "api": "estimation.StreamedRenderCompare (C ABI sdfr_compare_fused + sdfr_scale_grads per "
                        f"chunk of {args.e2e_chunk} hypotheses; 3 streams; pinned host buffers; the 64^3 grids "
                        "themselves cross PCIe every step)",
                 "ms_per_step_eager": e2e_eager_s / Ke * 1e3,
                 "ms_per_step_cuda_graph": (e2e_graph_s / Ke * 1e3) if e2e_graph_s else e2e_check_g,
                 "d2h": "loss, n_overlap, 8 pose gradients per hypothesis; SDF gradients stay on the device",
                 "checksum": e2e_check}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_object(B, distributed),
        "render_hyp_iter_per_s": world * B * K / (total_ms * 1e-3),
        "step": {"what": "sdfr_skew_grids_bounds (layout + empty-space bounds, one read of the grids) -> "
                         "sdfr_compare_fused (render + masked L1 + backward in one traversal) -> sdfr_scale_grads "
                         "(upstream/n_overlap inside the bounds box); the outputs cleared on a second stream beside the layout pass"
                         + ("" if args.no_step_graph else "; the launches replayed as one CUDA graph"),
                 "ms_issued_launch_by_launch": step_eager_ms,
                 "ms_launch_by_launch_library_clears_in_front_of_the_render": step_serial_clears_ms},
        "exchange": ({"what": "every step's per-hypothesis losses kept in a device ring, all-gathered as one block",
                      "steps_per_all_gather": Kg, "bytes_per_rank_and_gather": 4 * Kg * B} if distributed else None),
        "loop": loop,
        "roofline": roofline,
        # the contract's `e2e`: the step from the inputs the reference's callers hold (latents, poses, observation
        # in pinned host memory); `e2e_grids`: the same renderer step when the host ships the decoded grids
        "e2e": e2e_decoded if "value" in e2e_decoded else e2e_grids,
        "e2e_grids": e2e_grids,
        # kernels launched inside the timed region, counted per C-ABI call made (KERNELS_PER_CALL)
        "gpu_launches": kernels_timed,
        "clocks": clocks.summary(),
        "lib": lib.sdfr_build_info().decode(),
    }

    if not args.no_cpu_baseline and world == 1:  # reported at N = 1 only
        try:
            mpix, ms, cores = time_cpu(min(args.cpu_sample, args.hypotheses), 40, 1)
            line["cpu_baseline"] = {
                "value": mpix, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"{args.cpu_sample} hypotheses x {W}x{H} fwd+L1+bwd per step, 40 steps (oracle/liboracle.so, OpenMP)"}
        except Exception as e:  # the oracle is a checker, never required by the product path
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port",
                                    "sample": f"unavailable: {e}"}

    if not args.no_ref_ext:
        try:
            line["reference_cuda_ext"] = time_reference_extension(
                torch, dev, grids, pos, quat, inv_s, obs, flush_l2, min(K, 10))
        except Exception as e:
            line["reference_cuda_ext"] = {"unavailable": str(e)[:200]}

    emit(line)
    if distributed:
        dist.destroy_process_group()


def time_reference_extension(torch, dev, grids, pos, quat, inv_s, obs, flush_l2, steps):
    """The reference's own CUDA extension (compiled from /root/reference into oracle/_ref) on the
    same GPU and the same step: per hypothesis forward, masked L1 in torch, backward -- the way
    the reference pipeline drives it (simple_setup.py:432-456), one hypothesis at a time."""
    from oracle import build_ref

    ext = build_ref.load_module()
    if ext is None:
        raise RuntimeError("oracle/_ref/sdf_renderer_cpp.so not present")
    B = grids.shape[0]

    def ref_step():
        for b in range(B):
            sdf, p, q, s = grids[b], pos[b], quat[b], inv_s[b:b + 1]
            (d,) = ext.forward(sdf, p, q, s, W, H, CX, CY, FX, FY, THRESHOLD)
            mask = (obs > 0) & (d > 0)
            g = torch.where(mask, torch.sign(d - obs), torch.zeros_like(d)) / mask.sum()
            ext.backward(g, d, sdf, p, q, s, W, H, CX, CY, FX, FY)

    for _ in range(2):
        ref_step()
    torch.cuda.synchronize()
    ms = 0.0
    for _ in range(steps):
        flush_l2()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ref_step()
        b.record()
        torch.cuda.synchronize()
        ms += a.elapsed_time(b)
    ms /= steps
    return {"value": B * W * H / (ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": ms,
            "what": "sdf_renderer_cpp.forward + torch masked-L1 + sdf_renderer_cpp.backward per hypothesis"}


if __name__ == "__main__":
    main()
