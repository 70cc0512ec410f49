"""The bench line's contract.  The pure pieces of bench.py (config object, algorithmic bytes, roofline
object, launch accounting) are exercised on CPU with stub timings, so the test fails when bench.py's
output regresses, not only when a committed artefact is edited; the last committed measurement of each
arm (profiles/) is then checked for every key the driver reads."""
import glob
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def _latest(pattern):
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", pattern)))
    assert files, pattern
    return json.loads(open(files[-1]).read().strip().splitlines()[-1])


def test_pure_pieces_of_the_line():
    cfg = bench.config_object(64, False)
    assert "model" not in cfg and cfg["workload"].startswith("C2") and "l2" in cfg and cfg["collective"] == "none"
    assert bench.config_object(64, True)["collective"].startswith("all_gather")
    # SURVEY 8d's formula on round numbers
    S, P, B, RRR, hits, n_over = 1000, 10, 2, 8, 5, 3
    fwd, bwd, fused = bench.algorithmic_bytes(S, P, B, RRR, hits, n_over)
    assert fwd == 32 * 1000 + 4 * 10 * 2 + 4 * 8 * 2 + 4 * 5
    assert fused == fwd + 96 * 3 + 4 * 8 * 2 and bwd == 4 * 10 * 2 + 4 * 5 + 96 * 3 + 4 * 8 * 2
    r = bench.roofline_object(fused_bytes=10 ** 9, fused_ms=0.2, S=20 * 10 ** 6, peak=6547.5, peak_src="measured",
                              traffic=150_000_000,
                              peaks={"l1_skewed_gsamples": 372.0, "l2_skewed_gsamples": 201.0, "source": "x"})
    assert r["bound"] in ("hbm", "tensor") and r["unit"] == "GB/s"
    assert abs(r["achieved"] - 5000.0) < 1e-9 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    g = r["gather"]
    assert abs(g["achieved_gsamples_per_s"] - 100.0) < 1e-9
    assert abs(g["frac_of_l2_gather_peak"] - 100.0 / 201.0) < 1e-12 and "limiter" in g
    assert "gather" in bench.roofline_object(10 ** 9, 0.2, 10 ** 6, 6547.5, "m", None, None)
    assert sum(bench.KERNELS_PER_CALL.values()) == 4  # the step: bounds (2) + fused (1) + scale (1); clears are memset nodes
    peaks = bench.gather_peaks()  # the committed micro-benchmark result
    assert peaks and peaks["l1_skewed_gsamples"] > peaks["l2_skewed_gsamples"] > 50


def _check_own_arm(d):
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "roofline", "e2e", "gpu_launches", "clocks"):
        assert k in d, k
    assert d["unit"] == "Mpix/s" and d["dtype"] == "f32" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and "workload" in d["config"]
    assert "model" not in d["config"] and "l2" in d["config"]
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["unit"] in ("GB/s", "TFLOP/s")
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["traffic"] > 0
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and 0 < e["value"] < d["value"]
    assert d["gpu_launches"] > 0
    assert d["clocks"]["sm_mhz"] > 0 and not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown",
                                                                              "sw_thermal_slowdown"}
    cfg = d["config"]  # value is pixels of the whole job over the step time
    pix = d["n_gpus"] * cfg["hypotheses_per_gpu"] * cfg["width"] * cfg["height"]
    assert abs(d["value"] - pix / (d["ms_per_step"] * 1e-3) / 1e6) < 1e-6 * d["value"]


def test_own_arm_line_of_the_last_committed_runs():
    for pattern in ("r01zx_bench.json", "r02*_bench.json"):
        if not glob.glob(os.path.join(ROOT, "profiles", pattern)):
            continue
        d = _latest(pattern)
        _check_own_arm(d)
        if d["n_gpus"] == 1:
            c = d["cpu_baseline"]
            assert c["kind"] in ("reference", "port") and c["cores"] >= 1 and c["value"] > 0 and c["sample"]
        if pattern.startswith("r02"):  # this round's additions
            per_step = 4 if "step" in d else 5  # since the step clears its outputs with memset nodes
            gathers = 0
            if d["n_gpus"] > 1:  # the division + NCCL's kernel, per step or per block of steps
                gathers = -(-d["steps"] // d["exchange"]["steps_per_all_gather"]) if d.get("exchange") else d["steps"]
            assert d["gpu_launches"] == per_step * d["steps"] + 2 * gathers
            assert d["config"] == bench.config_object(d["config"]["hypotheses_per_gpu"], d["n_gpus"] > 1)
            assert 0 < d["roofline"]["gather"]["frac_of_l1_gather_peak"] < d["roofline"]["gather"]["frac_of_l2_gather_peak"]
            if "e2e_grids" in d:  # e2e = host latents -> device decode; e2e_grids = the grids cross PCIe
                assert d["e2e"]["h2d_bytes_per_step"] < d["e2e_grids"]["h2d_bytes_per_step"] / 10
                assert d["e2e"]["value"] > d["e2e_grids"]["value"]
            else:  # lines from before the swap
                assert d["e2e_decoded"]["h2d_bytes_per_step"] < d["e2e"]["h2d_bytes_per_step"] / 10


def test_reference_arm_line():
    for pattern in ("r01zv_bench_ref.json", "r02*_bench_ref.json"):
        if not glob.glob(os.path.join(ROOT, "profiles", pattern)):
            continue
        d = _latest(pattern)
        assert d["impl"] == "reference" and d["unit"] == "Mpix/s" and d["value"] > 0
        assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
        assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["kind"] in ("reference", "port")
        if pattern.startswith("r02"):
            assert d["config"] == bench.config_object(d["config"]["hypotheses_per_gpu"], False)


def test_dump_outputs_writes_float32_and_samples_large_outputs_at_fixed_positions(tmp_path):
    import numpy as np
    import pytest

    big = np.arange(bench.DUMP_SAMPLE + 1000, dtype=np.float64)  # values = flat indices
    small = np.ones((4, 3), np.float32)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"big": big, "small": small})
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert a.dtype == np.float32 and a.shape == (bench.DUMP_SAMPLE,) and np.array_equal(a, b)
    assert (np.diff(a) > 0).all() and a[-1] <= big[-1]  # distinct positions, in index order
    s = np.load(tmp_path / "a" / "small.npy")
    assert s.dtype == np.float32 and np.array_equal(s, small)
    with pytest.raises(SystemExit):  # over the size limit: nothing is written
        bench.dump_outputs(str(tmp_path / "c"), {f"x{i}": big for i in range(4)})
    assert not (tmp_path / "c").exists()
