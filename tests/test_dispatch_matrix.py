"""Every render-kernel instantiation and every launch regime, against the CPU oracle.

The host launchers of libsdfrender pick one of the separately compiled render kernels (resolution and
layout, mode, gradient set) and a launch shape (CTAs per hypothesis, CTA stealing, ray tables, slices
of 65535 hypotheses, composite passes) from their arguments, so a scene's size silently decides what a
test runs.  Here `selected` restates that host dispatch (sdfest_b200/csrc/sdfrender.cu) in plain
Python, and `CASES` is a table of explicit C-ABI calls that together reach every instantiation and
every regime.

Without a GPU: the union of `selected` over `CASES` must be exactly the set of render kernels compiled
into the library (`nm -C`), and every regime must be reached -- a new resolution in SDFR_DISPATCH_RT_LT
or a new variant in a launcher fails here until a case covers it.

On the GPU: every case runs once into NaN-filled outputs surrounded by guard elements, and its depth,
compare sums, forward statistics and gradients are compared with the oracle under the suite's usual
gates (tests/util.py); one test checks in a torch.profiler trace that the launches are the kernels and
grids `selected` predicts.
"""
from __future__ import annotations

import ctypes
import json
import os
import re
import shutil
import subprocess
import tempfile
from dataclasses import dataclass

import numpy as np
import pytest
import torch

import oracle
from sdfest_b200 import _lib
from sdfest_b200 import synthetic as syn
from util import cell_face_mask, depth_parity, pose_grad_parity, sdf_grad_parity

# ------------------------------------------------------------------------------------------
# the host dispatch of sdfrender.cu, restated
# ------------------------------------------------------------------------------------------
SM_COUNT_B200 = 148
FWD_BLOCKS = 5          # kFwdBlocks: resident forward CTAs per SM
MAX_OBJ_PER_PASS = 32   # kMaxObjPerPass of the composite kernels
SLICE = 65535           # gridDim.y limit: launches are split into slices of this many hypotheses
POSE = _lib.GRAD_POSITION | _lib.GRAD_ORIENTATION | _lib.GRAD_INV_SCALE
ALL, SDF, Z, X = _lib.GRAD_ALL, _lib.GRAD_SDF, _lib.ZERO_GRADS, _lib.SDF_GRAD_EXACT
DENSE, SKEWED = _lib.LAYOUT_DENSE, _lib.LAYOUT_SKEWED


def n_tiles(W, H):
    return -(-W // 32) * -(-H // 8)


def ctas_per_hypothesis(batch, W, H, sm):
    g = -(-sm * (16 if batch >= 16 else 32) // batch)
    return max(1, min(g, n_tiles(W, H), 65535))


def table_bytes(W, H):
    n = 4 * (-(-W // 32) * 32 + -(-H // 8) * 8)
    return n if n <= 40 * 1024 else 0


def rt_lt(R, layout):
    """SDFR_DISPATCH_RT_LT: compile-time pitches for 64, 128 and 32 in both layouts, else the run-time kernel"""
    return (R, layout) if R in (64, 128, 32) else (0, DENSE)


def _b(v):
    return "true" if v else "false"


def _want(flags):
    return bool(flags & SDF), bool(flags & POSE)


def _slices(B):
    return [(z0, min(SLICE, B - z0)) for z0 in range(0, B, SLICE)]


def _gs_stride(R, gs):
    return {"dense": R ** 3, "padded": R ** 3 + 17, "shared": 0}[gs]


@dataclass(frozen=True)
class Call:
    """One entry point of the C ABI, with the launches a caller makes around it:
    forward | forward_stats | compare_forward: the entry alone;
    backward: sdfr_forward, then sdfr_backward with an explicit upstream image;
    compare_backward: sdfr_compare_forward, then sdfr_compare_backward;
    compare_fused | compare_fused_inliers: the fused entry, then sdfr_scale_grads (with gradient flags);
    composite: sdfr_forward_composite, then sdfr_backward_composite (with gradient flags)."""
    entry: str
    flags: int = 0          # gradient flags | SDFR_SDF_GRAD_EXACT | SDFR_ZERO_GRADS (without: accumulate)
    gs: str = "dense"       # grad_sdf_stride: R^3 ("dense"), R^3 + 17 ("padded"), 0 ("shared")
    upstream: bool = False  # per-hypothesis upstream factors of the compare gradients (else NULL)
    offset: int = 0         # every output pointer this many floats past a 16-byte boundary


@dataclass(frozen=True)
class Case:
    name: str
    R: int
    layout: int
    B: int                  # hypotheses (composite: objects)
    W: int
    H: int
    calls: tuple
    grids: str = "per"      # "per": one grid per hypothesis; "shared": one grid, sdf_stride 0
    bounds: bool = False    # empty-space bounds from sdfr_grid_bounds (one entry per grid)
    obs: str = "shared"     # obs_stride 0, or "per" hypothesis (the last one observes nothing)
    poses: int = 0          # > 0: this many distinct poses (and grids) cycled over the batch
    z: float = -0.3         # distance of the objects
    f: float = 0.0          # focal length in pixels (0: W / 2)
    tiled: bool = False     # objects side by side on an 8 x 5 grid (many-object composites)


def _forward(c, mode, stats, flags, call, sm):
    rt, lt = rt_lt(c.R, c.layout)
    ws = wp = False
    if mode == 2:
        ws, wp = _want(flags)
        mode = 2 if (ws or wp) else 1  # no gradient requested: the compare kernel
    name = f"sdfr_forward_kernel<{rt}, {lt}, {mode}, {_b(stats)}, {_b(ws)}, {_b(wp)}>"
    use_tables = table_bytes(c.W, c.H) != 0
    G = ctas_per_hypothesis(c.B, c.W, c.H, sm)
    sl = _slices(c.B)
    out = []
    for _, nz in sl:
        steal = G * nz > sm * FWD_BLOCKS
        out.append(dict(kernel=name, grid=(G, nz, 1), G=G, slices=len(sl), steal=steal, use_tables=use_tables,
                        image_tables=use_tables and steal and G < n_tiles(c.W, c.H),
                        vec_fill=c.W % 4 == 0 and call.offset % 4 == 0))
    return out


def _grad_memset(c, call):
    if not (call.flags & Z and call.flags & SDF):
        return "none"
    return "per_grid" if call.gs == "padded" else "one"


def _backward(c, mode, call, sm):
    ws, wp = _want(call.flags)
    if not (ws or wp):
        return []
    rt, lt = rt_lt(c.R, c.layout)
    name = f"sdfr_backward_kernel<{rt}, {lt}, {mode}, {_b(ws)}, {_b(wp)}>"
    sl = _slices(c.B)
    return [dict(kernel=name, grid=(ctas_per_hypothesis(nz, c.W, c.H, sm), nz, 1), slices=len(sl),
                 use_tables=table_bytes(c.W, c.H) != 0, grad_memset=_grad_memset(c, call)) for _, nz in sl]


def _zero_small(c, flags):
    if not (flags & Z and flags & POSE):
        return []
    n = c.B * (3 * bool(flags & _lib.GRAD_POSITION) + 4 * bool(flags & _lib.GRAD_ORIENTATION)
               + bool(flags & _lib.GRAD_INV_SCALE))
    return [dict(kernel="sdfr_zero_small_kernel", grid=(16 if n > 4096 else 1, 1, 1))]


def _scale_grads(c, call):
    if not call.flags & ALL:
        return []
    gx = max(1, (c.R ** 3 // 4 + 2047) // 2048) if call.flags & SDF else 1
    paths = set()
    if call.flags & SDF:  # scale_sdf_grads: per hypothesis, by its bounds and the alignment of its grid
        stride = _gs_stride(c.R, call.gs)
        for b in range(min(c.B, 4)):
            aligned = (call.offset + b * stride) % 4 == 0
            if c.bounds:
                paths.add("box_float4" if aligned and c.R % 4 == 0 else "box_rows")
            else:
                paths.add("grid_float4" if aligned else "grid_scalar")
    sl = _slices(c.B)
    return [dict(kernel="sdfr_scale_grads_kernel", grid=(gx, nz, 1), slices=len(sl), scale_paths=paths)
            for _, nz in sl]


def _composite(c, call):
    rt, lt = rt_lt(c.R, c.layout)
    grid = (-(-c.W // 32), -(-c.H // 8), 1)
    out = [dict(kernel=f"sdfr_forward_composite_kernel<{rt}, {lt}>", grid=grid,
                passes=-(-c.B // MAX_OBJ_PER_PASS))]
    ws, wp = _want(call.flags)
    if ws or wp:
        out += _zero_small(c, call.flags)
        out.append(dict(kernel=f"sdfr_backward_composite_kernel<{rt}, {lt}, {_b(ws)}, {_b(wp)}>", grid=grid))
    return out


def selected(c, sm):
    """Every launch of the case's calls: kernel instantiation (as `nm -C` prints it), grid and regime."""
    out = []
    for call in c.calls:
        e, fl = call.entry, call.flags
        if e == "forward":
            out += _forward(c, 0, False, 0, call, sm)
        elif e == "forward_stats":
            out += _forward(c, 0, True, 0, call, sm)
        elif e == "compare_forward":
            out += _forward(c, 1, False, 0, call, sm)
        elif e == "backward":
            out += _forward(c, 0, False, 0, call, sm) + _zero_small(c, fl) + _backward(c, 0, call, sm)
        elif e == "compare_backward":
            out += _forward(c, 1, False, 0, call, sm) + _zero_small(c, fl) + _backward(c, 1, call, sm)
        elif e in ("compare_fused", "compare_fused_inliers"):
            if fl & Z:
                out.append(dict(kernel="sdfr_zero_sums_and_small_kernel", grid=(16 if c.B > 512 else 1, 1, 1)))
            out += _forward(c, 2, False, fl, call, sm) + _scale_grads(c, call)
        elif e == "composite":
            out += _composite(c, call)
        else:
            raise ValueError(e)
    return out


# ------------------------------------------------------------------------------------------
# the table
# ------------------------------------------------------------------------------------------
def every_variant(exact=False, accumulate=False, gs="dense", upstream=False, offset=0):
    """The 16 render kernels of one (resolution, layout) pair: forward MODE 0 with and without
    statistics, MODE 1, MODE 2 with each gradient set; backward MODE 0 and 1 with each gradient set;
    the composite forward and its three backward variants."""
    x = X if exact else 0
    z = 0 if accumulate else Z
    calls = [Call("forward_stats", offset=offset)]
    for fl in (ALL, SDF, POSE):
        calls += [Call("backward", fl | x | z, gs=gs, offset=offset),
                  Call("compare_backward", fl | x | z, gs=gs, upstream=upstream, offset=offset),
                  Call("compare_fused_inliers" if fl == ALL else "compare_fused", fl | x | Z,
                       gs="dense" if gs == "shared" else gs, upstream=upstream, offset=offset),
                  Call("composite", fl | x | z, gs=gs, offset=offset)]
    return tuple(calls)


CASES = [
    # every variant of every (RT, LT) pair; B = 3, partial tiles, W % 4 != 0 for some
    Case("r64_dense", 64, DENSE, 3, 148, 66, every_variant(), obs="per"),
    Case("r64_skewed", 64, SKEWED, 3, 190, 91, every_variant(accumulate=True, gs="padded", upstream=True),
         bounds=True),
    Case("r128_dense", 128, DENSE, 3, 144, 75, every_variant(exact=True, offset=1), bounds=True),
    Case("r128_skewed", 128, SKEWED, 3, 134, 63, every_variant(exact=True, gs="shared"), obs="per"),
    Case("r32_dense", 32, DENSE, 3, 115, 57, every_variant(accumulate=True, upstream=True), grids="shared",
         bounds=True),
    Case("r32_skewed", 32, SKEWED, 3, 180, 105, every_variant(exact=True, gs="padded", offset=1), obs="per"),
    Case("r24_dense", 24, DENSE, 3, 151, 59, every_variant(exact=True, gs="shared", upstream=True)),
    Case("r24_skewed", 24, SKEWED, 3, 132, 78, every_variant(accumulate=True), bounds=True, obs="per"),
    Case("r37_dense", 37, DENSE, 3, 117, 61, every_variant(offset=1, upstream=True), bounds=True),
    Case("r37_skewed", 37, SKEWED, 3, 156, 71, every_variant(exact=True, gs="padded"), obs="per"),
    # launch regimes
    Case("steal_image_tables", 64, DENSE, 64, 160, 120,
         (Call("forward"), Call("compare_fused_inliers", ALL | Z, upstream=True)), bounds=True),
    Case("steal_tile_tables", 32, SKEWED, 64, 64, 64, (Call("forward"), Call("compare_fused", POSE | Z)),
         z=-0.25),
    Case("steal_tile_tables_one_frame", 64, SKEWED, 1, 640, 480,
         (Call("forward"), Call("compare_fused_inliers", ALL | Z), Call("backward", ALL | Z),
          Call("compare_backward", ALL | Z)), bounds=True),
    Case("no_ray_tables", 128, DENSE, 1, 10240, 24,
         (Call("forward"), Call("compare_fused", ALL | X | Z, offset=1), Call("backward", ALL | Z)), f=400.0),
    Case("slices", 12, DENSE, 65539, 40, 12,
         (Call("backward", ALL | Z), Call("compare_fused", ALL | Z, upstream=True),
          Call("compare_backward", ALL | Z, upstream=True)), poses=4),
    Case("composite_two_passes", 32, SKEWED, 40, 200, 120, (Call("composite", ALL | Z),), z=-0.8, tiled=True),
    Case("compare_without_gradients", 37, SKEWED, 3, 64, 40,
         (Call("compare_forward"), Call("compare_fused", Z)), grids="shared", bounds=True),
]
CASE_IDS = [c.name for c in CASES]
BY_NAME = {c.name: c for c in CASES}


# ------------------------------------------------------------------------------------------
# without a GPU: the table against the library
# ------------------------------------------------------------------------------------------
RENDER_KERNEL = re.compile(r"(?<![\w])(sdfr_(?:forward|backward)(?:_composite)?_kernel<[^>]*>)")


def compiled_render_kernels():
    nm = shutil.which("nm")
    if nm is None:
        pytest.skip("nm not found")
    out = subprocess.run([nm, "-C", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    return set(RENDER_KERNEL.findall(out))


def _all_launches(sm=SM_COUNT_B200):
    return [l for c in CASES for l in selected(c, sm)]


def test_cases_reach_every_compiled_render_kernel():
    compiled = compiled_render_kernels()
    reached = {l["kernel"] for l in _all_launches() if RENDER_KERNEL.fullmatch(l["kernel"])}
    assert len(compiled) > 0
    assert not compiled - reached, f"compiled, reached by no case: {sorted(compiled - reached)}"
    assert not reached - compiled, f"selected, not compiled: {sorted(reached - compiled)}"


def test_cases_reach_every_launch_regime():
    ls = _all_launches()
    fwd = [l for l in ls if l["kernel"].startswith("sdfr_forward_kernel")]
    bwd = [l for l in ls if l["kernel"].startswith("sdfr_backward_kernel")]
    scale = [l for l in ls if l["kernel"] == "sdfr_scale_grads_kernel"]
    comp = [l for l in ls if l["kernel"].startswith("sdfr_forward_composite_kernel")]
    regimes = {
        "forward in one wave, no stealing": any(not l["steal"] for l in fwd),
        "stealing, ray tables of the whole image": any(l["steal"] and l["image_tables"] for l in fwd),
        "stealing, per-item ray tables (G == tiles)":
            any(l["steal"] and l["use_tables"] and not l["image_tables"] for l in fwd),
        "forward without ray tables": any(not l["use_tables"] for l in fwd),
        "forward in several slices": any(l["slices"] > 1 for l in fwd),
        "forward zero fill, float4 and scalar": {l["vec_fill"] for l in fwd} == {True, False},
        "backward without ray tables": any(not l["use_tables"] for l in bwd),
        "backward in several slices": any(l["slices"] > 1 for l in bwd),
        "backward, gradient grids cleared per grid, at once, not at all":
            {l["grad_memset"] for l in bwd} == {"per_grid", "one", "none"},
        "scale_grads in several slices": any(l["slices"] > 1 for l in scale),
        "scale_grads, every path": set().union(*(l["scale_paths"] for l in scale))
            == {"box_float4", "box_rows", "grid_float4", "grid_scalar"},
        "composite, one pass and several": {l["passes"] > 1 for l in comp} == {True, False},
        "zero kernels with 16 CTAs": {l["grid"][0] for l in ls if l["kernel"].startswith("sdfr_zero")} == {1, 16},
    }
    missed = [k for k, v in regimes.items() if not v]
    assert not missed, f"no case reaches: {missed}"


def test_flag_and_stride_combinations_are_covered():
    """Each option at least once away from the <64, skewed> kernels the benchmark runs."""
    away = [(c, call) for c in CASES for call in c.calls if rt_lt(c.R, c.layout) != (64, SKEWED)]
    grads = [(c, call) for c, call in away if call.flags & ALL]
    assert {bool(call.flags & X) for _, call in grads} == {True, False}
    assert {bool(call.flags & Z) for _, call in grads} == {True, False}
    assert {call.gs for _, call in grads} == {"dense", "padded", "shared"}
    assert {call.offset for _, call in away} == {0, 1}
    compare = [(c, call) for c, call in away if "compare" in call.entry]
    assert {c.obs for c, _ in compare} == {"shared", "per"}
    assert {call.upstream for _, call in compare if call.flags & ALL} == {True, False}
    assert {(c.bounds, c.grids) for c, _ in away} == {(False, "per"), (True, "per"), (True, "shared")}


# ------------------------------------------------------------------------------------------
# on the GPU
# ------------------------------------------------------------------------------------------
GUARD = 64              # guard elements on either side of every output (256 bytes: keeps 16-byte alignment)
SENTINEL = -12345.0     # value of the guards
PREFILL = 1.0 / 64      # gradient buffers accumulated into (no SDFR_ZERO_GRADS) start at this value
THR = 0.005
INLIER_REL = 0.03
NAN = float("nan")
NCPU = os.cpu_count() or 1


def _stream():
    return torch.cuda.current_stream().cuda_stream


class Buf:
    """A device output: `n` elements filled with `fill`, `offset` elements past a 16-byte boundary, GUARD
    sentinel elements on either side."""

    def __init__(self, n, fill, dev, offset=0, dtype=torch.float32):
        sent = SENTINEL if dtype.is_floating_point else int(SENTINEL)
        self.raw = torch.full((n + offset + 2 * GUARD,), sent, dtype=dtype, device=dev)
        self.lo, self.n, self.fill, self.sent = GUARD + offset, n, fill, sent
        self.body = self.raw[self.lo:self.lo + n]
        self.body.fill_(fill)

    @property
    def ptr(self):
        return self.body.data_ptr()

    def guards_intact(self):
        return bool((self.raw[:self.lo] == self.sent).all()) and bool((self.raw[self.lo + self.n:] == self.sent).all())


class HostScene:
    """The host-side inputs of one case: grids (dense), poses, camera, observation."""

    def __init__(self, c):
        self.c = c
        n = c.poses or c.B
        self.pidx = np.arange(c.B) % n  # pose (and grid) class of every hypothesis
        if c.tiled:
            k = np.arange(n)
            pos = np.stack([-0.35 + 0.1 * (k % 8), -0.2 + 0.1 * ((k // 8) % 5), c.z - 0.02 * (k % 3)], 1)
            hyp = syn.make_hypotheses(n, seed=7)
            inv = np.full(n, 1 / 0.06, np.float32)
        else:
            hyp = syn.make_hypotheses(n, seed=7, base_position=(0.02, -0.01, c.z))
            pos = hyp["position"].numpy().copy()
            pos[:, 0] += 0.12 * (np.arange(n) % 3 - 1)
            inv = hyp["inv_scale"].numpy()
        self.pos, self.inv = np.float32(pos), np.float32(inv)
        self.quat = hyp["orientation"].numpy().astype(np.float32)
        if c.grids == "shared":
            self.grids = syn.category_grid("mug", c.R, "cpu").numpy()[None]
            self.gidx = np.zeros(n, int)
        else:
            self.grids = syn.hypothesis_grids(hyp["shape_param"], c.R, "cpu").numpy()
            self.gidx = np.arange(n)
        f = c.f or c.W / 2
        self.cam = dict(cx=c.W / 2, cy=c.H / 2, fx=f, fy=f)
        # the observation: the first (up to) three pose classes, moved by 1 cm and scaled by 2 %
        k = range(min(n, 3))
        obs, _ = oracle.render_composite([self.grid(i) for i in k], self.pos[:3] + np.float32([0.01, 0, 0]),
                                         self.quat[:3], self.inv[:3] * np.float32(1.02), c.W, c.H, threshold=THR,
                                         nthreads=NCPU, **self.cam)
        if c.obs == "per":
            self.obs = np.stack([obs * np.float32(1 + 0.01 * (b % 7)) for b in range(c.B)])
            self.obs[-1] = 0  # a hypothesis without overlap: n_overlap == 0
            self.obs_stride = c.W * c.H
        else:
            self.obs, self.obs_stride = obs, 0
        self.upstream = np.float32(0.5 + 0.25 * (self.pidx % 5))  # the same within a pose class
        self.reps = [int(np.flatnonzero(self.pidx == k)[0]) for k in range(n)]  # first hypothesis of each class

    # the oracle's view of pose class k
    def pose(self, k):
        return self.pos[k], self.quat[k], self.inv[k]

    def grid(self, k):
        return self.grids[self.gidx[k]]

    def obs_of(self, b):
        return self.obs[b] if self.c.obs == "per" else self.obs

    def members(self, k):
        return np.flatnonzero(self.pidx == k)


class Scene(HostScene):
    """The device inputs of one case: grids in the case's layout, poses, bounds, observation."""

    def __init__(self, c, dev):
        super().__init__(c)
        self.dev = dev
        lib = _lib.lib()
        dense = torch.as_tensor(self.grids, device=dev).reshape(len(self.grids), -1)
        if c.grids == "per":
            dense = dense[torch.as_tensor(self.pidx, device=dev)].contiguous()
        n_dev = dense.shape[0]
        if c.layout == SKEWED:
            elems = ctypes.c_longlong(0)
            _lib.check(lib.sdfr_skewed_pitches(c.R, None, None, ctypes.byref(elems)), "sdfr_skewed_pitches")
            self.sdf = torch.zeros(n_dev, elems.value, device=dev)
            _lib.check(lib.sdfr_skew_grids(dense.data_ptr(), c.R, c.R ** 3, n_dev, self.sdf.data_ptr(), elems.value,
                                           _stream()), "sdfr_skew_grids")
            stride = elems.value
        else:
            self.sdf, stride = dense, c.R ** 3
        self.sdf_stride = 0 if c.grids == "shared" else stride
        cycle = lambda a: torch.as_tensor(np.ascontiguousarray(a[self.pidx]), device=dev)  # noqa: E731
        self.t_pos, self.t_quat, self.t_inv = cycle(self.pos), cycle(self.quat), cycle(self.inv)
        self.bounds = None
        if c.bounds:
            self.bounds = torch.zeros(n_dev, 8, dtype=torch.int32, device=dev)
            _lib.check(lib.sdfr_grid_bounds(self.sdf.data_ptr(), c.R, self.sdf_stride, c.layout, self.t_pos.data_ptr(),
                                            self.t_inv.data_ptr(), c.B, THR, self.bounds.data_ptr(), _stream()),
                       "sdfr_grid_bounds")
        self.t_obs = torch.as_tensor(np.ascontiguousarray(self.obs), device=dev)
        self.t_upstream = torch.as_tensor(self.upstream, device=dev)

    def common(self):
        c = self.c
        return (self.sdf.data_ptr(), c.R, self.sdf_stride, c.layout, self.t_pos.data_ptr(), self.t_quat.data_ptr(),
                self.t_inv.data_ptr())

    def camera(self):
        c, m = self.c, self.cam
        return (c.W, c.H, m["cx"], m["cy"], m["fx"], m["fy"])

    def bounds_ptr(self):
        return None if self.bounds is None else self.bounds.data_ptr()


def _grad_bufs(s, call, n_objects):
    c, dev, off = s.c, s.dev, call.offset
    fill = NAN if call.flags & Z else PREFILL
    stride = _gs_stride(c.R, call.gs)
    return dict(gsdf=Buf(c.R ** 3 if stride == 0 else n_objects * stride, fill, dev, off),
                gpos=Buf(3 * n_objects, fill, dev, off), gquat=Buf(4 * n_objects, fill, dev, off),
                ginv=Buf(n_objects, fill, dev, off), gs_stride=stride)


def _grad_args(o):
    return (o["gsdf"].ptr, o["gs_stride"], o["gpos"].ptr, o["gquat"].ptr, o["ginv"].ptr)


def _face_masked(s, k, depth, seed):
    """A random upstream image, zero on the pixels whose hit point lies on a cell face (tests/util.py)."""
    c = s.c
    g = np.random.default_rng(seed).standard_normal((c.H, c.W)).astype(np.float32)
    p, q, i = s.pose(k)
    g[cell_face_mask(depth, p, q, i, c.R, **s.cam)] = 0
    return g


def run_call(s, call, i):
    """The launches of one call into fresh outputs; returns the outputs and the upstream images used."""
    c, dev, lib, st = s.c, s.dev, _lib.lib(), _stream()
    B, HW, off, fl = c.B, c.H * c.W, call.offset, call.flags
    o = dict(call=call)
    if call.entry == "composite":
        o["depth"] = Buf(HW, NAN, dev, off)
        o["winner"] = Buf(HW, -99, dev, off, torch.int32)
        _lib.check(lib.sdfr_forward_composite(*s.common(), B, *s.camera(), THR, o["depth"].ptr, o["winner"].ptr,
                                              s.bounds_ptr(), st), "sdfr_forward_composite")
        if fl & ALL:
            o.update(_grad_bufs(s, call, B))
            d = o["depth"].body.view(c.H, c.W).cpu().numpy()
            w = o["winner"].body.view(c.H, c.W).cpu().numpy()
            g = np.random.default_rng(100 + i).standard_normal((c.H, c.W)).astype(np.float32)
            for k in range(B):
                p, q, inv = s.pose(k)
                g[cell_face_mask(np.where(w == k, d, 0), p, q, inv, c.R, **s.cam)] = 0
            o["g"] = g
            tg = torch.as_tensor(g, device=dev)
            _lib.check(lib.sdfr_backward_composite(tg.data_ptr(), o["depth"].ptr, o["winner"].ptr, *s.common(), B,
                                                   *s.camera(), *_grad_args(o), fl, st), "sdfr_backward_composite")
        return o
    o["depth"] = Buf(B * HW, NAN, dev, off)
    if call.entry in ("forward", "backward"):
        _lib.check(lib.sdfr_forward(*s.common(), B, *s.camera(), THR, o["depth"].ptr, s.bounds_ptr(), st),
                   "sdfr_forward")
    elif call.entry == "forward_stats":
        o["stats"] = Buf(4, 0, dev, 0, torch.int64)
        _lib.check(lib.sdfr_forward_stats(*s.common(), B, *s.camera(), THR, o["depth"].ptr, o["stats"].ptr, None, st),
                   "sdfr_forward_stats")
    elif call.entry in ("compare_forward", "compare_backward"):
        o["loss"], o["n"] = Buf(B, NAN, dev, off), Buf(B, NAN, dev, off)
        _lib.check(lib.sdfr_compare_forward(*s.common(), B, *s.camera(), THR, s.t_obs.data_ptr(), s.obs_stride,
                                            o["depth"].ptr, o["loss"].ptr, o["n"].ptr, Z, s.bounds_ptr(), st),
                   "sdfr_compare_forward")
    else:  # the fused compare
        o["loss"], o["n"] = Buf(B, NAN, dev, off), Buf(B, NAN, dev, off)
        o.update(_grad_bufs(s, call, B))
        head = (*s.common(), B, *s.camera(), THR, s.t_obs.data_ptr(), s.obs_stride, o["depth"].ptr, o["loss"].ptr,
                o["n"].ptr)
        if call.entry == "compare_fused_inliers":
            o["inl"] = Buf(B, NAN, dev, off)
            _lib.check(lib.sdfr_compare_fused_inliers(*head, INLIER_REL, o["inl"].ptr, *_grad_args(o), fl,
                                                      s.bounds_ptr(), st), "sdfr_compare_fused_inliers")
        else:
            _lib.check(lib.sdfr_compare_fused(*head, *_grad_args(o), fl, s.bounds_ptr(), st), "sdfr_compare_fused")
        if fl & ALL:
            up = s.t_upstream.data_ptr() if call.upstream else None
            _lib.check(lib.sdfr_scale_grads(o["n"].ptr, up, c.R, B, *_grad_args(o), fl, s.bounds_ptr(),
                                            1 if s.sdf_stride else 0, st), "sdfr_scale_grads")
    if call.entry == "backward":
        o.update(_grad_bufs(s, call, B))
        depth = o["depth"].body.view(B, c.H, c.W)
        # one upstream image per pose class (the slice case cycles four poses over 65539 hypotheses)
        gk = [_face_masked(s, k, depth[r].cpu().numpy(), 10 * i + k) for k, r in enumerate(s.reps)]
        o["g"] = gk
        tg = torch.as_tensor(np.stack(gk), device=dev)[torch.as_tensor(s.pidx, device=dev)].contiguous()
        _lib.check(lib.sdfr_backward(tg.data_ptr(), o["depth"].ptr, *s.common(), B, *s.camera(), *_grad_args(o), fl,
                                     s.bounds_ptr(), st), "sdfr_backward")
    elif call.entry == "compare_backward":
        o.update(_grad_bufs(s, call, B))
        up = s.t_upstream.data_ptr() if call.upstream else None
        _lib.check(lib.sdfr_compare_backward(o["depth"].ptr, s.t_obs.data_ptr(), s.obs_stride, o["n"].ptr, up,
                                             *s.common(), B, *s.camera(), *_grad_args(o), fl, s.bounds_ptr(), st),
                   "sdfr_compare_backward")
    return o


def run_case(s, i=0):
    return [run_call(s, call, i) for call in s.c.calls]


_RESULTS = {}


def results(name, dev):
    """Scene, first run and second run of a case (each case runs once per session)."""
    if name not in _RESULTS:
        s = Scene(BY_NAME[name], dev)
        first, second = run_case(s), run_case(s)
        torch.cuda.synchronize()
        _RESULTS[name] = (s, first, second)
    return _RESULTS[name]


def _depth(s, o):
    c = s.c
    return o["depth"].body.view(-1, c.H, c.W)


def _cases_with(pred):
    return [c.name for c in CASES if any(pred(call) for call in c.calls)]


# --- coverage ------------------------------------------------------------------------------
def _requested(call, key):
    fl = call.flags
    return {"gsdf": fl & SDF, "gpos": fl & _lib.GRAD_POSITION, "gquat": fl & _lib.GRAD_ORIENTATION,
            "ginv": fl & _lib.GRAD_INV_SCALE}.get(key, True)


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASE_IDS)
def test_every_output_written_guards_intact_and_reproducible(cuda_device, name):
    s, first, second = results(name, cuda_device)
    c = s.c
    for o, o2 in zip(first, second):
        call = o["call"]
        for key, buf in o.items():
            if not isinstance(buf, Buf):
                continue
            what = f"{call}: {key}"
            assert buf.guards_intact(), f"{what}: guard elements overwritten"
            if key == "stats":  # counters, accumulated into a zeroed buffer
                continue
            body = buf.body
            if key == "gsdf" and call.gs == "padded":  # the padding between the grids is never touched
                pad = body.view(c.B, -1)[:, c.R ** 3:]
                assert bool(pad.isnan().all() if call.flags & Z else (pad == PREFILL).all()), f"{what}: padding"
                body = body.view(c.B, -1)[:, :c.R ** 3]
            if not _requested(call, key):
                assert bool(body.isnan().all() if call.flags & Z else (body == PREFILL).all()), f"{what}: not requested"
            elif body.dtype.is_floating_point:
                assert not bool(body.isnan().any()), f"{what}: {int(body.isnan().sum())} elements not written"
            else:
                assert not bool((body == buf.fill).any()), f"{what}: elements not written"
        for key in ("depth", "n", "winner"):
            if key in o:
                assert torch.equal(o[key].body, o2[key].body), f"{call}: {key} differs between two launches"
    # every render of the same hypotheses gives the same depth, whatever the mode, gradients or bounds
    plain = [o for o in first if o["call"].entry != "composite"]
    for o in plain[1:]:
        assert torch.equal(o["depth"].body, plain[0]["depth"].body), f"{o['call']}: depth differs from {plain[0]['call']}"


# --- depth ---------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", _cases_with(lambda call: call.entry != "composite"))
def test_depth_matches_oracle(cuda_device, name):
    s, first, _ = results(name, cuda_device)
    c = s.c
    o = next(o for o in first if o["call"].entry != "composite")
    depth = _depth(s, o)
    got, ref = [], []
    for k, r in enumerate(s.reps):
        got.append(depth[r].cpu().numpy())
        ref.append(oracle.render(s.grid(k), *s.pose(k), c.W, c.H, threshold=THR, nthreads=NCPU, **s.cam))
        assert (ref[-1] > 0).sum() > 10, f"pose class {k} hits nothing"
    # one gate over the case's hypotheses: at a few hundred hit pixels per hypothesis, a single step flip
    # would otherwise already exceed the 0.1 % that the gate leaves to them
    depth_parity(np.stack(got), np.stack(ref), THR)
    if c.poses:  # every hypothesis renders bit for bit what the first of its pose class renders
        pidx = torch.as_tensor(s.pidx, device=cuda_device)
        reps = depth[torch.as_tensor(s.reps, device=cuda_device)]
        assert torch.equal(depth, reps[pidx])


@pytest.mark.gpu
def test_every_slice_equals_single_launches(cuda_device):
    """The slice case: each of the 65 539 hypotheses renders and counts exactly what a launch of its pose
    alone does."""
    s, first, _ = results("slices", cuda_device)
    c, lib = s.c, _lib.lib()
    pidx = torch.as_tensor(s.pidx, device=cuda_device)
    one_depth, one_n = [], []
    for k, r in enumerate(s.reps):
        d, loss, n = torch.empty(c.H, c.W, device=cuda_device), torch.empty(1, device=cuda_device), torch.empty(1, device=cuda_device)
        ptrs = (s.sdf[r].data_ptr(), c.R, c.R ** 3, c.layout, s.t_pos[r].data_ptr(), s.t_quat[r].data_ptr(),
                s.t_inv[r].data_ptr())
        _lib.check(lib.sdfr_compare_forward(*ptrs, 1, *s.camera(), THR, s.t_obs.data_ptr(), 0, d.data_ptr(),
                                            loss.data_ptr(), n.data_ptr(), Z, None, _stream()), "sdfr_compare_forward")
        one_depth.append(d)
        one_n.append(n)
    one_depth, one_n = torch.stack(one_depth), torch.cat(one_n)
    for o in first:
        assert torch.equal(_depth(s, o), one_depth[pidx]), f"{o['call']}: depth"
        if "n" in o:
            assert torch.equal(o["n"].body, one_n[pidx]), f"{o['call']}: n_overlap"
    assert float(one_n.min()) > 0


# --- compare sums --------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", _cases_with(lambda call: "compare" in call.entry))
def test_compare_sums_match_oracle(cuda_device, name):
    s, first, _ = results(name, cuda_device)
    for o in first:
        if "n" not in o:
            continue
        depth = _depth(s, o)
        loss, n = o["loss"].body.cpu().numpy(), o["n"].body.cpu().numpy()
        inl = o["inl"].body.cpu().numpy() if "inl" in o else None
        for k, r in enumerate(s.reps):
            d, obs = depth[r].cpu().numpy(), s.obs_of(r)
            lo, _, n_or = oracle.l1_depth_loss(d, obs)
            members = s.members(k)
            assert (n[members] == n_or).all(), (o["call"], k, n_or, np.unique(n[members]))
            assert np.abs(loss[members] - lo * n_or).max() <= 1e-5 * lo * n_or, (o["call"], k, lo * n_or)
            if inl is not None:
                with np.errstate(divide="ignore", invalid="ignore"):
                    rel = np.abs(obs - d) / obs  # IEEE float32, the expression the kernel evaluates
                want = int(((rel < np.float32(INLIER_REL)) & (obs > 0) & (d > 0)).sum())
                assert (inl[members] == want).all(), (o["call"], k, want, np.unique(inl[members]))
        if s.c.obs == "per":
            assert n[-1] == 0 and loss[-1] == 0


# --- forward statistics --------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", _cases_with(lambda call: call.entry == "forward_stats"))
def test_forward_stats_match_oracle(cuda_device, name):
    s, first, _ = results(name, cuda_device)
    c, lib = s.c, _lib.lib()
    o = next(o for o in first if o["call"].entry == "forward_stats")
    stats = o["stats"].body.cpu().numpy()
    steps = hits = 0
    for k in range(len(s.reps)):
        d, st, _ = oracle.render(s.grid(k), *s.pose(k), c.W, c.H, threshold=THR, extras=True, nthreads=NCPU, **s.cam)
        steps += int(st.sum()) * len(s.members(k))
        hits += int((d > 0).sum()) * len(s.members(k))
    assert abs(int(stats[0]) - steps) <= 2e-3 * steps, (stats, steps)
    assert abs(int(stats[2]) - hits) <= 5, (stats, hits)
    assert stats[3] == 0
    # the counters are integers: a batched launch counts exactly what one launch per hypothesis counts
    total = torch.zeros(4, dtype=torch.int64, device=cuda_device)
    d = torch.empty(c.H, c.W, device=cuda_device)
    for b in range(c.B):
        sdf = s.sdf[0] if s.sdf_stride == 0 else s.sdf[b]
        _lib.check(lib.sdfr_forward_stats(sdf.data_ptr(), c.R, 0, c.layout, s.t_pos[b].data_ptr(), s.t_quat[b].data_ptr(),
                                          s.t_inv[b].data_ptr(), 1, *s.camera(), THR, d.data_ptr(), total.data_ptr(),
                                          None, _stream()), "sdfr_forward_stats")
    assert (total.cpu().numpy() == stats).all(), (total, stats)


# --- gradients -----------------------------------------------------------------------------
def _worst(got, ref):
    """Per component, the member whose value is furthest from the reference (m, ...) -> (...)."""
    idx = np.abs(got - ref[None]).argmax(0)
    return np.take_along_axis(got, idx[None], 0)[0]


def _check_grads(s, o, bws, gs_up, what):
    """bws[k]: oracle backward of pose class (or object) k with upstream image gs_up[k]."""
    c, call = s.c, o["call"]
    base = 0.0 if call.flags & Z else PREFILL
    n_obj = len(bws)
    members = [s.members(k) for k in range(n_obj)] if call.entry != "composite" else [np.array([k]) for k in range(n_obj)]
    if call.flags & POSE:
        gp = o["gpos"].body.cpu().numpy().reshape(-1, 3).astype(np.float64) - base
        gq = o["gquat"].body.cpu().numpy().reshape(-1, 4).astype(np.float64) - base
        gi = o["ginv"].body.cpu().numpy().astype(np.float64) - base
        for k, (bw, m) in enumerate(zip(bws, members)):
            got = (_worst(gp[m], bw["g_position"]), _worst(gq[m], bw["g_orientation"]),
                   _worst(gi[m], np.float64(bw["g_inv_scale"])))
            p, _, inv = s.pose(k)
            pose_grad_parity(got, bw, gs_up[k], what=f"{what} [{k}]", position=p, inv_scale=inv)
    if call.flags & SDF:
        gsdf = o["gsdf"].body
        if call.gs == "shared":
            got = gsdf.cpu().numpy().astype(np.float64) - base
            ref = sum(bw["g_sdf"].reshape(-1) * len(m) for bw, m in zip(bws, members))
            bound = max(np.abs(g).max() / s.pose(k)[2] for k, g in enumerate(gs_up))
            sdf_grad_parity(got, ref, pixel_bound=bound, max_flip_pixels=4 * c.B, what=f"{what} shared sdf")
        else:
            per = gsdf.view(-1, o["gs_stride"])[:, :c.R ** 3]
            for k, (bw, m) in enumerate(zip(bws, members)):
                got = _worst(per[torch.as_tensor(m, device=gsdf.device)].cpu().numpy().astype(np.float64) - base,
                             bw["g_sdf"].reshape(-1))
                sdf_grad_parity(got, bw["g_sdf"].reshape(-1), pixel_bound=np.abs(gs_up[k]).max() / s.pose(k)[2],
                                what=f"{what} sdf [{k}]")


@pytest.mark.gpu
@pytest.mark.parametrize("name", _cases_with(lambda call: call.entry != "composite" and call.flags & ALL))
def test_gradients_match_oracle(cuda_device, name):
    s, first, _ = results(name, cuda_device)
    c = s.c
    for o in first:
        call = o["call"]
        if call.entry == "composite" or not call.flags & ALL:
            continue
        mode = "exact" if call.flags & X else "reference"
        depth = _depth(s, o)
        bws, ups = [], []
        for k, r in enumerate(s.reps):
            d = depth[r].cpu().numpy()
            if call.entry == "backward":
                g = o["g"][k]
            else:  # d loss_r / d depth of the masked L1 (sum over pixels / n_overlap), times upstream[r]
                _, g, _ = oracle.l1_depth_loss(d, s.obs_of(r))
                g = (g * (s.upstream[r] if call.upstream else 1.0)).astype(np.float32)
            ups.append(g)
            bws.append(oracle.render_backward(g, d, s.grid(k), *s.pose(k), c.W, c.H, sdf_grad_mode=mode,
                                              want_sdf=bool(call.flags & SDF), want_deriv=True, nthreads=NCPU, **s.cam))
        _check_grads(s, o, bws, ups, str(call))


# --- composite -----------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", _cases_with(lambda call: call.entry == "composite"))
def test_composite_matches_oracle(cuda_device, name):
    s, first, _ = results(name, cuda_device)
    c = s.c
    grids = [s.grid(k) for k in range(c.B)]
    d_or, w_or = oracle.render_composite(grids, s.pos, s.quat, s.inv, c.W, c.H, threshold=THR, nthreads=NCPU, **s.cam)
    for o in first:
        call = o["call"]
        if call.entry != "composite":
            continue
        d = o["depth"].body.view(c.H, c.W).cpu().numpy()
        w = o["winner"].body.view(c.H, c.W).cpu().numpy()
        depth_parity(d, d_or, THR)
        assert (w == w_or).mean() >= 0.999, (call, (w != w_or).sum())
        assert len(set(np.unique(w)) - {-1}) >= min(c.B, 3)
        mode = "exact" if call.flags & X else "reference"
        bws = oracle.render_composite_backward(o["g"], d, w, grids, s.pos, s.quat, s.inv, c.W, c.H, sdf_grad_mode=mode,
                                               nthreads=NCPU, want_deriv=True, **s.cam)
        _check_grads(s, o, bws, [o["g"]] * c.B, str(call))


# --- the mirror on the device --------------------------------------------------------------
TRACE_KERNEL = re.compile(r"(?<![\w])(sdfr_\w+(?:<[^>]*>)?)")


@pytest.mark.gpu
def test_launches_are_the_ones_the_mirror_selects(cuda_device):
    """Every case's launches under torch.profiler: kernel names and grids equal `selected`'s."""
    from torch.profiler import ProfilerActivity, profile

    sm = torch.cuda.get_device_properties(cuda_device).multi_processor_count
    scenes = {c.name: Scene(c, cuda_device) for c in CASES}
    torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        for c in CASES:
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                run_case(scenes[c.name], 1)
                torch.cuda.synchronize()
            path = os.path.join(tmp, f"{c.name}.json")
            prof.export_chrome_trace(path)
            with open(path) as f:
                events = json.load(f)["traceEvents"]
            got = []
            for e in events:
                m = TRACE_KERNEL.search(e.get("name", "")) if e.get("cat") == "kernel" else None
                if m:
                    got.append((m.group(1), tuple(e["args"]["grid"])))
            want = [(l["kernel"], l["grid"]) for l in selected(c, sm)]
            assert sorted(got) == sorted(want), f"{c.name}: traced {sorted(got)}\nselected {sorted(want)}"
