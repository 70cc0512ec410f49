"""The C-ABI library loads and exports every symbol include/sdfrender.h declares; argument
validation works without a GPU (no kernel is launched by these calls)."""
import ctypes
import os
import re

import pytest

from sdfest_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "sdfrender.h")


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.lib()


def declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(sdfr_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_the_expected_entry_points():
    syms = declared_symbols()
    for s in ("sdfr_forward", "sdfr_backward", "sdfr_compare_forward", "sdfr_compare_backward",
              "sdfr_forward_composite", "sdfr_backward_composite", "sdfr_forward_stats",
              "sdfr_abi_version", "sdfr_last_error", "sdfr_build_info", "sdfr_max_steps"):
        assert s in syms


def test_library_exports_every_declared_symbol(lib):
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for s in declared_symbols():
        assert hasattr(raw, s), f"{s} declared in sdfrender.h but not exported"
    assert set(declared_symbols()) == set(_lib.SIGNATURES), "ctypes binding out of sync with header"


def test_version_and_build_info(lib):
    assert lib.sdfr_abi_version() == _lib.ABI_VERSION
    assert b"sm_100a" in lib.sdfr_build_info()
    assert lib.sdfr_max_steps() >= 1024


def test_flag_values_match_header():
    text = open(HEADER).read()
    for name, val in (("SDFR_GRAD_SDF", _lib.GRAD_SDF), ("SDFR_GRAD_POSITION", _lib.GRAD_POSITION),
                      ("SDFR_GRAD_ORIENTATION", _lib.GRAD_ORIENTATION),
                      ("SDFR_GRAD_INV_SCALE", _lib.GRAD_INV_SCALE),
                      ("SDFR_SDF_GRAD_EXACT", _lib.SDF_GRAD_EXACT),
                      ("SDFR_ZERO_GRADS", _lib.ZERO_GRADS)):
        m = re.search(rf"#define {name} (0x[0-9a-f]+)u", text)
        assert m and int(m.group(1), 16) == val


def test_argument_errors_need_no_gpu(lib):
    cam = (8, 8, 4.0, 4.0, 4.0, 4.0)
    # empty batch / empty image: success, nothing launched
    assert lib.sdfr_forward(None, 4, 0, 0, None, None, None, 0, *cam, 0.01, None, None, None) == 0
    assert lib.sdfr_forward(None, 4, 0, 0, None, None, None, 1, 0, 8, 4.0, 4.0, 4.0, 4.0, 0.01,
                            None, None, None) == 0
    # NULL inputs
    assert lib.sdfr_forward(None, 4, 0, 0, None, None, None, 1, *cam, 0.01, None, None, None) == -1
    assert b"NULL" in lib.sdfr_last_error()
    # bad resolution / negative sizes
    assert lib.sdfr_forward(None, 1, 0, 0, None, None, None, 1, *cam, 0.01, None, None, None) == -2
    assert lib.sdfr_forward(None, 4, 0, 0, None, None, None, -1, *cam, 0.01, None, None, None) == -2
    assert lib.sdfr_forward(None, 4, -5, 0, None, None, None, 1, *cam, 0.01, None, None, None) == -2
    # unknown flags in backward
    assert lib.sdfr_backward(None, None, None, 4, 0, 0, None, None, None, 0, *cam, None, 0, None,
                             None, None, 0x8000, None, None) == -3
    # grid bounds: empty batch is a no-op, NULL pointers and bad sizes are argument errors
    assert lib.sdfr_grid_bounds(None, 64, 0, 0, None, None, 0, 0.005, None, None) == 0
    assert lib.sdfr_grid_bounds(None, 64, 0, 0, None, None, 1, 0.005, None, None) == -1
    assert lib.sdfr_grid_bounds(None, 1, 0, 0, None, None, 1, 0.005, None, None) == -2
    assert lib.sdfr_grid_bounds(None, 64, 0, 0, None, None, 1, -1.0, None, None) == -2
    with pytest.raises(RuntimeError, match="argument error"):
        _lib.check(-1, "sdfr_forward")


def test_skewed_layout_geometry():
    """Pitches of the bank-conflict-free layout: pitch_y = 3, pitch_x = 9 (mod 32), no overlap."""
    import ctypes

    lib = _lib.lib()
    for R in (2, 16, 24, 32, 48, 64, 100, 128):
        py, px, n = ctypes.c_int(0), ctypes.c_int(0), ctypes.c_longlong(0)
        assert lib.sdfr_skewed_pitches(R, ctypes.byref(py), ctypes.byref(px), ctypes.byref(n)) == 0
        assert py.value >= R and py.value % 32 == 3 and py.value < R + 32
        assert px.value >= R * py.value and px.value % 32 == 9 and px.value < R * py.value + 32
        assert n.value == R * px.value
    assert lib.sdfr_skewed_pitches(64, None, None, None) == 0
    assert lib.sdfr_skewed_pitches(1, None, None, None) == -2
    # argument checks of the copy (nothing is launched)
    assert lib.sdfr_skew_grids(None, 64, 0, 0, None, 0, None) == 0
    assert lib.sdfr_skew_grids(None, 64, 0, 1, None, 0, None) == -1
    # unknown layout id
    cam = (8, 8, 4.0, 4.0, 4.0, 4.0)
    assert lib.sdfr_forward(None, 4, 0, 7, None, None, None, 1, *cam, 0.01, None, None, None) == -3


def test_argument_errors_of_the_round_two_entry_points_and_an_unknown_layout_need_no_gpu():
    """Views, point constraint, slab minima, scale-with-bounds, tail-with-bounds, compare layout: empty work is a
    no-op, NULL / bad sizes and unknown layouts are reported before anything is launched."""
    import ctypes

    lib = _lib.lib()
    f3 = (ctypes.c_float * 3)(0.0, 1.0, 0.0)
    assert lib.sdfr_view_poses(None, None, None, None, None, 0, 4, None, None, None, None) == 0
    assert lib.sdfr_view_poses(None, None, None, None, None, 2, 0, None, None, None, None) == 0
    assert lib.sdfr_view_poses(None, None, None, None, None, 2, 4, None, None, None, None) == -1
    assert lib.sdfr_view_poses(None, None, None, None, None, -1, 4, None, None, None, None) == -2
    assert lib.sdfr_views_pull_back(None, None, 2, 0, *[None] * 8, 1.0, None, None, None, None, None, 0, None) == 0
    assert lib.sdfr_views_pull_back(None, None, 2, 3, *[None] * 8, 1.0, None, None, None, None, None, 0, None) == -1
    assert lib.sdfr_views_pull_back(None, None, 2, 3, *[None] * 8, 1.0, None, None, None, None, None, 0x1, None) == -3
    assert lib.sdfr_point_constraint(None, 0, f3, f3, 1.0, None, None, None) == 0
    assert lib.sdfr_point_constraint(None, 2, f3, f3, 1.0, None, None, None) == -1
    assert lib.sdfr_point_constraint(None, -2, f3, f3, 1.0, None, None, None) == -2
    assert lib.sdfr_grid_slab_minima(None, 64, 0, 0, 0, None, None) == 0
    assert lib.sdfr_grid_slab_minima(None, 64, 0, 0, 2, None, None) == -1
    assert lib.sdfr_grid_slab_minima(None, 1, 0, 0, 2, None, None) == -2
    assert lib.sdfr_grid_slab_minima(None, 64, 0, 5, 2, None, None) == -3
    assert lib.sdfr_bounds_from_minima(None, 64, 0, None, None, 0, 0.005, None, None) == 0
    assert lib.sdfr_bounds_from_minima(None, 64, 2, None, None, 2, 0.005, None, None) == -1
    assert lib.sdfr_bounds_from_minima(None, 64, 3, None, None, 2, 0.005, None, None) == -2  # 1 or batch grids
    assert lib.sdfr_bounds_from_minima(None, 64, 2, None, None, 2, -1.0, None, None) == -2
    assert lib.sdfr_scale_grads(None, None, 64, 0, None, 0, None, None, None, 0x0F, None, 0, None) == -1  # NULL buffers
    assert lib.sdfr_scale_grads(None, None, 64, 0, None, 0, None, None, None, 0, None, 0, None) == 0
    assert lib.sdfr_decoder_tail_forward_bounds(None, 4, 30, None, None, None, 0, 64, None, 0, 0, None, None, 0.005,
                                                None, None) == 0
    assert lib.sdfr_decoder_tail_forward_bounds(None, 4, 30, None, None, None, 2, 64, None, 0, 0, None, None, 0.005,
                                                None, None) == -1
    assert lib.sdfr_decoder_tail_forward_bounds(None, 40, 30, None, None, None, 2, 64, None, 0, 0, None, None, 0.005,
                                                None, None) == -2
    cam = (8, 8, 4.0, 4.0, 4.0, 4.0)
    # layout id 2 (the removed z-pair layout) is refused like any other unknown id, also at 64^3
    assert lib.sdfr_forward(None, 64, 0, 2, None, None, None, 1, *cam, 0.01, None, None, None) == -3
    assert lib.sdfr_compare_forward(None, 32, 0, 2, None, None, None, 1, *cam, 0.01, None, 0, None, None, None, 0,
                                    None, None) == -3
    assert lib.sdfr_compare_forward(None, 64, 0, 2, None, None, None, 1, *cam, 0.01, None, 0, None, None, None, 0,
                                    None, None) == -3


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "libsdfrender.so"))
    with pytest.raises(RuntimeError, match="no CPU or PyTorch fallback"):
        _lib.lib()


def _header_prototypes():
    """{name: [C parameter declarations]} for every function the header declares."""
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    protos = {}
    for m in re.finditer(r"\b(?:int|const char\*)\s+(sdfr_[a-z0-9_]+)\s*\(([^;]*?)\)\s*;", text, flags=re.S):
        params = [p.strip() for p in m.group(2).replace("\n", " ").split(",")]
        protos[m.group(1)] = [] if params == ["void"] else params
    return protos


def test_ctypes_signatures_match_the_header_prototypes():
    """Same number of parameters and the same kind of parameter (pointer / int / long long / unsigned /
    float) at every position: a silently shifted argument would corrupt a launch, not fail it."""
    from ctypes import c_float, c_int, c_longlong, c_uint, c_void_p

    protos = _header_prototypes()
    assert set(protos) == set(_lib.SIGNATURES)
    for name, params in protos.items():
        _, argtypes = _lib.SIGNATURES[name]
        assert len(params) == len(argtypes), f"{name}: header has {len(params)} parameters, binding {len(argtypes)}"
        for i, (decl, ct) in enumerate(zip(params, argtypes)):
            if "*" in decl:
                want = "pointer"
            elif decl.startswith("long long"):
                want = c_longlong
            elif decl.startswith("unsigned"):
                want = c_uint
            elif decl.startswith("float"):
                want = c_float
            elif decl.startswith("int"):
                want = c_int
            else:
                raise AssertionError(f"{name}: cannot classify parameter {decl!r}")
            if want == "pointer":
                ok = ct is c_void_p or (isinstance(ct, type) and issubclass(ct, ctypes._Pointer))
            else:
                ok = ct is want
            assert ok, f"{name}: parameter {i} is {decl!r} in the header but {ct} in the binding"
