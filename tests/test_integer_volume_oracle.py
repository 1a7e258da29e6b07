"""CPU checks of integer volumes (keep_dtype, SURVEY App. B Q3): the C restatement of cv2.remap on 8U / 16U / 16S
images against live cv2, the oracle drivers against each other, against the committed digests
(tests/golden/integer_volumes.npz, oracle/gen_golden_integer.py) and against live cv2, and the plumbing of the typed
C ABI and of the Python / CLI surface. No GPU needed."""
import ctypes as C
import hashlib

import numpy as np
import pytest

from oracle import fd_oracle as O
from oracle import fd_oracle_int as I
from oracle import gen_golden_integer as G

REMAP_DTYPES = [(np.uint8, 0, 255), (np.uint16, 0, 65535), (np.int16, -32768, 32767)]
TOY_CASES = [c for c in G.CASES if not c.startswith("cfg1")]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def fraction_map(H, W, rng, lo=-3, hi=None):
    """Absolute coordinates whose 1/32-px fractions run through all 32 x 32 pairs, on integer bases that reach past
    every border."""
    hi = max(H, W) + 3 if hi is None else hi
    ay, ax = np.divmod(np.arange(H * W) % 1024, 32)
    base = rng.integers(lo, hi, (H * W, 2))
    mx = (base[:, 0] + ax / 32.0).reshape(H, W)
    my = (base[:, 1] + ay / 32.0).reshape(H, W)
    return np.dstack([mx, my]).astype(np.float32)


def cv2_remap(src, m):
    cv2 = pytest.importorskip("cv2")
    return cv2.remap(src, m, None, interpolation=cv2.INTER_LINEAR, borderMode=cv2.BORDER_REPLICATE)


def test_fixed_point_table_is_exact():
    """All 1024 entries of the 8U table are the integers (32 - ay or ay) * (32 - ax or ax) * 32 that the CUDA remap
    computes in registers, except entry 0, which OpenCV saturates to 32767 and corrects on tap 3."""
    t = I.remap_table_8u().astype(np.int64)
    ay, ax = np.divmod(np.arange(1024), 32)
    closed = np.stack([(32 - ay) * (32 - ax), (32 - ay) * ax, ay * (32 - ax), ay * ax], axis=1) * 32
    assert np.array_equal(t[1:], closed[1:])
    assert list(t[0]) == [32767, 0, 0, 1]
    assert np.all(t.sum(axis=1) == 32768)


@pytest.mark.parametrize("dtype,lo,hi", REMAP_DTYPES, ids=lambda v: getattr(v, "__name__", str(v)))
def test_remap_every_fraction_vs_cv2(dtype, lo, hi):
    """Every one of the 32 x 32 fractional positions, inside and past the borders, on random pixels and on pixels
    at the two ends of the range (saturation)."""
    rng = np.random.default_rng(7)
    for H, W in [(32, 32), (64, 48)]:
        m = fraction_map(H, W, rng)
        for src in (rng.integers(lo, hi + 1, (H, W)), np.where(rng.random((H, W)) < 0.5, lo, hi)):
            src = src.astype(dtype)
            assert np.array_equal(I.remap(src, m), cv2_remap(src, m))


@pytest.mark.parametrize("dtype,lo,hi", REMAP_DTYPES, ids=lambda v: getattr(v, "__name__", str(v)))
def test_remap_random_maps_odd_sizes_vs_cv2(dtype, lo, hi):
    rng = np.random.default_rng(11)
    for H, W in [(5, 3), (37, 53), (1, 17), (61, 1), (33, 101)]:
        src = rng.integers(lo, hi + 1, (H, W)).astype(dtype)
        m = np.dstack([rng.uniform(-6, W + 6, (H, W)), rng.uniform(-6, H + 6, (H, W))]).astype(np.float32)
        assert np.array_equal(I.remap(src, m), cv2_remap(src, m))
        flow = rng.uniform(-2.5, 2.5, (H, W, 2)).astype(np.float32)   # the map as warp_slice builds it
        assert np.array_equal(I.warp_slice(src, flow), O.warp_slice(src, flow))


def test_remap_rejects_what_cv2_rejects():
    with pytest.raises(ValueError):
        I.remap(np.zeros((4, 4), np.int8), np.zeros((4, 4, 2), np.float32))
    with pytest.raises(ValueError):
        I.remap(np.zeros((4, 4), np.float16), np.zeros((4, 4, 2), np.float32))


def test_cv2_backend_keeps_the_dtype():
    """The cv2 backend of OracleDenoiser is the reference's integer semantics: an integer filtered_vol, and an
    integer remap whose rounding differs from "float remap, then truncate"."""
    vol = I.integer_volume((4, 32, 40), np.uint8, seed=3)
    d = O.OracleDenoiser(1, vol.copy(), use_OF=True, backend="cv2")
    assert d.filtered_vol.dtype == np.uint8
    d.filter_along_Z(O.get_gaussian_kernel(1.0))
    assert d.filtered_vol.dtype == np.uint8
    rng = np.random.default_rng(1)
    flow = rng.uniform(-1.5, 1.5, (32, 40, 2)).astype(np.float32)
    warped = O.warp_slice(vol[0], flow)
    assert warped.dtype == np.uint8
    as_float = O.warp_slice(vol[0].astype(np.float32), flow)
    assert np.any(warped != np.trunc(as_float).astype(np.uint8))


def test_fixture_inputs_are_reproducible(golden):
    g = golden("integer_volumes.npz")
    for name in G.CASES:
        assert sha(G.case_volume(name)) == str(g[f"{name}_input_sha"]), name


@pytest.mark.parametrize("name", TOY_CASES)
def test_c_backend_equals_golden(golden, name):
    """The C backend (integer remap restated in C, C Farneback) reproduces the digests written from live cv2."""
    g = golden("integer_volumes.npz")
    z, zy, zyx = G.run_case(name, backend="c")
    for tag, a in (("Z", z), ("ZY", zy), ("ZYX", zyx)):
        assert a.dtype == np.dtype(G.CASES[name][0])
        assert sha(a) == str(g[f"{name}_sha_{tag}"]), (name, tag)


@pytest.mark.parametrize("name", ["uint8_of", "int16_ofr", "uint16_noof", "int8_noof", "uint8_gw"])
def test_live_cv2_equals_golden(golden, name):
    pytest.importorskip("cv2")
    g = golden("integer_volumes.npz")
    z, zy, zyx = G.run_case(name, backend="cv2")
    for tag, a in (("Z", z), ("ZY", zy), ("ZYX", zyx)):
        assert sha(a) == str(g[f"{name}_sha_{tag}"]), (name, tag)


def test_integer_semantics_differ_from_the_float_route():
    """What keep_dtype is for: the float32 route (cast, filter, truncate once) is not the reference's result."""
    name = "uint8_of"
    _z, _zy, zyx = G.run_case(name, backend="c")
    vol = G.case_volume(name).astype(np.float32)
    d = O.OracleDenoiser(4, vol, use_OF=True, backend="c")
    f = d.filter([O.get_gaussian_kernel(s) for s in G.CASES[name][4]])
    assert np.any(np.trunc(f).astype(np.uint8) != zyx)


# ---- ABI and API plumbing (the library is loaded, nothing runs on a device) ----
def _lib_or_skip():
    from flowdenoising_b200 import _lib
    try:
        return _lib.load()
    except Exception as e:   # no nvcc here and no build
        pytest.skip(f"libfdn_b200.so not available: {e}")


def test_typed_symbols_and_version():
    from flowdenoising_b200 import _lib
    lib = _lib_or_skip()
    assert lib.fdn_version() == 101
    for name in ("fdn_workspace_bytes_typed", "fdn_filter_axis_typed", "fdn_gauss_axis_typed", "fdn_gauss_rows_typed",
                 "fdn_transpose_yx_typed", "fdn_remap_typed"):
        assert name in _lib.SIGNATURES and hasattr(lib, name)
    assert C.sizeof(_lib.OfParams) == 32
    assert (_lib.DTYPE_F32, _lib.DTYPE_U8, _lib.DTYPE_I8, _lib.DTYPE_U16, _lib.DTYPE_I16) == (0, 1, 2, 3, 4)


def test_typed_calls_reject_unsupported_combinations():
    from flowdenoising_b200 import _lib
    lib = _lib_or_skip()
    v = _lib.View(8, 8, 0, 1, 16, 16, 256, 16, 256, 16)
    of = _lib.OfParams(3, 5, 3, 5, 1.2, 1, 0)
    k = (C.c_double * 5)(0.1, 0.2, 0.4, 0.2, 0.1)
    dummy = C.c_void_p(16)   # never dereferenced: every call below fails its argument checks first
    assert lib.fdn_workspace_bytes_typed(C.byref(v), 5, C.byref(of), 0, _lib.DTYPE_U8) > 0
    assert lib.fdn_workspace_bytes_typed(C.byref(v), 5, C.byref(of), 0, _lib.DTYPE_F32) == \
        lib.fdn_workspace_bytes(C.byref(v), 5, C.byref(of), 0)
    assert lib.fdn_workspace_bytes_typed(C.byref(v), 5, C.byref(of), 0, _lib.DTYPE_I8) == 0
    assert b"int8" in lib.fdn_last_error()
    assert lib.fdn_workspace_bytes_typed(C.byref(v), 5, C.byref(of), 0, 9) == 0
    assert b"dtype" in lib.fdn_last_error()
    assert lib.fdn_filter_axis_typed(dummy, dummy, _lib.DTYPE_I8, C.byref(v), k, 5, C.byref(of), 0, dummy, 1 << 30,
                                     None) == 1
    assert b"int8" in lib.fdn_last_error()
    assert lib.fdn_filter_axis_typed(dummy, dummy, 7, C.byref(v), k, 5, None, 0, None, 0, None) == 1
    assert lib.fdn_gauss_axis_typed(dummy, dummy, _lib.DTYPE_U16, C.byref(v), k, 5, 0, None) == 1
    assert b"exact" in lib.fdn_last_error()
    assert lib.fdn_gauss_rows_typed(dummy, dummy, _lib.DTYPE_U8, 16, 16, k, 5, 0, None) == 1
    assert b"exact" in lib.fdn_last_error()
    assert lib.fdn_remap_typed(dummy, dummy, dummy, _lib.DTYPE_I8, 1, 4, 4, None) == 1
    assert lib.fdn_transpose_yx_typed(dummy, dummy, -1, 1, 4, 4, None) == 1


def test_api_and_cli_defaults():
    import inspect
    from flowdenoising_b200 import flowdenoising as F
    for cls in (F.GaussianDenoising, F.FlowDenoising):
        assert inspect.signature(cls.__init__).parameters["keep_dtype"].default is False
    args = F.build_parser().parse_args([])
    assert args.keep_dtype is False
    assert F.build_parser().parse_args(["--keep_dtype"]).keep_dtype is True
    help_text = F.build_parser().format_help()
    assert "--keep_dtype" in help_text and "integer arithmetic" in " ".join(help_text.split())


def test_keep_dtype_off_is_the_float_route():
    from flowdenoising_b200 import flowdenoising as F
    vol = np.zeros((4, 8, 8), np.uint8)
    assert F.GaussianDenoising(1, vol)._typed() is False
    assert F.FlowDenoising(1, np.zeros((4, 8, 8), np.float32), keep_dtype=True)._typed() is False
