"""CPU checks of typed (integer) volumes on the sharded and streamed routes: the C ABI of the typed re-slab kernels, the
routing of `keep_dtype` volumes that do not stay in core (memory maps, several devices, volumes larger than the device)
to typed streaming, the buffer roles of that route (with a CPU stand-in for StreamingDenoiser built on the integer
oracle), and the combinations that are still rejected. Nothing here needs a device."""
import ctypes as C
import hashlib
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import fd_oracle as O
from oracle import fd_oracle_int as I
from oracle import gen_golden_integer as G


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _lib_or_skip():
    from flowdenoising_b200 import _lib
    try:
        return _lib.load()
    except Exception as e:   # no nvcc here and no build
        pytest.skip(f"libfdn_b200.so not available: {e}")


# ---- C ABI ----
def test_typed_reslab_symbols_and_version():
    from flowdenoising_b200 import _lib
    lib = _lib_or_skip()
    assert lib.fdn_version() == 101
    for name in ("fdn_copy3d_typed", "fdn_transpose_strided_typed", "fdn_copy3d", "fdn_transpose_strided"):
        assert name in _lib.SIGNATURES and hasattr(lib, name)
    assert C.sizeof(_lib.OfParams) == 32 and C.sizeof(_lib.View) == 56


def test_typed_reslab_calls_reject_bad_dtype():
    from flowdenoising_b200 import _lib
    lib = _lib_or_skip()
    dummy = C.c_void_p(16)   # never dereferenced: every call below fails its argument checks first
    for bad in (-1, 5, 9):
        assert lib.fdn_copy3d_typed(dummy, bad, 1, 1, 0, 1, 0, 1, dummy, 1, 1, 1, 1, 1, None) == 1
        assert b"unknown dtype" in lib.fdn_last_error()
        assert lib.fdn_transpose_strided_typed(dummy, bad, 1, 1, dummy, 1, 1, 1, 1, 1, None) == 1
        assert b"unknown dtype" in lib.fdn_last_error()
    assert lib.fdn_copy3d_typed(dummy, _lib.DTYPE_U16, 1, 1, 0, 1, 0, 1, dummy, 1, 1, 0, 1, 1, None) == 1
    assert b"bad argument" in lib.fdn_last_error()
    assert lib.fdn_copy3d_typed(dummy, _lib.DTYPE_U8, 1, 1, 0, 0, 0, 1, dummy, 1, 1, 1, 1, 1, None) == 1
    assert b"wrap" in lib.fdn_last_error()
    assert lib.fdn_transpose_strided_typed(None, _lib.DTYPE_I16, 1, 1, dummy, 1, 1, 1, 1, 1, None) == 1


# ---- routing ----
def _fake_engine(monkeypatch, free):
    from flowdenoising_b200 import flowdenoising as F
    eng = SimpleNamespace(device="cuda:0", torch=SimpleNamespace(cuda=SimpleNamespace(mem_get_info=lambda d: (free, free))))
    monkeypatch.setattr(F, "_get_engine", lambda: eng)
    return F


def test_integer_memmap_and_several_devices_route_to_typed_streaming(monkeypatch, tmp_path):
    F = _fake_engine(monkeypatch, 1 << 40)
    path = tmp_path / "v.raw"
    np.arange(4 * 8 * 8, dtype=np.uint16).reshape(4, 8, 8).tofile(path)
    mm = np.memmap(path, dtype=np.uint16, mode="r", shape=(4, 8, 8))
    d = F.GaussianDenoising(1, mm, keep_dtype=True)
    assert d._typed() is True and d._streaming_needed() is True
    d = F.FlowDenoising(1, np.zeros((4, 8, 8), np.uint8), keep_dtype=True)
    d.devices = [0, 0]
    assert d._typed() is True and d._streaming_needed() is True
    d = F.GaussianDenoising(1, np.zeros((4, 8, 8), np.int16), keep_dtype=True)
    d.streaming = True
    assert d._typed() is True and d._streaming_needed() is True
    d = F.GaussianDenoising(1, np.zeros((4, 8, 8), np.int8), keep_dtype=True)
    assert d._typed() is True and d._streaming_needed() is False


def test_streaming_decision_sizes_with_the_itemsize(monkeypatch):
    """In core: the volume, two intermediates and the result in the pass dtype plus 2 GiB must fit 90 % of the free
    memory. A 1 M-voxel uint8 volume needs 4 MB of them as uint8 and 16 MB as float32."""
    n = 1 << 20
    F = _fake_engine(monkeypatch, int(((2 << 30) + 10 * n) / 0.9))
    vol = np.zeros((16, 256, 256), np.uint8)
    assert vol.size == n
    assert F.GaussianDenoising(1, vol, keep_dtype=True)._streaming_needed() is False
    assert F.GaussianDenoising(1, vol)._streaming_needed() is True              # the float route: 4 B/voxel
    F = _fake_engine(monkeypatch, int(((2 << 30) + 3 * n) / 0.9))               # "larger than the device"
    d = F.GaussianDenoising(1, vol, keep_dtype=True)
    assert d._typed() is True and d._streaming_needed() is True


def test_still_rejected_combinations(monkeypatch, tmp_path):
    F = _fake_engine(monkeypatch, 1 << 40)
    k = [O.get_gaussian_kernel(1.0)] * 3
    d = F.GaussianDenoising(1, np.zeros((4, 8, 8), np.uint8), keep_dtype=True)
    d.border = "mean"
    with pytest.raises(ValueError, match="streaming"):
        d.filter(k)
    d.devices = [0, 0]
    with pytest.raises(ValueError, match="mean"):
        d._typed()
    with pytest.raises(ValueError, match="int8"):
        F.FlowDenoising(1, np.zeros((4, 8, 8), np.int8), keep_dtype=True)._typed()
    with pytest.raises(ValueError, match="float16"):
        F.GaussianDenoising(1, np.zeros((4, 8, 8), np.float16), keep_dtype=True)._typed()
    path = tmp_path / "be.raw"
    np.zeros((4, 8, 8), ">u2").tofile(path)
    be = np.memmap(path, dtype=">u2", mode="r", shape=(4, 8, 8))
    with pytest.raises(ValueError, match="not supported"):
        F.GaussianDenoising(1, be, keep_dtype=True)._typed()


# ---- the streamed filter()'s buffer roles, on a CPU stand-in for StreamingDenoiser ----
class _OracleStreamer:
    """StreamingDenoiser's contract (filter_axis: one periodic pass of src into dst, typed when keep_dtype) computed by
    the integer oracle; records what it was given."""
    calls = []

    def __init__(self, flow, exact=True, border="wrap", slab_slices=None, devices=None, progress=None,
                 keep_dtype=False):
        assert keep_dtype is True and border == "wrap"
        self.flow = flow

    def filter_axis(self, src, dst, axis, kernel, mean=None):
        _OracleStreamer.calls.append((np.dtype(src.dtype), np.dtype(dst.dtype), axis))
        kw = {} if self.flow is None else dict(l=self.flow.levels, w=self.flow.winsize,
                                               recompute_flow=not self.flow.use_prev_flow)
        o = I.IntegerDenoiser(1, np.array(src), use_OF=self.flow is not None, backend="c", **kw)
        o.filter_along_axis(axis, kernel)
        np.copyto(dst, o.filtered_vol, casting="unsafe")

    def release(self):
        pass


@pytest.mark.parametrize("name,kind", [("uint16_noof", "array"), ("int8_noof", "readonly_map"),
                                       ("int16_noof", "float_result")])
def test_streamed_filter_buffer_roles(monkeypatch, tmp_path, golden, name, kind):
    from flowdenoising_b200 import streaming
    g = golden("integer_volumes.npz")
    F = _fake_engine(monkeypatch, 1 << 40)
    monkeypatch.setattr(streaming, "StreamingDenoiser", _OracleStreamer)
    _OracleStreamer.calls = []
    vol = G.case_volume(name)
    ks = [O.get_gaussian_kernel(s) for s in G.CASES[name][4]]
    if kind == "readonly_map":
        path = tmp_path / "v.raw"
        vol.tofile(path)
        src = np.memmap(path, dtype=vol.dtype, mode="r", shape=vol.shape)
    else:
        src = vol.copy()
    d = F.GaussianDenoising(1, src, keep_dtype=True)
    d.streaming = True
    if kind == "float_result":
        d.filtered_vol = np.full(vol.shape, np.nan, np.float32)     # e.g. the CLI's float32 output map
    res = d.filter(ks)
    assert res is d.filtered_vol
    assert [c[2] for c in _OracleStreamer.calls] == [0, 1, 2]
    assert all(c[0] == vol.dtype for c in _OracleStreamer.calls)           # every pass reads T ...
    assert all(c[1] == vol.dtype for c in _OracleStreamer.calls[:2])       # ... and the intermediates are T arrays
    assert sha(np.asarray(res).astype(vol.dtype)) == str(g[f"{name}_sha_ZYX"])
    if kind == "readonly_map":
        assert np.array_equal(np.asarray(src), vol)                        # a read-only map is left alone
    else:
        assert sha(d.vol) == str(g[f"{name}_sha_ZY"])                      # vol ends as the Z+Y intermediate
    assert d.progress == sum(vol.shape)
