"""CPU tests of the batch surface that need no device: filter_volumes' grouping by shape, result order and host
sub-batches on an oracle-backed stand-in engine, the C ABI's argument checks of the batch entry points, and the
--inputs / --output_dir CLI (rejections and output naming)."""
import ctypes as C
import os
import struct

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from flowdenoising_b200 import _lib  # noqa: E402
from flowdenoising_b200 import flowdenoising as fd  # noqa: E402
from flowdenoising_b200 import volume_io  # noqa: E402

FDN_ERR_INVALID = 1   # include/fdn_b200.h


class _FakeCuda:
    """Stream / event stand-ins (copies on CPU tensors are synchronous) and a chosen amount of free memory."""
    free = 1 << 40

    class Event:
        def record(self, stream=None):
            pass

        def synchronize(self):
            pass

    class _Stream:
        def synchronize(self):
            pass

    @classmethod
    def current_stream(cls):
        return cls._Stream()

    @classmethod
    def mem_get_info(cls, _dev):
        return cls.free, cls.free


class _FakeTorch:
    cuda = _FakeCuda

    def __getattr__(self, name):
        return getattr(torch, name)


class _BatchEngine:
    """Stand-in for DeviceEngine.filter_batch: each volume of the batch through the C oracle's filter()."""

    def __init__(self):
        self.torch = _FakeTorch()
        self.device = torch.device("cpu")
        self.batches = []

    def filter_batch(self, vols, kernels, flow, exact=True):
        from oracle import fd_oracle as O
        assert vols.dtype == torch.float32 and vols.dim() == 4 and vols.is_contiguous()
        self.batches.append(tuple(vols.shape))
        zy, zyx = torch.empty_like(vols), torch.empty_like(vols)
        for g in range(vols.shape[0]):
            kw = {} if flow is None else dict(l=flow.levels, w=flow.winsize, recompute_flow=not flow.use_prev_flow)
            o = O.OracleDenoiser(1, vols[g].numpy().copy(), use_OF=flow is not None, backend="c", **kw)
            zyx[g] = torch.from_numpy(o.filter(kernels))
            zy[g] = torch.from_numpy(o.vol)
        return zy, zyx


class _CpuDownload:
    def __init__(self, t, dst, _torch):
        np.copyto(dst, t.numpy(), casting="unsafe")

    def wait(self):
        pass


@pytest.fixture
def batch_engine(monkeypatch):
    eng = _BatchEngine()
    monkeypatch.setattr(fd, "_get_engine", lambda: eng)
    monkeypatch.setattr(fd, "_Download", _CpuDownload)
    monkeypatch.setattr(fd, "_pinned_pair", lambda t: [torch.empty(fd._STAGE_BYTES // 4, dtype=torch.float32)
                                                       for _ in range(2)])
    monkeypatch.setattr(_FakeCuda, "free", 1 << 40)
    return eng


def _vols(shapes, dtype=np.float32):
    from oracle import fd_oracle as O
    return [np.clip(O.synthetic_volume(s, seed=20 + i, noise_sigma=6.0), 0, 255).astype(dtype)
            for i, s in enumerate(shapes)]


def _oracle(vol, kernels, of):
    from oracle import fd_oracle as O
    o = O.OracleDenoiser(1, np.asarray(vol, np.float32).copy(), use_OF=of, l=2, w=5, backend="c")
    return o.filter(kernels)


def test_filter_volumes_groups_by_shape_and_keeps_the_input_order(batch_engine):
    from oracle import fd_oracle as O
    shapes = [(6, 10, 12), (5, 8, 9), (6, 10, 12), (5, 8, 9), (6, 10, 12), (3, 4, 5)]
    vols = _vols(shapes)
    vols[3] = vols[3].astype(np.uint8)          # any dtype NumPy casts: filtered as float32
    kernels = [O.get_gaussian_kernel(0.5), O.get_gaussian_kernel(0.5), O.get_gaussian_kernel(0.75)]
    res = fd.filter_volumes(vols, kernels, l=2, w=5, no_OF=True)
    assert [r.shape for r in res] == shapes and all(r.dtype == np.float32 for r in res)
    for v, r in zip(vols, res):
        assert np.array_equal(r, _oracle(v, kernels, False))
    # one device batch per shape, in order of first appearance
    assert batch_engine.batches == [(3, 6, 10, 12), (2, 5, 8, 9), (1, 3, 4, 5)]


def test_filter_volumes_with_optical_flow_and_a_4d_array(batch_engine):
    from oracle import fd_oracle as O
    vols = np.stack(_vols([(6, 10, 12)] * 3))
    kernels = [O.get_gaussian_kernel(0.5)] * 3
    res = fd.filter_volumes(vols, kernels, l=2, w=5)
    assert len(res) == 3 and batch_engine.batches == [(3, 6, 10, 12)]
    for v, r in zip(vols, res):
        assert np.array_equal(r, _oracle(v, kernels, True))


def test_filter_volumes_splits_a_group_that_does_not_fit_the_device(batch_engine, monkeypatch):
    """A quarter of the free memory goes to the batch buffers (16 bytes per voxel): 2 volumes of 6x10x12 per part."""
    from oracle import fd_oracle as O
    monkeypatch.setattr(_FakeCuda, "free", 4 * 16 * 6 * 10 * 12 * 2 + 100)
    vols = _vols([(6, 10, 12)] * 5)
    kernels = [O.get_gaussian_kernel(0.5)] * 3
    res = fd.filter_volumes(vols, kernels, no_OF=True)
    assert batch_engine.batches == [(2, 6, 10, 12), (2, 6, 10, 12), (1, 6, 10, 12)]
    for v, r in zip(vols, res):
        assert np.array_equal(r, _oracle(v, kernels, False))
    monkeypatch.setattr(_FakeCuda, "free", 10)      # less than one volume: still one at a time
    batch_engine.batches.clear()
    fd.filter_volumes(vols[:2], kernels, no_OF=True)
    assert batch_engine.batches == [(1, 6, 10, 12), (1, 6, 10, 12)]


def test_filter_volumes_rejects_volumes_that_are_not_3d(batch_engine):
    with pytest.raises(ValueError):
        fd.filter_volumes([np.zeros((4, 4))], [np.ones(1)] * 3)
    assert fd.filter_volumes([], [np.ones(1)] * 3) == []


# ---- C ABI: the batch entry points reject bad arguments before any launch ----
def test_batch_entry_points_reject_bad_arguments():
    lib = _lib.load()
    whole = _lib.View(16, 16, 0, 1, 8, 8, 64, 8, 64, 8)
    of = _lib.OfParams(3, 5, 3, 5, 1.2, 1, 0)
    k = (C.c_double * 257)(*([1.0 / 257] * 257))
    assert lib.fdn_workspace_bytes_batch(C.byref(whole), 4, 17, C.byref(of)) > \
        lib.fdn_workspace_bytes_batch(C.byref(whole), 1, 17, C.byref(of)) > 0
    # batch == 1 sizes exactly what the single-volume pass of the whole axis needs
    assert lib.fdn_workspace_bytes_batch(C.byref(whole), 1, 17, C.byref(of)) == \
        lib.fdn_workspace_bytes(C.byref(whole), 17, C.byref(of), 0)
    bad_views = [_lib.View(16, 16, 0, 0, 8, 8, 64, 8, 64, 8),     # not periodic
                 _lib.View(16, 15, 1, 1, 8, 8, 64, 8, 64, 8),     # a window
                 _lib.View(16, 15, 0, 1, 8, 8, 64, 8, 64, 8)]     # n_out < n_in
    bad_of = _lib.OfParams(3, 99, 3, 5, 1.2, 1, 0)
    cases = [(whole, 0, 17, of), (whole, -3, 17, of), (whole, 2, 259, of), (whole, 2, 16, of), (whole, 2, 17, bad_of)]
    cases += [(v, 2, 17, of) for v in bad_views]
    cases += [(whole, (1 << 30), 17, of)]                         # 2^35 image pairs in one launch
    dummy = C.c_void_p(256)   # never dereferenced: every call fails its checks first
    n0 = lib.fdn_launch_count()
    for v, b, klen, p in cases:
        assert lib.fdn_workspace_bytes_batch(C.byref(v), b, klen, C.byref(p)) == 0
        assert lib.fdn_filter_axis_batch(dummy, dummy, C.byref(v), b, 1024, 1024, k, klen, C.byref(p), dummy, 1 << 40,
                                         None) == FDN_ERR_INVALID
        if p is of and b < (1 << 30):
            assert lib.fdn_gauss_axis_batch(dummy, dummy, C.byref(v), b, 1024, 1024, k, klen, 1, None) == \
                FDN_ERR_INVALID
            assert lib.fdn_filter_axis_batch(dummy, dummy, C.byref(v), b, 1024, 1024, k, klen, None, None, 0,
                                             None) == FDN_ERR_INVALID
    assert lib.fdn_launch_count() == n0


# ---- CLI ----
def _cli(argv):
    with pytest.raises(SystemExit) as e:
        fd.main(argv)
    return e.value.code


@pytest.mark.parametrize("extra", [
    [],                                              # --inputs without --output_dir
    ["--output_dir", "OUT", "-i", "x.mrc"],
    ["--output_dir", "OUT", "--input", "x.mrc"],
    ["--output_dir", "OUT", "-o", "y.mrc"],
    ["--output_dir", "OUT", "--output=y.mrc"],
    ["--output_dir", "OUT", "-m"],
    ["--output_dir", "OUT", "--gpus", "2"],
    ["--output_dir", "OUT", "--border", "mean"],
    ["--output_dir", "OUT", "--slab_slices", "8"],
    ["--output_dir", "OUT", "--keep_dtype"],
    ["--output_dir", "OUT", "--compat_zy_output"],
])
def test_cli_rejects_unsupported_combinations(tmp_path, monkeypatch, extra):
    called = []
    monkeypatch.setattr(fd, "filter_volumes", lambda *a, **k: called.append(1))
    argv = ["--inputs", str(tmp_path / "a.mrc"), str(tmp_path / "b.mrc")] + \
        [str(tmp_path / x) if x == "OUT" else x for x in extra]
    assert _cli(argv) == 2 and not called


def test_cli_rejects_output_dir_alone_and_repeated_basenames(tmp_path, monkeypatch):
    monkeypatch.setattr(fd, "filter_volumes", lambda *a, **k: pytest.fail("must not run"))
    assert _cli(["--output_dir", str(tmp_path)]) == 2
    os.makedirs(tmp_path / "d1"); os.makedirs(tmp_path / "d2")
    assert _cli(["--inputs", str(tmp_path / "d1" / "t.mrc"), str(tmp_path / "d2" / "t.mrc"),
                 "--output_dir", str(tmp_path / "out")]) == 2


def test_cli_writes_each_result_under_its_basename(tmp_path, monkeypatch):
    """Inputs of several shapes and formats: DIR is created, DIR/<basename> holds the float32 result of that input,
    and the flags reach filter_volumes with their -i / -o meaning."""
    rng = np.random.default_rng(3)
    src = tmp_path / "src"
    os.makedirs(src)
    vols = {"a.mrc": rng.random((4, 6, 8)).astype(np.float32), "b.mrc": (rng.random((3, 5, 7)) * 60000).astype(np.uint16),
            "c.tif": rng.random((4, 6, 8)).astype(np.float32)}
    for name, v in vols.items():
        volume_io.write_volume(str(src / name), v) if name.endswith(".tif") else _write_mrc_any(src / name, v)
    assert volume_io.read_volume(str(src / "b.mrc")).dtype == np.uint16     # an integer file: the CLI casts it
    seen = {}

    def fake(vs, kernels, l, w, get_flow, **kw):
        seen.update(kw, l=l, w=w, get_flow=get_flow, n=len(vs), k=[len(k) for k in kernels],
                    dtypes={v.dtype for v in vs})
        return [np.asarray(v, np.float32) * 2 + i for i, v in enumerate(vs)]
    monkeypatch.setattr(fd, "filter_volumes", fake)
    out = tmp_path / "new" / "dir"
    assert fd.main(["--inputs"] + [str(src / n) for n in vols] + ["--output_dir", str(out), "-s", "1", "-l", "2",
                    "-w", "7", "--recompute_flow", "--iterations", "4", "--gaussian_window", "-n"]) == 0
    assert seen["n"] == 3 and seen["l"] == 2 and seen["w"] == 7 and seen["k"] == [9, 9, 9]
    assert seen["get_flow"] is fd.get_flow_without_prev_flow and seen["no_OF"] and seen["iterations"] == 4
    assert seen["gaussian_window"] and seen["dtypes"] == {np.dtype(np.float32)}
    assert sorted(os.listdir(out)) == sorted(vols)
    for i, (name, v) in enumerate(vols.items()):
        got = volume_io.read_volume(str(out / name))
        assert got.dtype == np.float32 and np.array_equal(got, v.astype(np.float32) * 2 + i)


def _write_mrc_any(path, v):
    """An MRC file in the volume's own mode: float32 as mode 2, uint16 as mode 6 (an integer file)."""
    v = np.ascontiguousarray(v)
    if v.dtype == np.float32:
        volume_io.write_mrc(str(path), v)
        return
    assert v.dtype == np.uint16
    h = bytearray(volume_io._mrc_header(*v.shape, *volume_io._stats(v)))
    struct.pack_into("<i", h, 12, 6)            # mode 6: uint16
    with open(path, "wb") as f:
        f.write(h)
        v.astype("<u2").tofile(f)
