"""CPU tests of the reflect / mirror / nearest borders that need no device: the host index maps and the streaming halo
gather against np.pad, the routing of GaussianDenoising (in core or streamed, typed or not), the neighbour lists of
the reference's per-slice entry points, the CLI and the C ABI's rejection of an unknown border before any launch."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from flowdenoising_b200 import _lib  # noqa: E402
from flowdenoising_b200 import engine  # noqa: E402
from flowdenoising_b200 import flowdenoising as fd  # noqa: E402
from flowdenoising_b200.streaming import StreamingDenoiser, _runs  # noqa: E402

FDN_ERR_INVALID = 1   # include/fdn_b200.h
NP_MODE = {"reflect": "symmetric", "mirror": "reflect", "nearest": "edge", "wrap": "wrap"}   # SciPy name -> np.pad


@pytest.mark.parametrize("border", ["reflect", "mirror", "nearest", "wrap"])
def test_index_map_equals_np_pad(border):
    """The formulas of include/fdn_b200.h equal np.pad(arange(n), w, mode) for every n in 1..7 and w in 0..24."""
    for n in range(1, 8):
        for w in range(25):
            got = engine.border_indices(np.arange(-w, n + w), n, border)
            assert np.array_equal(got, np.pad(np.arange(n), w, mode=NP_MODE[border])), (n, w)


def _gather(sd, src, axis, lo, hi):
    shape = list(src.shape)
    shape[axis] = hi - lo
    dst = np.full(shape, -1.0, np.float32)
    sd._gather(src, axis, lo, hi, dst, None)
    return dst


@pytest.mark.parametrize("border", ["reflect", "mirror", "nearest", "wrap"])
@pytest.mark.parametrize("n", [1, 2, 5, 11])
def test_streaming_halo_gather_equals_np_pad(border, n):
    """Every slab of every axis with an r = 8 halo (n < r included) is the slab of the np.pad-ed volume."""
    r = 8
    sd = StreamingDenoiser.__new__(StreamingDenoiser)
    sd.border = border
    rng = np.random.default_rng(n)
    for axis in range(3):
        shape = [3, 4, 5]
        shape[axis] = n
        vol = rng.random(shape).astype(np.float32)
        pad = [(0, 0)] * 3
        pad[axis] = (r, r)
        padded = np.pad(vol, pad, mode=NP_MODE[border])
        for a in range(n):
            for b in range(a + 1, n + 1):
                sl = [slice(None)] * 3
                sl[axis] = slice(a, b + 2 * r)
                assert np.array_equal(_gather(sd, vol, axis, a - r, b + r), padded[tuple(sl)]), (axis, a, b)


def test_halo_runs_are_reversed_and_repeated():
    assert _runs(-3, 4, 4, "reflect") == [(0, 2, 3, -1, False), (3, 0, 4, 1, True)]
    assert _runs(-3, 4, 4, "mirror") == [(0, 3, 4, -1, False), (4, 1, 3, 1, True)]
    assert _runs(-3, 5, 4, "nearest") == [(0, 0, 4, 0, False), (4, 1, 3, 1, True), (7, 3, 1, 1, False)]
    assert _runs(-2, 6, 4, "wrap") == [(0, 2, 2, 1, False), (2, 0, 4, 1, True), (6, 0, 2, 1, False)]


# ---- routing ----
def _denoiser(border, dtype=np.float32, keep=False, of=True, vol=None):
    vol = np.zeros((6, 5, 4), dtype) if vol is None else vol
    d = fd.FlowDenoising(1, vol, keep_dtype=keep) if of else fd.GaussianDenoising(1, vol, keep_dtype=keep)
    d.border = border
    return d


@pytest.mark.parametrize("border", ["reflect", "mirror", "nearest"])
def test_new_borders_run_in_core_and_mean_streams(border, monkeypatch):
    class _Eng:
        class torch:
            class cuda:
                @staticmethod
                def mem_get_info(_dev):
                    return 1 << 40, 1 << 40
        device = None
    monkeypatch.setattr(fd, "_get_engine", lambda: _Eng())
    assert not _denoiser(border)._streaming_needed()
    assert _denoiser("mean")._streaming_needed()
    assert not _denoiser("wrap")._streaming_needed()
    d = _denoiser(border)
    d.devices = [0, 1]
    assert d._streaming_needed()          # several devices stream whatever the border


@pytest.mark.parametrize("border", ["reflect", "mirror", "nearest"])
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.int16])
def test_typed_accepts_the_new_borders_and_rejects_mean(border, dtype):
    assert _denoiser(border, dtype, keep=True)._typed()
    with pytest.raises(ValueError):
        _denoiser("mean", dtype, keep=True)._typed()
    assert _denoiser(border, np.int8, keep=True, of=False)._typed()


def test_streaming_denoiser_border_names(monkeypatch):
    monkeypatch.setattr(_lib, "require_cuda", lambda: (_ for _ in ()).throw(AssertionError("checked first")))
    with pytest.raises(ValueError):
        StreamingDenoiser(None, border="constant")
    sd = StreamingDenoiser.__new__(StreamingDenoiser)
    sd.keep_dtype = True
    for b in ("reflect", "mirror", "nearest", "wrap"):
        sd.border = b
        assert sd.pass_dtype(np.zeros(1, np.uint16)) == np.uint16
    sd.border = "mean"
    with pytest.raises(ValueError):
        sd.pass_dtype(np.zeros(1, np.uint16))


def test_engine_border_names():
    assert [engine.border_code(b) for b in ("wrap", "reflect", "mirror", "nearest")] == [1, 2, 3, 4]
    for bad in ("mean", "constant", "", None):
        with pytest.raises(ValueError):
            engine.border_code(bad)


def test_filter_volumes_rejects_mean_and_unknown_borders(monkeypatch):
    monkeypatch.setattr(fd, "_get_engine", lambda: pytest.fail("must not reach the device"))
    for bad in ("mean", "constant"):
        with pytest.raises(ValueError):
            fd.filter_volumes([np.zeros((3, 4, 5), np.float32)], [np.ones(1)] * 3, border=bad)


# ---- the reference's per-slice / per-chunk entry points ----
class _ViewRecorder:
    """Stand-in engine: records the slab and the view filter_view receives and writes the centre slices."""

    def __init__(self):
        self.torch = torch
        self.device = torch.device("cpu")
        self.calls = []

    def filter_view(self, d_in, d_out, v, kernel, flow, exact=True):
        self.calls.append((d_in.clone(), (v.n_in, v.n_out, v.halo, v.periodic)))
        d_out.copy_(d_in[v.halo:v.halo + v.n_out])


@pytest.mark.parametrize("border", ["reflect", "mirror", "nearest", "wrap", "mean"])
def test_slice_and_chunk_take_the_border_neighbours(border, monkeypatch):
    eng = _ViewRecorder()
    monkeypatch.setattr(fd, "_get_engine", lambda: eng)
    n, r = 5, 3
    vol = np.arange(n * 2 * 3, dtype=np.float32).reshape(n, 2, 3)
    d = _denoiser(border, of=False, vol=vol)
    mode = NP_MODE["wrap" if border == "mean" else border]      # mean keeps the reference's `% n` here
    padded = np.pad(vol, [(r, r), (0, 0), (0, 0)], mode=mode)
    k = np.ones(2 * r + 1) / (2 * r + 1)
    for z in range(n):
        d._slice(0, z, k)
        slab, view = eng.calls[-1]
        assert view == (2 * r + 1, 1, r, 0)
        assert np.array_equal(slab.numpy(), padded[z:z + 2 * r + 1])
    d._chunk(0, 1, 3, k)
    slab, view = eng.calls[-1]
    assert view == (3 + 2 * r, 3, r, 0) and np.array_equal(slab.numpy(), padded[1:1 + 3 + 2 * r])
    assert np.array_equal(d.filtered_vol, vol)
    # along X the slab is the moved axis
    padx = np.pad(vol, [(0, 0), (0, 0), (r, r)], mode=mode)
    d._chunk(2, 0, 3, k)
    slab, _ = eng.calls[-1]
    assert np.array_equal(slab.numpy(), np.moveaxis(padx[:, :, 0:3 + 2 * r], 2, 0))


# ---- CLI ----
def _cli(argv):
    with pytest.raises(SystemExit) as e:
        fd.main(argv)
    return e.value.code


def test_cli_border_choices_and_help(capsys):
    for b in ("wrap", "reflect", "mirror", "nearest", "mean"):
        assert fd.build_parser().parse_args(["--border", b]).border == b
    assert fd.build_parser().parse_args([]).border == "wrap"
    with pytest.raises(SystemExit):
        fd.build_parser().parse_args(["--border", "constant"])
    help_text = " ".join(fd.build_parser().format_help().split())
    for word in ("reflect", "mirror", "nearest", "the reference", "BORDER_REFLECT_101"):
        assert word in help_text


@pytest.mark.parametrize("border", ["reflect", "mirror", "nearest", "wrap"])
def test_cli_inputs_pass_the_border(tmp_path, monkeypatch, border):
    from flowdenoising_b200 import volume_io
    seen = {}

    def fake(vs, kernels, l, w, get_flow, **kw):
        seen.update(kw)
        return [np.asarray(v, np.float32) for v in vs]
    monkeypatch.setattr(fd, "filter_volumes", fake)
    volume_io.write_mrc(str(tmp_path / "a.mrc"), np.zeros((3, 4, 5), np.float32))
    assert fd.main(["--inputs", str(tmp_path / "a.mrc"), "--output_dir", str(tmp_path / "o"), "--border", border]) == 0
    assert seen["border"] == border


def test_cli_inputs_still_reject_mean(tmp_path, monkeypatch):
    monkeypatch.setattr(fd, "filter_volumes", lambda *a, **k: pytest.fail("must not run"))
    assert _cli(["--inputs", str(tmp_path / "a.mrc"), "--output_dir", str(tmp_path), "--border", "mean"]) == 2


# ---- C ABI ----
def test_abi_rejects_unknown_borders_before_any_launch():
    lib = _lib.load()
    k = (C.c_double * 5)(*([0.2] * 5))
    dummy = C.c_void_p(256)   # never dereferenced: every call fails its checks first
    n0 = lib.fdn_launch_count()
    for border in (0, 5, -1, 7, 1 << 20):
        for dt in (_lib.DTYPE_F32, _lib.DTYPE_U8, _lib.DTYPE_I16):
            assert lib.fdn_gauss_rows_border(dummy, dummy, dt, 4, 8, k, 5, 1, border, None) == FDN_ERR_INVALID
    # the extent the border arithmetic takes: a reflected axis of more than 2^30 slices is refused, a wrapped one not
    big = _lib.View((1 << 30) + 1, 1, 0, _lib.BORDER_REFLECT, 1, 1, 1, 1, 1, 1)
    assert lib.fdn_gauss_axis(dummy, dummy, C.byref(big), k, 5, 1, None) == FDN_ERR_INVALID
    of = _lib.OfParams(3, 5, 3, 5, 1.2, 1, 0)
    assert lib.fdn_workspace_bytes(C.byref(big), 5, C.byref(of), 1) == 0
    assert lib.fdn_gauss_rows_border(dummy, dummy, 0, 1, (1 << 30) + 1, k, 5, 1, _lib.BORDER_MIRROR, None) == \
        FDN_ERR_INVALID
    assert lib.fdn_launch_count() == n0


@pytest.mark.parametrize("border", [2, 3, 4])
def test_abi_sizes_bordered_views_like_wrapped_ones(border):
    """A bordered view (whole axis, window, batch member) takes the workspace of the wrapped one: same R cache."""
    lib = _lib.load()
    of = _lib.OfParams(3, 5, 3, 5, 1.2, 1, 0)
    for n_in, n_out, halo in ((16, 16, 0), (40, 7, 5), (3, 3, 0), (1, 1, 0)):
        for chunk in (0, 2):
            w = _lib.View(n_in, n_out, halo, 1, 8, 8, 64, 8, 64, 8)
            b = _lib.View(n_in, n_out, halo, border, 8, 8, 64, 8, 64, 8)
            assert lib.fdn_workspace_bytes(C.byref(b), 17, C.byref(of), chunk) == \
                lib.fdn_workspace_bytes(C.byref(w), 17, C.byref(of), chunk) > 0
            assert lib.fdn_workspace_bytes_typed(C.byref(b), 17, C.byref(of), chunk, _lib.DTYPE_U16) == \
                lib.fdn_workspace_bytes_typed(C.byref(w), 17, C.byref(of), chunk, _lib.DTYPE_U16) > 0
    w = _lib.View(16, 16, 0, 1, 8, 8, 64, 8, 64, 8)
    b = _lib.View(16, 16, 0, border, 8, 8, 64, 8, 64, 8)
    assert lib.fdn_workspace_bytes_batch(C.byref(b), 5, 17, C.byref(of)) == \
        lib.fdn_workspace_bytes_batch(C.byref(w), 5, 17, C.byref(of)) > 0
