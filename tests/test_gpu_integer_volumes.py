"""B200 checks of typed (integer) volumes, keep_dtype: the integer remap against the C oracle, whole passes and filter()
against the cv2 digests of tests/golden/integer_volumes.npz, every other entry (chunks, odd widths, views, the per-slice
and per-chunk entry points, the CLI) against those results, guard bands, and the float32 route left as it was."""
import ctypes as C
import hashlib
import struct

import numpy as np
import pytest

from oracle import fd_oracle as O
from oracle import fd_oracle_int as I
from oracle import gen_golden_integer as G

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

TOY_CASES = [c for c in G.CASES if not c.startswith("cfg1")]


@pytest.fixture(scope="module")
def eng():
    from flowdenoising_b200.engine import DeviceEngine
    return DeviceEngine()


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def case_flow(name):
    """FlowParams of a fixture case (None without OF) and its kernels."""
    from flowdenoising_b200.engine import FlowParams
    _dt, _shape, _seed, _noise, sigmas, mode, w = G.CASES[name]
    ks = [O.get_gaussian_kernel(s) for s in sigmas]
    if mode == "noof":
        return None, ks
    return FlowParams(3, w, 3, 5, 1.2, mode != "ofr", mode == "gw"), ks


def module_denoiser(name, vol, **kw):
    from flowdenoising_b200 import flowdenoising as F
    _dt, _shape, _seed, _noise, _s, mode, w = G.CASES[name]
    if mode == "noof":
        return F.GaussianDenoising(1, vol, keep_dtype=True, **kw)
    get_flow = F.get_flow_without_prev_flow if mode == "ofr" else F.get_flow_with_prev_flow
    return F.FlowDenoising(1, vol, 3, w, get_flow, gaussian_window=mode == "gw", keep_dtype=True, **kw)


@pytest.mark.parametrize("dtype,lo,hi", [(np.uint8, 0, 255), (np.uint16, 0, 65535), (np.int16, -32768, 32767)],
                         ids=["uint8", "uint16", "int16"])
def test_remap_typed_vs_oracle(dtype, lo, hi):
    from flowdenoising_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(5)
    for n, H, W in [(3, 32, 32), (2, 37, 53), (1, 64, 48)]:
        src = rng.integers(lo, hi + 1, (n, H, W)).astype(dtype)
        src[0, ::3] = lo
        src[0, 1::3] = hi                                                   # saturation
        flow = rng.uniform(-4, 4, (n, H, W, 2)).astype(np.float32)
        ay, ax = np.divmod(np.arange(H * W) % 1024, 32)                      # every 1/32-px fraction
        flow[-1, ..., 0] = (rng.integers(-3, 4, H * W) + ax / 32.0).reshape(H, W)
        flow[-1, ..., 1] = (rng.integers(-3, 4, H * W) + ay / 32.0).reshape(H, W)
        d_src, d_flow = dev(src), dev(flow)
        d_dst = torch.empty_like(d_src)
        _lib.check(lib.fdn_remap_typed(d_src.data_ptr(), d_flow.data_ptr(), d_dst.data_ptr(),
                                       I.DTYPE_CODES[np.dtype(dtype)], n, H, W, None))
        torch.cuda.synchronize()
        got = d_dst.cpu().numpy()
        for b in range(n):
            assert np.array_equal(got[b], I.warp_slice(src[b], flow[b])), (n, H, W, b)


@pytest.mark.parametrize("name", TOY_CASES)
def test_passes_and_filter_vs_golden(eng, golden, name):
    g = golden("integer_volumes.npz")
    vol = G.case_volume(name)
    flow, ks = case_flow(name)
    d_in = dev(vol)
    z = torch.empty_like(d_in)
    eng.filter_along_axis(d_in, z, 0, ks[0], flow)
    zy, zyx = eng.filter(d_in, ks, flow)
    for tag, t in (("Z", z), ("ZY", zy), ("ZYX", zyx)):
        assert t.dtype == d_in.dtype
        assert sha(t.cpu().numpy()) == str(g[f"{name}_sha_{tag}"]), (name, tag)
    d = module_denoiser(name, vol.copy())
    res = d.filter(ks)
    assert res.dtype == vol.dtype and d.vol.dtype == vol.dtype
    assert sha(res) == str(g[f"{name}_sha_ZYX"]) and sha(d.vol) == str(g[f"{name}_sha_ZY"])


def test_cfg1_uint8_after_each_pass(eng, golden):
    g = golden("integer_volumes.npz")
    name = "cfg1_uint8"
    vol = G.case_volume(name)
    flow, ks = case_flow(name)
    cur = dev(vol)
    for axis, tag in ((0, "Z"), (1, "ZY"), (2, "ZYX")):
        out = torch.empty_like(cur)
        eng.filter_along_axis(cur, out, axis, ks[axis], flow)
        assert sha(out.cpu().numpy()) == str(g[f"{name}_sha_{tag}"]), tag
        cur = out


@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.int16])
def test_chunks_views_and_odd_widths(eng, dtype):
    """Chunked passes, windows of a periodic view, non-periodic slabs and widths that are not multiples of 4 or 16
    give the bits of the whole-axis call, which equals the C-backend oracle. (Comparisons on the host: torch has few
    device kernels for uint16.)"""
    from flowdenoising_b200._lib import View
    from flowdenoising_b200.engine import FlowParams
    p = FlowParams()
    k = O.get_gaussian_kernel(1.0)
    r = k.size // 2
    for shape in ((9, 40, 37), (7, 33, 50)):
        vol = I.integer_volume(shape, dtype, seed=sum(shape))
        Z, Y, X = shape
        d_in = dev(vol)
        t_full = torch.empty_like(d_in)
        eng.filter_along_axis(d_in, t_full, 0, k, p)
        full = t_full.cpu().numpy()
        ref = I.IntegerDenoiser(4, vol.copy(), use_OF=True, backend="c")
        ref.filter_along_Z(k)
        assert np.array_equal(full, ref.filtered_vol), shape
        for chunk in (1, 4):
            out = torch.empty_like(d_in)
            eng.filter_view(d_in, out, View(Z, Z, 0, 1, Y, X, Y * X, X, Y * X, X), k, p, chunk=chunk)
            assert np.array_equal(out.cpu().numpy(), full), chunk
        for first, count in ((0, 3), (3, 6)):
            out = dev(np.full(shape, 7, dtype))
            eng.filter_view(d_in, out[first:], View(Z, count, first, 1, Y, X, Y * X, X, Y * X, X), k, p, chunk=2)
            o = out.cpu().numpy()
            assert np.array_equal(o[first:first + count], full[first:first + count])
            assert (o[:first] == 7).all() and (o[first + count:] == 7).all()
        idx = [z % Z for z in range(2 - r, 2 + 3 + r)]
        slab = dev(vol[idx])
        o = torch.empty((3, Y, X), dtype=d_in.dtype, device="cuda")
        eng.filter_view(slab, o, View(len(idx), 3, r, 0, Y, X, Y * X, X, Y * X, X), k, p)
        assert np.array_equal(o.cpu().numpy(), full[2:5])
        # small workspace limit: the pass picks a chunk that fits
        from flowdenoising_b200.engine import DeviceEngine
        small = DeviceEngine(workspace_limit_bytes=3 * 1024 * 1024)
        out = torch.empty_like(d_in)
        small.filter_along_axis(d_in, out, 0, k, p)
        assert np.array_equal(out.cpu().numpy(), full)


@pytest.mark.parametrize("name", ["uint8_of", "int16_noof"])
def test_slice_and_chunk_entry_points(golden, name):
    g = golden("integer_volumes.npz")
    vol = G.case_volume(name)
    _flow, ks = case_flow(name)
    d = module_denoiser(name, vol.copy())
    for z in range(vol.shape[0]):
        d.filter_along_Z_slice(z, ks[0])
    assert sha(d.filtered_vol) == str(g[f"{name}_sha_Z"])
    d2 = module_denoiser(name, vol.copy())
    for ci in range(3):
        d2.filter_along_Z_chunk(ci, 3, 0, ks[0])
    assert sha(d2.filtered_vol) == str(g[f"{name}_sha_Z"])
    d2.vol[...] = d2.filtered_vol
    d2.filter_along_Y(ks[1])
    assert sha(d2.filtered_vol) == str(g[f"{name}_sha_ZY"])


def test_guard_bands(eng):
    """Typed outputs and the workspace are written exactly where they should be."""
    from flowdenoising_b200 import _lib
    from flowdenoising_b200._lib import View
    from flowdenoising_b200.engine import FlowParams
    lib = _lib.load()
    k = O.get_gaussian_kernel(1.0)
    kk = np.ascontiguousarray(k)
    for dtype, code in ((np.uint8, _lib.DTYPE_U8), (np.int16, _lib.DTYPE_I16)):
        Z, Y, X = 6, 35, 41
        vol = I.integer_volume((Z, Y, X), dtype, seed=2)
        d_in = dev(vol)
        n = Z * Y * X
        G_ = 4096
        for flow in (FlowParams(), None):
            buf = torch.full((n + 2 * G_,), 93, dtype=d_in.dtype, device="cuda")
            v = View(Z, Z, 0, 1, Y, X, Y * X, X, Y * X, X)
            ofp = flow.c_struct() if flow else None
            need = lib.fdn_workspace_bytes_typed(C.byref(v), k.size, C.byref(ofp) if ofp else None, 0, code)
            ws = torch.full((need + G_,), 0xA5, dtype=torch.uint8, device="cuda")
            _lib.check(lib.fdn_filter_axis_typed(d_in.data_ptr(), buf[G_:].data_ptr(), code, C.byref(v),
                                                 kk.ctypes.data_as(C.POINTER(C.c_double)), k.size,
                                                 C.byref(ofp) if ofp else None, 0, ws.data_ptr(), need, None))
            torch.cuda.synchronize()
            assert bool((buf[:G_] == 93).all()) and bool((buf[G_ + n:] == 93).all())
            assert bool((ws[need:] == 0xA5).all())
            ref = torch.empty_like(d_in)
            eng.filter_along_axis(d_in, ref, 0, k, flow)
            assert torch.equal(buf[G_:G_ + n].view(Z, Y, X), ref)


def test_keep_dtype_on_float32_and_off_on_integers():
    from flowdenoising_b200 import _lib
    from flowdenoising_b200 import flowdenoising as F
    lib = _lib.load()
    ks = [O.get_gaussian_kernel(s) for s in G.TOY_SIGMAS]
    vol = G.case_volume("uint8_of")
    vf = vol.astype(np.float32)
    logs, outs = [], []
    for keep in (False, True):
        lib.fdn_launch_log_enable(1)
        outs.append(F.FlowDenoising(1, vf.copy(), keep_dtype=keep).filter(ks).copy())
        logs.append([lib.fdn_launch_log_name(i) for i in range(lib.fdn_launch_log_count())])
        lib.fdn_launch_log_enable(0)
    assert logs[0] == logs[1] and np.array_equal(outs[0], outs[1])
    # keep_dtype off on an integer volume: today's float32 route, truncated once into the integer result
    vi = vol.copy()
    res = F.FlowDenoising(1, vi).filter(ks)
    assert np.array_equal(res, outs[0].astype(np.uint8))


def test_unsupported_combinations_raise():
    from flowdenoising_b200 import flowdenoising as F
    k = [O.get_gaussian_kernel(1.0)] * 3
    with pytest.raises(ValueError, match="int8"):
        F.FlowDenoising(1, np.zeros((4, 32, 32), np.int8), keep_dtype=True).filter(k)
    with pytest.raises(ValueError, match="float16"):
        F.GaussianDenoising(1, np.zeros((4, 32, 32), np.float16), keep_dtype=True).filter(k)
    d = F.GaussianDenoising(1, np.zeros((4, 32, 32), np.uint8), keep_dtype=True)
    d.border = "mean"
    with pytest.raises(ValueError, match="streaming"):
        d.filter(k)
    d = F.GaussianDenoising(1, np.zeros((4, 32, 32), np.uint16), keep_dtype=True)
    d.exact = False
    with pytest.raises(ValueError, match="exact"):
        d.filter(k)


def _write_mrc(path, vol, mode):
    from flowdenoising_b200 import volume_io
    nz, ny, nx = vol.shape
    h = volume_io._mrc_header(nz, ny, nx, float(vol.min()), float(vol.max()), float(vol.mean()), 0.0)
    struct.pack_into("<i", h, 12, mode)
    with open(path, "wb") as f:
        f.write(h)
        vol.astype(vol.dtype.newbyteorder("<")).tofile(f)


@pytest.mark.parametrize("name,mode", [("int16_of", 1), ("uint16_ofr", 6)])
def test_cli_round_trip(golden, tmp_path, name, mode):
    from flowdenoising_b200 import flowdenoising as F
    from flowdenoising_b200 import volume_io
    g = golden("integer_volumes.npz")
    vol = G.case_volume(name)
    src, dst = str(tmp_path / "in.mrc"), str(tmp_path / "out.mrc")
    _write_mrc(src, vol, mode)
    assert volume_io.read_volume(src).dtype == vol.dtype
    argv = ["-i", src, "-o", dst, "-s", *[str(s) for s in G.CASES[name][4]], "--keep_dtype"]
    if G.CASES[name][5] == "ofr":
        argv.append("--recompute_flow")
    assert F.main(argv) == 0
    out = volume_io.read_volume(dst)
    assert out.dtype == np.float32
    assert sha(out.astype(vol.dtype)) == str(g[f"{name}_sha_ZYX"])
