"""B200 checks of typed (integer) volumes on several devices and out of core (keep_dtype with DistributedDenoiser,
StreamingDenoiser, memory maps and --gpus): the typed re-slab kernels (fdn_copy3d_typed, fdn_transpose_strided_typed)
against NumPy with guard bands, the sharded and the streamed passes against the cv2 digests of
tests/golden/integer_volumes.npz, the module surface and the CLI, and the float32 route's launch sequence left as it
was."""
import hashlib
import json
import os
import socket
import struct

import numpy as np
import pytest

from oracle import fd_oracle as O
from oracle import gen_golden_integer as G

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
import torch.distributed as dist  # noqa: E402
import torch.multiprocessing as mp  # noqa: E402

TOY_CASES = [f"{dt}_{m}" for dt in ("uint8", "uint16", "int16") for m in ("of", "ofr", "noof")] + ["int8_noof"]
DTYPES = [np.uint8, np.int8, np.uint16, np.int16, np.float32]
GUARD = 4096


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def case_flow(name):
    from flowdenoising_b200.engine import FlowParams
    _dt, _shape, _seed, _noise, sigmas, mode, w = G.CASES[name]
    ks = [O.get_gaussian_kernel(s) for s in sigmas]
    return (None if mode == "noof" else FlowParams(3, w, 3, 5, 1.2, mode != "ofr")), ks


@pytest.fixture(scope="module")
def eng():
    from flowdenoising_b200.engine import DeviceEngine
    return DeviceEngine()


def _values(n, dtype, seed):
    rng = np.random.default_rng(seed)
    if np.dtype(dtype).kind == "f":
        return rng.standard_normal(n).astype(dtype)
    info = np.iinfo(dtype)
    return rng.integers(info.min, int(info.max) + 1, n).astype(dtype)


def _guarded(n, dtype, seed):
    """A flat device buffer of n elements plus GUARD elements of noise on both sides, and its host copy."""
    h = _values(n + 2 * GUARD, dtype, seed)
    return torch.from_numpy(h.copy()).cuda(), h


# (A, B, C, b0, bw, c0, cw, in pad, out pad, src_off, dst_off): odd sizes, negative / wrapping b0 and c0, element
# offsets that are not 4-byte aligned, runs that cross the wrap (cw smaller than a run included), long rows
COPY_CASES = [
    (3, 5, 37, -3, 7, -5, 41, 3, 1, 1, 3),
    (2, 4, 11, 9, 4, 2, 3, 0, 0, 0, 1),
    (1, 3, 13, 0, 3, 11, 12, 1, 2, 3, 2),
    (2, 2, 1025, -1, 2, 517, 1030, 0, 0, 0, 0),
    (4, 3, 1000, 2, 3, -999, 1000, 2, 5, 5, 6),
    (2, 1, 2, 0, 1, 1, 1, 0, 0, 1, 1),
    (65, 2, 5, -70, 9, 3, 5, 0, 3, 2, 7),
]


@pytest.mark.parametrize("dtype", DTYPES, ids=lambda d: np.dtype(d).name)
def test_copy3d_typed_vs_numpy(eng, dtype):
    for i, (A, B, C, b0, bw, c0, cw, ipad, opad, soff, doff) in enumerate(COPY_CASES):
        in_sb = cw + ipad
        in_sa = bw * in_sb + ipad
        out_sb = C + opad
        out_sa = B * out_sb + opad
        src_h = _values(soff + A * in_sa, dtype, seed=i)
        src = torch.from_numpy(src_h.copy()).cuda()
        dst, want = _guarded(A * out_sa, dtype, seed=100 + i)
        eng.copy3d(src, soff, in_sa, in_sb, b0, bw, c0, cw, dst, GUARD + doff, out_sa, out_sb, A, B, C)
        a = np.arange(A)[:, None, None]
        b = np.arange(B)[None, :, None]
        c = np.arange(C)[None, None, :]
        want[GUARD + doff + a * out_sa + b * out_sb + c] = src_h[soff + a * in_sa + ((b0 + b) % bw) * in_sb + (c0 + c) % cw]
        torch.cuda.synchronize()
        assert np.array_equal(dst.cpu().numpy().view(np.uint8), want.view(np.uint8)), (np.dtype(dtype).name, i)


@pytest.mark.parametrize("dtype", DTYPES, ids=lambda d: np.dtype(d).name)
def test_transpose_strided_typed_vs_numpy(eng, dtype):
    for i, (n, A, B, ipad, opad, soff, doff) in enumerate([(3, 37, 45, 3, 1, 1, 3), (2, 1, 33, 0, 0, 0, 1),
                                                           (5, 64, 31, 2, 7, 3, 2), (1, 70, 70, 0, 0, 0, 0)]):
        in_sa = B + ipad
        in_sn = A * in_sa + ipad
        out_sb = A + opad
        out_sn = B * out_sb + opad
        src_h = _values(soff + n * in_sn, dtype, seed=i)
        src = torch.from_numpy(src_h.copy()).cuda()
        dst, want = _guarded(n * out_sn, dtype, seed=200 + i)
        eng.transpose_strided(src, soff, in_sn, in_sa, dst, GUARD + doff, out_sn, out_sb, n, A, B)
        j = np.arange(n)[:, None, None]
        a = np.arange(A)[None, :, None]
        b = np.arange(B)[None, None, :]
        want[GUARD + doff + j * out_sn + b * out_sb + a] = src_h[soff + j * in_sn + a * in_sa + b]
        torch.cuda.synchronize()
        assert np.array_equal(dst.cpu().numpy().view(np.uint8), want.view(np.uint8)), (np.dtype(dtype).name, i)


def test_copy3d_profile_bytes(eng):
    """The profiler's model counts 2 sizeof(T) bytes per element (8 for float32, as before)."""
    import ctypes as C
    from flowdenoising_b200 import _lib
    lib = _lib.load()
    kid = [lib.fdn_profile_kernel_name(i).decode() for i in range(lib.fdn_profile_kernel_count())].index("k_copy3d")
    for dtype, per in ((torch.uint8, 2), (torch.int16, 4), (torch.float32, 8)):
        src = torch.zeros(4 * 5 * 6, dtype=dtype, device="cuda")
        dst = torch.empty_like(src)
        lib.fdn_profile_reset()
        lib.fdn_profile_enable(1)
        eng.copy3d(src, 0, 30, 6, 0, 5, 0, 6, dst, 0, 30, 6, 4, 5, 6)
        lib.fdn_profile_enable(0)
        ms, n, by = C.c_double(), C.c_int64(), C.c_double()
        _lib.check(lib.fdn_profile_read(kid, C.byref(ms), C.byref(n), C.byref(by)))
        lib.fdn_profile_reset()
        assert n.value == 1 and by.value == per * 120


# ---- DistributedDenoiser over NCCL ----
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _dist_worker(rank, world, port, names, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from flowdenoising_b200.dist import DistributedDenoiser
        from flowdenoising_b200.engine import DeviceEngine
        eng = DeviceEngine(torch.device("cuda", rank))
        for name in names:
            vol = G.case_volume(name)
            flow, ks = case_flow(name)
            dd = DistributedDenoiser(eng, vol.shape, flow)
            zs, ze = dd.z_range
            zy, zyx = dd.filter(torch.from_numpy(vol[zs:ze].copy()).cuda(), ks, want_zy=True)
            torch.cuda.synchronize()
            np.save(os.path.join(out_dir, f"{name}_zy_{rank}.npy"), zy.cpu().numpy())
            np.save(os.path.join(out_dir, f"{name}_zyx_{rank}.npy"), zyx.cpu().numpy())
            host = torch.from_numpy(vol[zs:ze].copy()).pin_memory()
            out_host = torch.from_numpy(np.full(host.shape, 77, vol.dtype)).pin_memory()
            for _ in range(2):      # the second call re-uses cached buffers while copies of the first may be queued
                res = dd.filter_host(host, out_host, ks)
            torch.cuda.synchronize()
            assert np.array_equal(res.cpu().numpy(), out_host.numpy())
            np.save(os.path.join(out_dir, f"{name}_zyxh_{rank}.npy"), out_host.numpy())
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [1, 2])
def test_distributed_typed_equals_golden(tmp_path, golden, world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    g = golden("integer_volumes.npz")
    names = TOY_CASES + ["cfg1_uint8"]
    mp.spawn(_dist_worker, args=(world, _free_port(), names, str(tmp_path)), nprocs=world, join=True)
    for name in names:
        for tag, key in (("zy", "ZY"), ("zyx", "ZYX"), ("zyxh", "ZYX")):
            got = np.concatenate([np.load(tmp_path / f"{name}_{tag}_{r}.npy") for r in range(world)])
            assert got.dtype == np.dtype(G.CASES[name][0])
            assert sha(got) == str(g[f"{name}_sha_{key}"]), (name, tag, world)


# ---- StreamingDenoiser, typed ----
def _readonly_map(tmp_path, vol):
    path = tmp_path / "vol.raw"
    vol.tofile(path)
    return np.memmap(path, dtype=vol.dtype, mode="r", shape=vol.shape)


@pytest.mark.parametrize("name", TOY_CASES + ["cfg1_uint8"])
def test_streaming_typed_equals_golden(tmp_path, golden, name):
    """Slabs of 3 (8 = 3 + 3 + 2: a ragged last slab) and 5 slices, two lanes on one device, a read-only memory map,
    and slabs sized from a small device budget."""
    from flowdenoising_b200.streaming import StreamingDenoiser
    g = golden("integer_volumes.npz")
    vol = G.case_volume(name)
    flow, ks = case_flow(name)
    runs = [dict(slab_slices=3), dict(slab_slices=5), dict(slab_slices=3, devices=[0, 0])]
    if name == "cfg1_uint8":
        runs = [dict(slab_slices=5), dict(slab_slices=7, devices=[0, 0])]
    for kw in runs:
        sd = StreamingDenoiser(flow, keep_dtype=True, **kw)
        v = vol.copy()
        zy, zyx = sd.filter(v, ks)
        sd.release()
        assert zy is v and zyx.dtype == vol.dtype, kw                       # vol ends as the Z+Y intermediate
        assert sha(zy) == str(g[f"{name}_sha_ZY"]) and sha(zyx) == str(g[f"{name}_sha_ZYX"]), kw
    mm = _readonly_map(tmp_path, vol)
    sd = StreamingDenoiser(flow, keep_dtype=True, slab_slices=5)
    res = np.full(vol.shape, np.nan, np.float32)                            # a float32 result array holds T exactly
    zy, zyx = sd.filter(mm, ks, filtered_vol=res)
    assert zyx is res and zy.dtype == vol.dtype and np.array_equal(np.asarray(mm), vol)
    assert sha(zy) == str(g[f"{name}_sha_ZY"]) and sha(res.astype(vol.dtype)) == str(g[f"{name}_sha_ZYX"])
    budgets = {"uint16_of": (2_621_440, [0]), "int8_noof": (120_000, [0, 1, 2])}   # bytes, axes cut into slabs
    if name in budgets:
        budget, axes = budgets[name]
        sd = StreamingDenoiser(flow, keep_dtype=True, device_budget_bytes=budget)
        for axis in axes:
            assert sd._slab_len(vol.shape, axis, ks[axis].size // 2, vol.dtype) < vol.shape[axis], axis
        zy, zyx = sd.filter(vol.copy(), ks)
        assert sha(zyx) == str(g[f"{name}_sha_ZYX"])


# ---- module surface and CLI ----
def module_denoiser(name, vol):
    from flowdenoising_b200 import flowdenoising as F
    _dt, _shape, _seed, _noise, _s, mode, w = G.CASES[name]
    if mode == "noof":
        return F.GaussianDenoising(1, vol, keep_dtype=True)
    get_flow = F.get_flow_without_prev_flow if mode == "ofr" else F.get_flow_with_prev_flow
    return F.FlowDenoising(1, vol, 3, w, get_flow, keep_dtype=True)


@pytest.mark.parametrize("name", ["uint8_of", "uint16_ofr", "int16_of", "int8_noof", "uint16_noof"])
def test_module_surface_typed_streaming(tmp_path, golden, name):
    g = golden("integer_volumes.npz")
    vol = G.case_volume(name)
    _flow, ks = case_flow(name)
    for how in ("streaming", "devices", "memmap"):
        src = _readonly_map(tmp_path, vol) if how == "memmap" else vol.copy()
        d = module_denoiser(name, src)
        d.slab_slices = 3
        if how == "streaming":
            d.streaming = True
        elif how == "devices":
            d.devices = [0, 0]
        assert d._typed() and d._streaming_needed()
        res = d.filter(ks)
        assert res is d.filtered_vol and res.dtype == vol.dtype, how
        assert sha(res) == str(g[f"{name}_sha_ZYX"]), how
        if how == "memmap":
            assert np.array_equal(np.asarray(src), vol)
        else:
            assert sha(d.vol) == str(g[f"{name}_sha_ZY"]), how
        assert d.progress == sum(vol.shape)
    d = module_denoiser(name, vol.copy())            # the per-pass entry points take the same route
    d.streaming = True
    d.slab_slices = 5
    for axis, (tag, f) in enumerate((("Z", d.filter_along_Z), ("ZY", d.filter_along_Y), ("ZYX", d.filter_along_X))):
        f(ks[axis])
        assert sha(d.filtered_vol) == str(g[f"{name}_sha_{tag}"]), tag
        d.vol[...] = d.filtered_vol


def test_typed_streaming_rejects_fast_no_of():
    from flowdenoising_b200 import flowdenoising as F
    d = F.GaussianDenoising(1, G.case_volume("uint16_noof"), keep_dtype=True)
    d.streaming = True
    d.exact = False
    with pytest.raises(ValueError, match="exact"):
        d.filter([O.get_gaussian_kernel(1.0)] * 3)


def _write_mrc(path, vol, mode):
    from flowdenoising_b200 import volume_io
    nz, ny, nx = vol.shape
    h = volume_io._mrc_header(nz, ny, nx, float(vol.min()), float(vol.max()), float(vol.mean()), 0.0)
    struct.pack_into("<i", h, 12, mode)
    with open(path, "wb") as f:
        f.write(h)
        vol.astype(vol.dtype.newbyteorder("<")).tofile(f)


@pytest.mark.parametrize("gpus", [1, 2])
@pytest.mark.parametrize("name,mode", [("int16_of", 1), ("uint16_ofr", 6)])
def test_cli_memory_map_keep_dtype(golden, tmp_path, name, mode, gpus):
    from flowdenoising_b200 import flowdenoising as F
    from flowdenoising_b200 import volume_io
    if torch.cuda.device_count() < gpus:
        pytest.skip(f"needs {gpus} GPUs")
    g = golden("integer_volumes.npz")
    vol = G.case_volume(name)
    src, dst = str(tmp_path / "in.mrc"), str(tmp_path / "out.mrc")
    _write_mrc(src, vol, mode)
    argv = ["-i", src, "-o", dst, "-s", *[str(s) for s in G.CASES[name][4]], "-m", "--keep_dtype",
            "--slab_slices", "5"]
    if gpus > 1:
        argv += ["--gpus", str(gpus)]
    if G.CASES[name][5] == "ofr":
        argv.append("--recompute_flow")
    assert F.main(argv) == 0
    out = volume_io.read_volume(dst)
    assert out.dtype == np.float32
    assert sha(out.astype(vol.dtype)) == str(g[f"{name}_sha_ZYX"])
    assert np.array_equal(volume_io.read_volume(src), vol)


# ---- the float32 route keeps its launch sequence ----
LOG_SHAPE = (10, 40, 48)
LOG_SIGMAS = (1.0, 0.5, 0.75)

# (launches, SHA-256 of the newline-joined kernel names) of the launch logs of the runs below, captured on a B200 from
# the library and Python layer as they were before typed slabs existed: the float32 route launches the same kernels in
# the same order since
PARENT_LOGS = {
    "streaming_0": (49, "c6003bd5b608ffea34616c5a382e1dc6af064546441c19f8e2e60460abd392ae"),
    "dist_0": (21, "9d1b595e02a1724cf407634de930948fc6d8d2b4858537dd3455cc9ec7f09b41"),
    "streaming_1": (522, "f3bd2f5975638b097958e6623e5721f18785dc7b08d7860efbea9f9eea1e2acf"),
    "dist_1": (147, "144920b53c091f5193a8ad3ccc3907f8ddef790bc0c3066fab2f465561a19fc1"),
}


def _log(lib):
    return [lib.fdn_launch_log_name(i).decode() for i in range(lib.fdn_launch_log_count())]


def _check_log(names, key):
    got = (len(names), hashlib.sha256("\n".join(names).encode()).hexdigest())
    rle = []
    for n in names:
        if rle and rle[-1][0] == n:
            rle[-1][1] += 1
        else:
            rle.append([n, 1])
    assert got == PARENT_LOGS[key], (key, rle)


def _f32_dist_worker(rank, port, use_of, path):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    try:
        from flowdenoising_b200 import _lib
        from flowdenoising_b200.dist import DistributedDenoiser
        from flowdenoising_b200.engine import DeviceEngine, FlowParams
        lib = _lib.load()
        vol = O.synthetic_volume(LOG_SHAPE, seed=3, noise_sigma=6.0)
        ks = [O.get_gaussian_kernel(s) for s in LOG_SIGMAS]
        dd = DistributedDenoiser(DeviceEngine(torch.device("cuda", 0)), LOG_SHAPE, FlowParams() if use_of else None)
        lib.fdn_launch_log_enable(1)
        dd.filter(torch.from_numpy(vol).cuda(), ks, want_zy=True)
        out = torch.empty(LOG_SHAPE, dtype=torch.float32).pin_memory()
        dd.filter_host(torch.from_numpy(vol).pin_memory(), out, ks)
        torch.cuda.synchronize()
        log = _log(lib)
        lib.fdn_launch_log_enable(0)
        with open(path, "w") as f:
            json.dump(log, f)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("use_of", [False, True], ids=["noof", "of"])
def test_float32_launch_logs_unchanged(tmp_path, use_of):
    from flowdenoising_b200 import _lib
    from flowdenoising_b200.engine import FlowParams
    from flowdenoising_b200.streaming import StreamingDenoiser
    lib = _lib.load()
    vol = O.synthetic_volume(LOG_SHAPE, seed=3, noise_sigma=6.0)
    ks = [O.get_gaussian_kernel(s) for s in LOG_SIGMAS]
    sd = StreamingDenoiser(FlowParams() if use_of else None, slab_slices=4)
    lib.fdn_launch_log_enable(1)
    sd.filter(vol.copy(), ks)
    torch.cuda.synchronize()
    log = _log(lib)
    lib.fdn_launch_log_enable(0)
    _check_log(log, f"streaming_{int(use_of)}")
    path = str(tmp_path / "dist.json")
    mp.spawn(_f32_dist_worker, args=(_free_port(), use_of, path), nprocs=1, join=True)
    with open(path) as f:
        _check_log(json.load(f), f"dist_{int(use_of)}")
