"""GPU tests of the Gaussian window (FDN_OF_FARNEBACK_GAUSSIAN = cv2.OPTFLOW_FARNEBACK_GAUSSIAN), all bit-exact: the
flow-iteration kernels against the C oracle (UpdateMatrices + Gaussian blur-solve), whole Farneback against the
cv2 fixtures of tests/golden/gaussian_window.npz, whole passes and filter(), and every other path (views, chunks,
hidden transfers, streaming, slabs, CLI) against the in-core device result."""
import ctypes as C
import hashlib

import numpy as np
import pytest

from oracle import fd_oracle as O
from oracle import fd_oracle_gw as GW
from oracle import gen_golden_gaussian as G

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

GUARD = 1 << 20
PATTERN = 0xA5


@pytest.fixture(scope="module")
def eng():
    from flowdenoising_b200.engine import DeviceEngine
    return DeviceEngine()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def gparams(l=3, w=5, use_prev=True, it=3, pn=5, ps=1.2):
    from flowdenoising_b200.engine import FlowParams
    return FlowParams(l, w, it, pn, ps, use_prev, gaussian_window=True)


def R_from_oracle_layout(R):  # (n, h, w, 5) -> (n, fdn_polyexp_floats(h, w))
    n, h, w, _ = R.shape
    p = h * w
    out = np.zeros((n, 4 * p + (p + 3) // 4 * 4), np.float32)
    out[:, :4 * p] = R[..., :4].reshape(n, -1)
    out[:, 4 * p:5 * p] = R[..., 4].reshape(n, -1)
    return out


def _launch_names(lib):
    return [lib.fdn_launch_log_name(i).decode() for i in range(lib.fdn_launch_log_count())]


def _iterations(lib, dR, n, flow, h, w, win, iters, variant=1):
    lib.fdn_set_flow_iter_variant(variant)
    try:
        cur = dev(flow)
        t1, t2 = torch.empty_like(cur), torch.empty_like(cur)
        res = C.c_void_p()
        rc = lib.fdn_flow_iterations_gaussian(dR[:n].data_ptr(), dR[n:].data_ptr(), cur.data_ptr(), t1.data_ptr(),
                                              t2.data_ptr(), n, h, w, win, iters, None, C.byref(res))
        assert rc == 0, lib.fdn_last_error()
        return {cur.data_ptr(): cur, t1.data_ptr(): t1, t2.data_ptr(): t2}[res.value].cpu().numpy()
    finally:
        lib.fdn_set_flow_iter_variant(1)


@pytest.mark.parametrize("shape", [(1024, 1024), (512, 1024), (77, 150), (12, 300), (33, 40)])
@pytest.mark.parametrize("win", [1, 3, 4, 5, 7, 9, 15, 31])
def test_flow_iterations_vs_oracle(eng, shape, win):
    """1-4 iterations for n pairs == UpdateMatrices + Gaussian blur-solve of the oracle, chained; the register-ring
    kernel (winsize 4, 5, 8, 9) and the shared-memory-ring kernel agree bit for bit."""
    h, w = shape
    n = 2 if h * w > 100000 else 3
    imgs = O.synthetic_volume((2 * n, h, w), seed=h + win, noise_sigma=10.0)
    R = np.stack([O.polyexp(imgs[i]) for i in range(2 * n)])
    rng = np.random.default_rng(win)
    flow = (rng.standard_normal((n, h, w, 2)) * 1.5).astype(np.float32)
    flow[0, :4, :4] = 50.0      # out-of-image lookups take the border branch
    dR = dev(R_from_oracle_layout(R))
    ref = [flow[i] for i in range(n)]
    for iters in range(1, 5):
        ref = [GW.gauss_blur_solve(O.update_matrices(R[i], R[n + i], ref[i]), win) for i in range(n)]
        got = _iterations(eng.lib, dR, n, flow, h, w, win, iters)
        for i in range(n):
            assert np.array_equal(got[i], ref[i]), f"iters {iters} pair {i}: bit-equal {np.mean(got[i] == ref[i])}"
        if (win // 2) in (2, 4):
            assert np.array_equal(_iterations(eng.lib, dR, n, flow, h, w, win, iters, variant=0), got), iters


@pytest.mark.parametrize("case", G.CASES, ids=G.case_key)
def test_farneback_vs_golden(eng, golden, case):
    g = golden("gaussian_window.npz")
    H, W, l, w, it, pn, ps = case
    prev, nxt = G.case_images(H, W)
    for flags in (256, 256 | 4):
        flow = dev(G.init_flow(H, W)[None]) if flags & 4 else torch.zeros((1, H, W, 2), device="cuda")
        eng.farneback(dev(prev[None]), dev(nxt[None]), flow, gparams(l, w, bool(flags & 4), it, pn, ps))
        assert sha(flow[0].cpu().numpy()) == str(g[f"sha_{G.case_key(case)}_f{flags}"]), flags


@pytest.mark.parametrize("levels", range(6))
def test_farneback_levels_vs_oracle(eng, levels):
    H, W = 520, 640
    v = O.synthetic_volume((3, H, W), seed=levels, noise_sigma=10.0)
    init = G.init_flow(H, W)
    for use_prev in (False, True):
        flow = dev(np.stack([init, init])) if use_prev else torch.zeros((2, H, W, 2), device="cuda")
        eng.farneback(dev(v[0:2]), dev(v[1:3]), flow, gparams(levels, 7, use_prev))
        got = flow.cpu().numpy()
        for i in range(2):
            ref = GW.farneback_c(v[i], v[i + 1], init.copy() if use_prev else None, levels, 7,
                                 flags=256 | (4 * use_prev))
            assert np.array_equal(got[i], ref), (i, use_prev)


@pytest.mark.parametrize("recompute", [False, True])
def test_filter_toy_vs_golden(golden, recompute):
    from flowdenoising_b200 import flowdenoising as fd
    g = golden("gaussian_window.npz")
    kernels = [fd.get_gaussian_kernel(s) for s in G.TOY_SIGMAS]
    get_flow = fd.get_flow_without_prev_flow if recompute else fd.get_flow_with_prev_flow
    obj = fd.FlowDenoising(1, G.toy_volume(), 3, 5, get_flow, fd.warp_slice, gaussian_window=True)
    zyx = obj.filter(kernels)
    prefix = "toyr" if recompute else "toy"
    assert sha(obj.vol) == str(g[f"{prefix}_sha_ZY"])
    assert sha(zyx) == str(g[f"{prefix}_sha_ZYX"])
    # the Z pass alone, and the module-level get_flow functions with the keyword
    obj = fd.FlowDenoising(1, G.toy_volume(), 3, 5, get_flow, fd.warp_slice, gaussian_window=True)
    obj.filter_along_Z(kernels[0])
    assert sha(obj.filtered_vol) == str(g[f"{prefix}_sha_Z"])
    toy = G.toy_volume()
    f = get_flow(toy[1], toy[0], 3, 5, None, gaussian_window=True)
    assert np.array_equal(f, GW.farneback_c(toy[0], toy[1], None, 3, 5))


def test_cfg1_passes_vs_golden(eng, golden):
    """BASELINE.json configs[0] (64 x 256 x 256, sigma 2, Farneback defaults) with the Gaussian window: SHA-256 after
    each pass equals cv2's, and FlowDenoising.filter() gives the same volume."""
    from flowdenoising_b200 import flowdenoising as fd
    g = golden("gaussian_window.npz")
    vol = G.cfg1_volume()
    assert sha(vol) == str(g["cfg1_input_sha256"])
    k = O.get_gaussian_kernel(2.0)
    cur = dev(vol)
    for axis, name in enumerate(("Z", "ZY", "ZYX")):
        out = torch.empty_like(cur)
        eng.filter_along_axis(cur, out, axis, k, gparams())
        assert sha(out.cpu().numpy()) == str(g[f"cfg1_sha_{name}"]), name
        cur = out
    res = fd.FlowDenoising(1, vol.copy(), gaussian_window=True).filter([k] * 3)
    assert sha(res) == str(g["cfg1_sha_ZYX"])


def test_views_and_chunks_equal_the_whole_axis(eng):
    """fdn_filter_axis in Gaussian mode: chunk < n_out, windows of a periodic view (halo > 0) and non-periodic slab
    views with an explicit halo give the bits of the whole-axis call."""
    from flowdenoising_b200._lib import View
    vol = O.synthetic_volume((20, 64, 96), seed=7, noise_sigma=8.0)
    k = O.get_gaussian_kernel(1.5)     # r = 6
    r = k.size // 2
    p = gparams(2, 9)
    Z, Y, X = vol.shape
    d_in = dev(vol)
    full = torch.empty_like(d_in)
    eng.filter_along_axis(d_in, full, 0, k, p)
    assert not torch.equal(full, _box_pass(eng, d_in, k))
    for chunk in (1, 3, 7):
        out = torch.empty_like(d_in)
        eng.filter_view(d_in, out, View(Z, Z, 0, 1, Y, X, Y * X, X, Y * X, X), k, p, chunk=chunk)
        assert torch.equal(out, full), chunk
    for first, count in ((0, 6), (6, 14), (17, 3)):
        out = torch.full_like(d_in, -7.0)
        eng.filter_view(d_in, out[first:], View(Z, count, first, 1, Y, X, Y * X, X, Y * X, X), k, p, chunk=2)
        assert torch.equal(out[first:first + count], full[first:first + count])
        assert bool((out[:first] == -7.0).all()) and bool((out[first + count:] == -7.0).all())
    for s0, cnt in ((0, 4), (9, 5), (16, 4)):
        idx = [(z % Z) for z in range(s0 - r, s0 + cnt + r)]
        slab = d_in[idx].contiguous()
        o = torch.empty((cnt, Y, X), dtype=torch.float32, device="cuda")
        eng.filter_view(slab, o, View(len(idx), cnt, r, 0, Y, X, Y * X, X, Y * X, X), k, p)
        assert torch.equal(o, full[s0:s0 + cnt]), s0


def _box_pass(eng, d_in, k):
    from flowdenoising_b200.engine import FlowParams
    out = torch.empty_like(d_in)
    eng.filter_along_axis(d_in, out, 0, k, FlowParams(2, 9))
    return out


def test_other_paths_equal_in_core(eng, monkeypatch, tmp_path):
    """Hidden-transfer filter() from a host array and the streaming path carry the Gaussian window: both equal the
    in-core device result."""
    from flowdenoising_b200 import flowdenoising as fd
    from flowdenoising_b200.streaming import StreamingDenoiser
    vol = O.synthetic_volume((21, 40, 52), seed=11, noise_sigma=8.0)
    kernels = [O.get_gaussian_kernel(s) for s in (1.0, 0.75, 0.5)]
    p = gparams(2, 5)
    zy_ref, zyx_ref = (t.cpu().numpy() for t in eng.filter(dev(vol), kernels, p))
    from flowdenoising_b200.engine import FlowParams
    assert not np.array_equal(eng.filter(dev(vol), kernels, FlowParams(2, 5))[1].cpu().numpy(), zyx_ref)
    # hidden transfers (forced on a toy volume)
    monkeypatch.setattr(fd, "_OVERLAP_MIN_BYTES", 0)
    plans = []
    orig = fd.GaussianDenoising._filter_overlapped

    def spy(self, e, ks, flow, head, tail):
        plans.append(flow)
        return orig(self, e, ks, flow, head, tail)
    monkeypatch.setattr(fd.GaussianDenoising, "_filter_overlapped", spy)
    obj = fd.FlowDenoising(1, vol.copy(), 2, 5, gaussian_window=True)
    res = obj.filter(kernels)
    assert plans and plans[0].gaussian_window
    assert np.array_equal(res, zyx_ref) and np.array_equal(obj.vol, zy_ref)
    # streaming (-m): a read-only memory map in slabs of 5 slices, and through FlowDenoising with streaming forced
    path = tmp_path / "vol.f32"
    vol.tofile(path)
    mm = np.memmap(path, dtype=np.float32, mode="r", shape=vol.shape)
    zy, zyx = StreamingDenoiser(p, slab_slices=5).filter(mm, kernels)
    assert np.array_equal(zy, zy_ref) and np.array_equal(zyx, zyx_ref)
    obj = fd.FlowDenoising(1, vol.copy(), 2, 5, gaussian_window=True)
    obj.streaming = True
    obj.slab_slices = 4
    assert np.array_equal(obj.filter(kernels), zyx_ref)


def _dist_worker(rank, world, port, out_dir):
    import os
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from flowdenoising_b200.dist import DistributedDenoiser
        from flowdenoising_b200.engine import DeviceEngine
        e = DeviceEngine(torch.device("cuda", rank))
        vol = O.synthetic_volume((18, 64, 80), seed=51, noise_sigma=8.0)
        kernels = [O.get_gaussian_kernel(s) for s in (1.0, 0.5, 0.75)]
        dd = DistributedDenoiser(e, vol.shape, gparams())
        zs, ze = dd.z_range
        _zy, zyx = dd.filter(torch.from_numpy(vol[zs:ze].copy()).cuda(), kernels, want_zy=True)
        torch.cuda.synchronize()
        np.save(os.path.join(out_dir, f"zyx_{rank}.npy"), zyx.cpu().numpy())
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [1, 2])
def test_distributed_equals_in_core(eng, tmp_path, world):
    """The slab-sharded DistributedDenoiser (one process per GPU, NCCL) carries the Gaussian window."""
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    import socket
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    vol = O.synthetic_volume((18, 64, 80), seed=51, noise_sigma=8.0)
    kernels = [O.get_gaussian_kernel(s) for s in (1.0, 0.5, 0.75)]
    ref = eng.filter(dev(vol), kernels, gparams())[1].cpu().numpy()
    mp.spawn(_dist_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    got = np.concatenate([np.load(tmp_path / f"zyx_{r}.npy") for r in range(world)])
    assert np.array_equal(got, ref)


class Arena:
    """One device allocation; sub-buffers separated by guard bands filled with a byte pattern."""

    def __init__(self, sizes):
        self.offsets = []
        off = GUARD
        for s in sizes:
            s = (int(s) + 255) // 256 * 256
            self.offsets.append((off, s))
            off += s + GUARD
        self.buf = torch.full((off,), PATTERN, dtype=torch.uint8, device="cuda")

    def view(self, i, dtype=torch.float32):
        off, s = self.offsets[i]
        return self.buf[off:off + s].view(dtype)

    def check(self):
        pos = 0
        for off, s in self.offsets:
            assert bool((self.buf[pos:off] == PATTERN).all()), f"guard band before offset {off} was written"
            pos = off + s
        assert bool((self.buf[pos:] == PATTERN).all()), "guard band at the end was written"


@pytest.mark.parametrize("shape,n", [((64, 1024), 4), ((40, 300), 3), ((33, 35), 2), ((9, 130), 3)])
@pytest.mark.parametrize("win", [5, 9, 15, 31])
def test_flow_iterations_stay_in_bounds_and_repeat(eng, shape, n, win):
    lib = eng.lib
    h, w = shape
    imgs = O.synthetic_volume((n + 1, h, w), seed=3, noise_sigma=6.0)
    rf = lib.fdn_polyexp_floats(h, w)
    fl_bytes = 8 * n * h * w
    ar = Arena([4 * rf * (n + 1), fl_bytes, fl_bytes, fl_bytes, 4 * (n + 1) * h * w])
    R, f0, f1, f2, d_img = ar.view(0), ar.view(1), ar.view(2), ar.view(3), ar.view(4)
    d_img[:(n + 1) * h * w].copy_(torch.from_numpy(imgs).cuda().view(-1))
    assert lib.fdn_polyexp(d_img.data_ptr(), n + 1, h, w, 5, 1.2, R.data_ptr(), None) == 0, lib.fdn_last_error()
    rng = np.random.default_rng(8)
    flow = torch.from_numpy((rng.standard_normal((n, h, w, 2)) * 3).astype(np.float32)).cuda()
    digests = set()
    for variant in (1, 0, 1):
        lib.fdn_set_flow_iter_variant(variant)
        try:
            for _ in range(2):
                f0[:2 * n * h * w].copy_(flow.view(-1))
                res = C.c_void_p()
                rc = lib.fdn_flow_iterations_gaussian(R.data_ptr(), R.data_ptr() + 4 * rf, f0.data_ptr(), f1.data_ptr(),
                                                      f2.data_ptr(), n, h, w, win, 4, None, C.byref(res))
                assert rc == 0, lib.fdn_last_error()
                out = {f0.data_ptr(): f0, f1.data_ptr(): f1, f2.data_ptr(): f2}[res.value]
                digests.add(hashlib.sha256(out[:2 * n * h * w].cpu().numpy().tobytes()).hexdigest())
        finally:
            lib.fdn_set_flow_iter_variant(1)
    ar.check()
    assert len(digests) == 1


def test_pass_stays_in_bounds(eng):
    """A whole Gaussian-window pass with an exactly sized workspace between guard bands, chunked."""
    from flowdenoising_b200._lib import OfParams, View
    lib = eng.lib
    vol = O.synthetic_volume((11, 64, 96), seed=6, noise_sigma=8.0)
    Z, Y, X = vol.shape
    k = np.ascontiguousarray(O.get_gaussian_kernel(1.0))
    kp = k.ctypes.data_as(C.POINTER(C.c_double))
    of = OfParams(3, 9, 3, 5, 1.2, 1, 256)
    v = View(Z, Z, 0, 1, Y, X, Y * X, X, Y * X, X)
    need = lib.fdn_workspace_bytes(C.byref(v), k.size, C.byref(of), 4)
    ar = Arena([4 * vol.size, 4 * vol.size, need])
    d_in, d_out, ws = ar.view(0), ar.view(1), ar.view(2, torch.uint8)
    d_in[:vol.size].copy_(torch.from_numpy(vol).cuda().view(-1))
    rc = lib.fdn_filter_axis(d_in.data_ptr(), d_out.data_ptr(), C.byref(v), kp, k.size, C.byref(of), 4, ws.data_ptr(),
                             need, None)
    assert rc == 0, lib.fdn_last_error()
    ar.check()
    ref = GW.flow_axis_c(vol, 0, k, winsize=9)
    assert np.array_equal(d_out[:vol.size].cpu().numpy().reshape(vol.shape), ref)


def test_launch_log(eng):
    """With the flag every flow iteration is one launch of the Gaussian kernel and no box kernel runs; without it the
    launches are those of the box path."""
    from flowdenoising_b200.engine import FlowParams, level_geometry
    lib = eng.lib
    H, W = 256, 1024
    v = O.synthetic_volume((2, H, W), seed=41, noise_sigma=10.0)
    nl = len(level_geometry(H, W, 3))
    logs = {}
    for name, p in (("gauss5", gparams(3, 5)), ("gauss15", gparams(3, 15)), ("box", FlowParams(3, 5))):
        flow = torch.zeros((1, H, W, 2), dtype=torch.float32, device="cuda")
        lib.fdn_launch_log_enable(1)
        eng.farneback(dev(v[0:1]), dev(v[1:2]), flow, p)
        torch.cuda.synchronize()
        lib.fdn_launch_log_enable(0)
        logs[name] = _launch_names(lib)
    g5, g15, box = logs["gauss5"], logs["gauss15"], logs["box"]
    assert g5.count("k_flow_gauss_iter") == 3 * nl and "k_flow_gauss_iter_smem" not in g5
    assert g15.count("k_flow_gauss_iter_smem") == 3 * nl and "k_flow_gauss_iter" not in g15
    for names in (g5, g15):
        assert not any(n.startswith("k_flow_iter") for n in names), names
    assert not any(n.startswith("k_flow_gauss") for n in box) and "k_flow_iter_ws" in box
    strip = lambda names: [n for n in names if not n.startswith("k_flow_gauss") and not n.startswith("k_flow_iter")]
    assert strip(g5) == strip(box) == strip(g15)


def test_profile_record(eng):
    from flowdenoising_b200 import _lib
    lib = eng.lib
    names = [lib.fdn_profile_kernel_name(i) for i in range(lib.fdn_profile_kernel_count())]
    kid = names.index(b"k_flow_gauss_iter")
    h, w = 96, 200
    v = O.synthetic_volume((2, h, w), seed=2, noise_sigma=10.0)
    lib.fdn_profile_reset()
    lib.fdn_profile_enable(1)
    try:
        eng.farneback(dev(v[0:1]), dev(v[1:2]), torch.zeros((1, h, w, 2), device="cuda"), gparams(0, 5))
        torch.cuda.synchronize()
    finally:
        lib.fdn_profile_enable(0)
    ms, n, by = C.c_double(), C.c_int64(), C.c_double()
    _lib.check(lib.fdn_profile_read(kid, C.byref(ms), C.byref(n), C.byref(by)))
    lib.fdn_profile_reset()
    assert n.value == 3 and by.value == 3 * 56.0 * h * w and ms.value > 0


def test_cli_writes_the_api_volume(tmp_path, golden):
    from flowdenoising_b200 import flowdenoising as fd
    from flowdenoising_b200 import volume_io
    g = golden("gaussian_window.npz")
    vol = G.toy_volume()
    sig = [str(s) for s in G.TOY_SIGMAS]
    src = tmp_path / "toy.mrc"
    volume_io.write_mrc(str(src), vol)
    out = tmp_path / "out.mrc"
    assert fd.main(["-i", str(src), "-o", str(out), "-s", *sig, "-l", "3", "-w", "5", "--gaussian_window"]) == 0
    got = volume_io.read_volume(str(out))
    api = fd.FlowDenoising(1, vol.copy(), 3, 5, gaussian_window=True).filter(
        [fd.get_gaussian_kernel(float(s)) for s in G.TOY_SIGMAS])
    assert np.array_equal(got, api) and sha(got) == str(g["toy_sha_ZYX"])
