"""Box-window Farneback (the default flow mode) over every parameter the C ABI accepts, bit for bit against the C
oracle, which tests/test_flow_params_oracle.py pins against live cv2 at the same points: every winsize 1..31 on every
dispatch edge of the flow iteration, poly_n 1..7 with any poly_sigma, the 39- and 79-tap pyramid levels, flow
resizes by 16 and 32, whole Farneback runs over a sampled grid, and images wider than 64 strips. Every case asserts
from the launch log which kernel ran, so a sweep cannot silently miss a branch.

It also holds the regression tests of the flow-iteration scratch: a coarser pyramid level can need more strip carries
than level 0 (a level-0 width of 97..128 px is one strip of k_flow_iter, the 48..64 px of level 1 are two, and
cvRound rounds an odd height up), so the scratch is sized by the largest level, checked here with the workspace
between guard bands and against a Python restatement of the layout."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import fd_oracle as O

torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu

GUARD = 1 << 20
PATTERN = 0xA5
WS_CWMAX = (120, 116)      # widest k_flow_iter_ws strip: winsize 4/5 (m = 2) and 8/9 (m = 4)


@pytest.fixture(scope="module")
def eng():
    from flowdenoising_b200.engine import DeviceEngine
    return DeviceEngine()


@pytest.fixture(scope="module")
def lib():
    from flowdenoising_b200 import _lib
    return _lib.load()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def images(shape, n, seed):
    return O.synthetic_volume((n,) + tuple(shape), seed=seed, noise_sigma=10.0)


def R_floats(h, w):
    p = h * w
    return 4 * p + (p + 3) // 4 * 4


def R_to_oracle_layout(R, h, w):   # library layout (n, R_floats): [h*w] float4 + [h*w] float  ->  (n, h, w, 5)
    n = R.shape[0]
    out = np.empty((n, h, w, 5), np.float32)
    out[..., :4] = R[:, :4 * h * w].reshape(n, h, w, 4)
    out[..., 4] = R[:, 4 * h * w:5 * h * w].reshape(n, h, w)
    return out


def R_from_oracle_layout(R):  # (n, h, w, 5) -> (n, R_floats)
    n, h, w, _ = R.shape
    out = np.zeros((n, R_floats(h, w)), np.float32)
    out[:, :4 * h * w] = R[..., :4].reshape(n, -1)
    out[:, 4 * h * w:5 * h * w] = R[..., 4].reshape(n, -1)
    return out


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


class LaunchLog:
    def __init__(self, lib):
        self.lib = lib

    def __enter__(self):
        self.lib.fdn_launch_log_enable(1)
        self.names = []
        return self

    def __exit__(self, *exc):
        torch.cuda.synchronize()
        self.lib.fdn_launch_log_enable(0)
        self.names[:] = [self.lib.fdn_launch_log_name(i).decode() for i in range(self.lib.fdn_launch_log_count())]


# ---- the dispatch rules of flow.cu, restated ----
def cdiv(a, b):
    return -(-a // b)


def ws_takes(h, w, winsize):
    """k_flow_iter_ws (variant 1) takes winsize 4/5/8/9 on images of w % 4 == 0, w >= 64, h >= 16."""
    return winsize // 2 in (2, 4) and w % 4 == 0 and w >= 64 and h >= 16


def strip_instantiation(w, winsize):
    """k_flow_iter<CW, TR, MT, MINB> that launch_flow_iter_strip picks."""
    m = winsize // 2
    if w > 96:
        return (128, 6, 2, 4) if m == 2 else (128, 4, 4, 4) if m == 4 else (128, 4, 0, 4)
    return (32, 4, 2, 8) if m == 2 else (32, 4, 0, 8)


def flow_kernels(h, w, winsize, iters, variant=1):
    if variant == 1 and ws_takes(h, w, winsize):
        return ["k_flow_iter_ws"] * cdiv(iters, 3)      # one launch runs up to three iterations
    return ["k_flow_iter"] * iters


def strip_width(w):
    return 128 if w > 96 else 32


def ws_strips_max(w):
    def strips(cwmax):
        s = cdiv(w, cwmax)
        return cdiv(w, (cdiv(w, s) + 3) // 4 * 4)
    return max(strips(c) for c in WS_CWMAX)


def a256(v):
    return (v + 255) // 256 * 256


def scratch_bytes(cap, levels_hw):
    """flow_scratch_make: counters, then flags, packets and carries of the largest level."""
    flags = max(cdiv(w, strip_width(w)) for h, w in levels_hw)
    packets = max(ws_strips_max(w) * h for h, w in levels_hw)
    carries = max(cdiv(w, strip_width(w)) * h for h, w in levels_hw)
    return 256 + a256(4 * 3 * cap) + a256(8 * cap * flags) + a256(16 * 5 * cap * packets) + a256(8 * 5 * cap * carries)


def workspace_bytes(n, H, W, klen, levels, chunk, esize):
    """make_plan of a periodic pass of n slices of H x W."""
    geo = [(h, w) for h, w, _k, _s in O.level_geometry(H, W, levels)]
    r = klen // 2
    chunk = n if chunk <= 0 or chunk > n else chunk
    slots = n if chunk + 2 * r >= n else chunk + 2 * r
    px = chunk * H * W
    total = a256(4 * sum(R_floats(h, w) for h, w in geo) * slots) + 3 * a256(16 * px) + a256(esize * px * r)
    total += a256(scratch_bytes(2 * chunk, geo))
    if esize != 4:
        total += a256(4 * px)
    return total


def carries_exceed_level0(H, W, levels):
    geo = [(h, w) for h, w, _k, _s in O.level_geometry(H, W, levels)]
    rows = [cdiv(w, strip_width(w)) * h for h, w in geo]
    return max(rows) > rows[0]


# ------------------------------------------------------------------------------------------------
# Stage 3: one pyramid level, every winsize, every dispatch edge
# ------------------------------------------------------------------------------------------------
# (16, 64) / (15, 64) / (16, 63): the h >= 16 and w >= 64 thresholds of k_flow_iter_ws; (20, 66) and (18, 97):
# w % 4 != 0; (17, 96) / (18, 97): narrow (32-column) vs wide (128-column) strips; (24, 100) and (33, 260): wide
# strips, 1 and 3 of them; the rest are smaller than the window in one direction, down to 1 x N and N x 1.
STAGE3_SHAPES = [(16, 64), (15, 64), (16, 63), (20, 66), (17, 96), (18, 97), (24, 100), (33, 260), (1, 40), (40, 1),
                 (3, 200), (9, 130), (70, 7)]
_R_CACHE = {}


def stage3_inputs(shape):
    """(R of 2 prev + 2 next images, initial flow of 2 pairs), computed once per shape."""
    if shape not in _R_CACHE:
        h, w = shape
        imgs = images(shape, 4, 40 + h + w)
        R = np.stack([O.polyexp(imgs[i]) for i in range(4)])
        rng = np.random.default_rng(h * 1000 + w)
        flow = (rng.standard_normal((2, h, w, 2)) * 1.5).astype(np.float32)
        flow[0, :3, :3] = 50.0      # out-of-image lookups take the border branch
        _R_CACHE[shape] = (R, flow)
    return _R_CACHE[shape]


def test_stage3_grid_reaches_every_kernel():
    """The shapes above reach k_flow_iter_ws (also at winsize 4 and 8) and each k_flow_iter instantiation."""
    ws_wins = {win for (h, w) in STAGE3_SHAPES for win in range(1, 32) if ws_takes(h, w, win)}
    assert ws_wins == {4, 5, 8, 9}
    inst = {strip_instantiation(w, win) for (h, w) in STAGE3_SHAPES for win in range(1, 32)}
    assert inst == {(128, 6, 2, 4), (128, 4, 4, 4), (128, 4, 0, 4), (32, 4, 2, 8), (32, 4, 0, 8)}
    assert {win % 5 + 1 for win in (4, 5, 8, 9)} >= {1, 4, 5}     # merged launches of 3 + 1 and 3 + 2 iterations


@gpu
@pytest.mark.parametrize("shape", STAGE3_SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
@pytest.mark.parametrize("winsize", range(1, 32))
def test_flow_iterations_every_winsize(eng, lib, shape, winsize):
    """UpdateMatrices + box mean + solve, chained `iters` times (1..5 over the winsizes), both flow-iteration variants,
    against O.blur_solve(O.update_matrices(...)). One iteration goes through fdn_flow_iteration, more through
    fdn_flow_iterations (k_flow_iter_ws runs up to three per launch: 4 and 5 are 3 + 1 and 3 + 2)."""
    h, w = shape
    n = 2
    iters = winsize % 5 + 1
    R, flow = stage3_inputs(shape)
    ref = flow.copy()
    for _ in range(iters):
        ref = np.stack([O.blur_solve(O.update_matrices(R[b], R[n + b], ref[b]), winsize) for b in range(n)])
    dR = dev(R_from_oracle_layout(R))
    nscr = lib.fdn_flow_iteration_scratch_bytes(n, h, w)
    scr = torch.zeros(nscr, dtype=torch.uint8, device="cuda")
    for variant in (0, 1):
        cur = dev(flow)
        lib.fdn_set_flow_iter_variant(variant)
        try:
            with LaunchLog(lib) as log:
                if iters == 1:
                    out = torch.empty_like(cur)
                    rc = lib.fdn_flow_iteration(dR[:n].data_ptr(), dR[n:].data_ptr(), cur.data_ptr(), out.data_ptr(), n,
                                                h, w, winsize, scr.data_ptr(), nscr, None)
                else:
                    t1, t2 = torch.empty_like(cur), torch.empty_like(cur)
                    res = C.c_void_p()
                    rc = lib.fdn_flow_iterations(dR[:n].data_ptr(), dR[n:].data_ptr(), cur.data_ptr(), t1.data_ptr(),
                                                 t2.data_ptr(), n, h, w, winsize, iters, scr.data_ptr(), nscr, None,
                                                 C.byref(res))
                    if rc == 0:
                        out = {cur.data_ptr(): cur, t1.data_ptr(): t1, t2.data_ptr(): t2}[res.value]
        finally:
            lib.fdn_set_flow_iter_variant(1)
        assert rc == 0, lib.fdn_last_error()
        assert log.names == flow_kernels(h, w, winsize, iters, variant), (variant, log.names)
        got = out.cpu().numpy()
        assert np.array_equal(got.view(np.int32), ref.view(np.int32)), \
            f"variant {variant}, {iters} iterations: bit-equal fraction {np.mean(got == ref):.5f}"


# ------------------------------------------------------------------------------------------------
# Stage 2: polynomial expansion
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("poly_n", range(1, 8))
@pytest.mark.parametrize("poly_sigma", [0.0, 0.6, 1.1, 1.5])
def test_polyexp_every_poly_n(lib, poly_n, poly_sigma):
    """FarnebackPolyExp for poly_n 1..7 (sigma 0 is n * 0.3). w % 4 == 0 takes the TMA kernel (k_polyexp_tma<5> for
    poly_n 5, k_polyexp_tma<0> otherwise), w % 4 != 0 the generic k_polyexp. The branches are reached through shapes:
    FDN_POLYEXP_TMA=0 (which disables the TMA kernel) is read once per process, so a test cannot switch it."""
    tma = os.environ.get("FDN_POLYEXP_TMA", "1").strip() != "0"
    n = 2
    for h, w in ((40, 64), (37, 70), (9, 8)):
        imgs = images((h, w), n, 3 + poly_n) * np.float32(0.731)
        R = torch.zeros((n, R_floats(h, w)), dtype=torch.float32, device="cuda")
        with LaunchLog(lib) as log:
            rc = lib.fdn_polyexp(dev(imgs).data_ptr(), n, h, w, poly_n, poly_sigma, R.data_ptr(), None)
        assert rc == 0, lib.fdn_last_error()
        assert log.names == ["k_polyexp_tma" if tma and w % 4 == 0 else "k_polyexp"], (h, w, log.names)
        got = R_to_oracle_layout(R.cpu().numpy(), h, w)
        for i in range(n):
            ref = O.polyexp(imgs[i], poly_n, poly_sigma)
            assert np.array_equal(got[i], ref), f"{h}x{w}: max|d|={np.abs(got[i] - ref).max()}"


# ------------------------------------------------------------------------------------------------
# Stage 1: pyramid levels 4 and 5, flow resizes by 16 and 32
# ------------------------------------------------------------------------------------------------
def blur_kernels(H, W, ksz, h, w):
    names = ["k_blur_rows4" if ksz in (3, 9, 19, 39, 79) and W % 4 == 0 and W >= 4 + ksz else "k_blur_rows",
             "k_blur_cols4" if ksz in (3, 9, 19, 39, 79) and H >= 4 + ksz else "k_blur_cols"]
    return names + (["k_resize_linear_img"] if (h, w) != (H, W) else [])


@gpu
@pytest.mark.parametrize("H,W", [(1024, 1024), (1030, 1030), (70, 1032), (70, 1030)])
@pytest.mark.parametrize("level", [4, 5])
def test_pyramid_deep_levels(lib, H, W, level):
    """The 39- and 79-tap smoothing of levels 4 and 5 (taps and sigma of a 1024 x 1024 image's geometry), through the
    4-outputs-per-thread blurs (W % 4 == 0, H >= 4 + taps) and the generic ones (W % 4 != 0, short images)."""
    _h, _w, ksz, sigma = O.level_geometry(1024, 1024, 5)[level]
    assert ksz == {4: 39, 5: 79}[level]
    h, w = int(np.rint(H / 2 ** level)), int(np.rint(W / 2 ** level))
    n = 2
    imgs = images((H, W), n, 50 + level) + np.float32(0.37)
    tmp = torch.empty(2 * n * H * W, dtype=torch.float32, device="cuda")
    out = torch.empty((n, h, w), dtype=torch.float32, device="cuda")
    with LaunchLog(lib) as log:
        rc = lib.fdn_pyramid_level(dev(imgs).data_ptr(), n, H, W, H * W, W, ksz, sigma, h, w, tmp.data_ptr(),
                                   out.data_ptr(), None)
    assert rc == 0, lib.fdn_last_error()
    assert log.names == blur_kernels(H, W, ksz, h, w), log.names
    got = out.cpu().numpy()
    for i in range(n):
        ref = O.pyramid_level(imgs[i], ksz, sigma, h, w)
        assert np.array_equal(got[i], ref), f"max|d|={np.abs(got[i] - ref).max()}"


@gpu
@pytest.mark.parametrize("H,W,factor", [(1024, 1040, 16), (1024, 1055, 32), (1030, 1030, 16)])
def test_flow_resize_by_16_and_32(lib, H, W, factor):
    """The initial flow of level 4 / 5 (INTER_AREA down, times 1/16 or 1/32) and a linear upsample over the same
    factor (the kernel's own factor-2 scale included)."""
    rng = np.random.default_rng(factor + W)
    n = 2
    h, w = int(np.rint(H / factor)), int(np.rint(W / factor))
    flow = (rng.standard_normal((n, H, W, 2)) * 3).astype(np.float32)
    out = torch.empty((n, h, w, 2), dtype=torch.float32, device="cuda")
    with LaunchLog(lib) as log:
        rc = lib.fdn_flow_area_down(dev(flow).data_ptr(), n, H, W, out.data_ptr(), h, w, 1.0 / factor, None)
    assert rc == 0, lib.fdn_last_error()
    assert log.names == ["k_flow_area_down"]
    for i in range(n):
        ref = O.resize_area(flow[i], h, w) * np.float32(1.0 / factor)
        assert np.array_equal(out[i].cpu().numpy(), ref)
    small = (rng.standard_normal((n, h, w, 2)) * 2).astype(np.float32)
    up = torch.empty((n, H, W, 2), dtype=torch.float32, device="cuda")
    with LaunchLog(lib) as log:
        rc = lib.fdn_flow_upsample(dev(small).data_ptr(), n, h, w, up.data_ptr(), H, W, None)
    assert rc == 0, lib.fdn_last_error()
    assert log.names == ["k_flow_upsample2" if W % 2 == 0 else "k_flow_upsample"], log.names
    for i in range(n):
        ref = O.resize_linear(small[i], H, W, ipp=False) * np.float32(2)
        assert np.array_equal(up[i].cpu().numpy(), ref)


# ------------------------------------------------------------------------------------------------
# End to end: calcOpticalFlowFarneback over a sampled parameter grid
# ------------------------------------------------------------------------------------------------
# (H, W, levels, winsize, iterations, poly_n, poly_sigma, use_prev_flow)
E2E_CASES = [
    (64, 80, 0, 5, 3, 5, 1.2, False),
    (64, 80, 1, 1, 2, 3, 0.0, True),
    (96, 128, 2, 2, 3, 1, 0.6, False),
    (96, 128, 3, 4, 4, 7, 1.5, True),
    (130, 200, 4, 8, 5, 6, 1.1, False),
    (260, 300, 5, 30, 1, 2, 0.0, True),
    (300, 260, 5, 31, 3, 4, 0.6, False),
    (1024, 1032, 5, 9, 2, 5, 1.1, True),
    (1030, 1024, 4, 5, 3, 5, 1.2, False),
    (67, 100, 3, 7, 3, 5, 1.2, True),          # level 1 (34 x 50) needs more strip carries than level 0
    (1, 40, 3, 5, 3, 5, 1.2, True),
    (2, 40, 3, 1, 1, 5, 1.2, False),
    (40, 1, 3, 15, 2, 5, 1.2, True),
    (3, 3, 3, 31, 3, 5, 1.2, False),
    (5, 200, 3, 4, 5, 7, 1.5, True),
    (200, 5, 3, 8, 4, 3, 0.6, False),
]


def test_e2e_grid_covers_the_parameter_ranges():
    levels_run = {len(O.level_geometry(H, W, lv)) - 1 for (H, W, lv, *_r) in E2E_CASES}
    assert levels_run == set(range(6))
    assert {c[3] for c in E2E_CASES} >= {1, 2, 4, 8, 30, 31}
    assert {c[5] for c in E2E_CASES} == set(range(1, 8))
    assert {c[4] for c in E2E_CASES} == set(range(1, 6))
    assert {c[7] for c in E2E_CASES} == {False, True}


def farneback_and_log(eng, lib, prev, nxt, init, params):
    flow = dev(init)
    with LaunchLog(lib) as log:
        eng.farneback(dev(prev), dev(nxt), flow, params)
    return flow.cpu().numpy(), log.names


def expected_flow_kernels(H, W, levels, winsize, iters):
    names = []
    for h, w, _k, _s in O.level_geometry(H, W, levels):
        names += flow_kernels(h, w, winsize, iters)
    return sorted(names)


@gpu
@pytest.mark.parametrize("case", E2E_CASES, ids=lambda c: "{}x{}_l{}_w{}_it{}_p{}-{}_{}".format(*c))
def test_farneback_grid(eng, lib, case):
    from flowdenoising_b200.engine import FlowParams
    H, W, levels, winsize, iters, poly_n, poly_sigma, use_prev = case
    n = 2
    imgs = images((H, W), n + 1, H + W + winsize)
    prev, nxt = imgs[:n], imgs[1:]
    rng = np.random.default_rng(winsize)
    init = (rng.standard_normal((n, H, W, 2)) * 0.8).astype(np.float32) if use_prev else np.zeros((n, H, W, 2),
                                                                                                  np.float32)
    got, names = farneback_and_log(eng, lib, prev, nxt, init,
                                   FlowParams(levels, winsize, iters, poly_n, poly_sigma, use_prev))
    assert sorted(x for x in names if x.startswith("k_flow_iter")) == expected_flow_kernels(H, W, levels, winsize, iters)
    for b in range(n):
        ref = O.farneback_c(prev[b], nxt[b], init[b].copy(), levels, winsize, iters, poly_n, poly_sigma,
                            flags=4 if use_prev else 0)
        assert np.array_equal(got[b].view(np.int32), ref.view(np.int32)), \
            f"pair {b}: bit-equal fraction {np.mean(got[b] == ref):.5f}"


@gpu
@pytest.mark.parametrize("shape,axis,params", [
    ((12, 20, 60), 0, (3, 31, 2, 5, 1.2)),      # winsize 31 on 20-row slices
    ((10, 48, 72), 1, (2, 4, 1, 7, 1.5)),       # winsize 4, poly_n 7, one iteration; slices of 10 x 72
], ids=["w31_short_slices", "w4_poly7_it1"])
def test_pass_with_non_default_flow_params(eng, lib, shape, axis, params):
    from flowdenoising_b200.engine import FlowParams
    levels, winsize, iters, poly_n, poly_sigma = params
    vol = O.synthetic_volume(shape, seed=17, noise_sigma=8.0)
    k = O.get_gaussian_kernel(1.0)
    d_in = dev(vol)
    out = torch.empty_like(d_in)
    with LaunchLog(lib) as log:
        eng.filter_along_axis(d_in, out, axis, k, FlowParams(levels, winsize, iters, poly_n, poly_sigma, True))
    H, W = [s for i, s in enumerate(shape) if i != axis]
    kinds = {x for x in log.names if x.startswith("k_flow_iter")}
    assert kinds == {"k_flow_iter_ws" if ws_takes(H, W, winsize) else "k_flow_iter"}, log.names
    ref = O.flow_axis_c(vol, axis, k, levels, winsize, iters, poly_n, poly_sigma)
    assert np.array_equal(out.cpu().numpy(), ref)


# ------------------------------------------------------------------------------------------------
# Scratch sized by the largest level (a coarser level can need more strip carries than level 0)
# ------------------------------------------------------------------------------------------------
# (Z, Y, X, axis): the slices of the pass are H x W with H = 3 (mod 4) and a level-0 width of 97..127
DEFECT1_CASES = [((64, 67, 100), 0), ((71, 10, 110), 1)]


def pass_view(shape, axis):
    from flowdenoising_b200._lib import View
    Z, Y, X = shape
    if axis == 0:
        return View(Z, Z, 0, 1, Y, X, Y * X, X, Y * X, X), Y, X
    return View(Y, Y, 0, 1, Z, X, X, Y * X, X, Y * X), Z, X


@pytest.mark.parametrize("n,H,W,levels,chunk", [(64, 67, 100, 3, 0), (10, 71, 110, 3, 4), (64, 256, 256, 3, 0),
                                                (16, 1024, 1024, 5, 8), (9, 40, 500, 3, 9), (6, 16, 8200, 3, 0),
                                                (12, 35, 12000, 3, 5), (7, 131, 127, 4, 3)])
@pytest.mark.parametrize("esize", [4, 1, 2])
def test_workspace_bytes_restated(lib, n, H, W, levels, chunk, esize):
    """fdn_workspace_bytes(_typed) equals a restatement of the pass layout whose flow-iteration scratch holds the
    largest level (not level 0); fdn_farneback_workspace_bytes likewise. Host code only: no GPU needed."""
    from flowdenoising_b200 import _lib
    from flowdenoising_b200._lib import OfParams, View
    of = OfParams(levels, 5, 3, 5, 1.2, 1, 0)
    v = View(n, n, 0, 1, H, W, 0, 0, 0, 0)
    klen = 9
    want = workspace_bytes(n, H, W, klen, levels, chunk, esize)
    if esize == 4:
        assert lib.fdn_workspace_bytes(C.byref(v), klen, C.byref(of), chunk) == want
    code = {4: _lib.DTYPE_F32, 1: _lib.DTYPE_U8, 2: _lib.DTYPE_I16}[esize]
    assert lib.fdn_workspace_bytes_typed(C.byref(v), klen, C.byref(of), chunk, code) == want
    geo = [(h, w) for h, w, _k, _s in O.level_geometry(H, W, levels)]
    fb = a256(4 * sum(R_floats(h, w) for h, w in geo) * 2 * n) + 2 * a256(8 * n * H * W) + a256(scratch_bytes(n, geo))
    assert lib.fdn_farneback_workspace_bytes(n, H, W, C.byref(of)) == fb
    assert lib.fdn_flow_iteration_scratch_bytes(n, H, W) == scratch_bytes(n, geo[:1])


@gpu
@pytest.mark.parametrize("shape,axis", DEFECT1_CASES, ids=["Z_64x67x100", "Y_71x10x110"])
def test_pass_with_coarse_level_carries_stays_in_bounds(eng, lib, shape, axis):
    """A float32 OF pass with the exactly sized workspace between guard bands, output guarded as well. Level 1 runs
    k_flow_iter on more strip-rows than level 0 (e.g. 34 x 50: 2 strips x 34 rows against 1 x 67)."""
    v, H, W = pass_view(shape, axis)
    assert carries_exceed_level0(H, W, 3)
    from flowdenoising_b200._lib import OfParams
    vol = O.synthetic_volume(shape, seed=61, noise_sigma=8.0)
    k = np.ascontiguousarray(O.get_gaussian_kernel(1.0))
    of = OfParams(3, 5, 3, 5, 1.2, 1, 0)
    need = lib.fdn_workspace_bytes(C.byref(v), k.size, C.byref(of), 0)
    assert need == workspace_bytes(v.n_in, H, W, k.size, 3, 0, 4)
    ar = Arena([4 * vol.size, 4 * vol.size, need])
    d_in, d_out, ws = ar.view(0), ar.view(1), ar.view(2, torch.uint8)
    d_in[:vol.size].copy_(torch.from_numpy(vol).cuda().view(-1))
    with LaunchLog(lib) as log:
        rc = lib.fdn_filter_axis(d_in.data_ptr(), d_out.data_ptr(), C.byref(v), k.ctypes.data_as(C.POINTER(C.c_double)),
                                 k.size, C.byref(of), 0, ws.data_ptr(), need, None)
    assert rc == 0, lib.fdn_last_error()
    assert "k_flow_iter" in log.names
    ar.check()
    ref = O.flow_axis_c(vol, axis, k)
    assert np.array_equal(d_out[:vol.size].cpu().numpy().reshape(shape), ref)


@gpu
@pytest.mark.parametrize("shape,axis", DEFECT1_CASES, ids=["Z_64x67x100", "Y_71x10x110"])
@pytest.mark.parametrize("dtype", [np.uint8, np.int16], ids=["uint8", "int16"])
def test_typed_pass_with_coarse_level_carries(lib, shape, axis, dtype):
    """The same geometry through fdn_filter_axis_typed: there the flow-iteration scratch is followed by the chunk's
    float32 accumulator, so carries written past the scratch would change the output."""
    from flowdenoising_b200 import _lib
    from flowdenoising_b200._lib import OfParams
    from oracle import fd_oracle_int as I
    v, H, W = pass_view(shape, axis)
    code = {np.uint8: _lib.DTYPE_U8, np.int16: _lib.DTYPE_I16}[dtype]
    esize = np.dtype(dtype).itemsize
    vol = I.integer_volume(shape, dtype, seed=62)
    k = np.ascontiguousarray(O.get_gaussian_kernel(1.0))
    of = OfParams(3, 5, 3, 5, 1.2, 1, 0)
    need = lib.fdn_workspace_bytes_typed(C.byref(v), k.size, C.byref(of), 0, code)
    assert need == workspace_bytes(v.n_in, H, W, k.size, 3, 0, esize)
    nb = vol.nbytes
    ar = Arena([nb, nb, need])
    d_in, d_out, ws = ar.view(0, torch.uint8), ar.view(1, torch.uint8), ar.view(2, torch.uint8)
    d_in[:nb].copy_(torch.from_numpy(vol.view(np.uint8).reshape(-1)).cuda())
    rc = lib.fdn_filter_axis_typed(d_in.data_ptr(), d_out.data_ptr(), code, C.byref(v),
                                   k.ctypes.data_as(C.POINTER(C.c_double)), k.size, C.byref(of), 0, ws.data_ptr(),
                                   need, None)
    assert rc == 0, lib.fdn_last_error()
    torch.cuda.synchronize()
    ar.check()
    o = I.IntegerDenoiser(8, vol.copy(), True, 3, 5, backend="c")
    o.filter_along_axis(axis, k)
    got = d_out[:nb].cpu().numpy().view(dtype).reshape(shape)
    assert np.array_equal(got, o.filtered_vol), f"equal fraction {np.mean(got == o.filtered_vol):.5f}"


# ------------------------------------------------------------------------------------------------
# Images wider than 64 strips
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("W", [7700, 8192, 8200, 12000])
@pytest.mark.parametrize("winsize", [5, 9, 7])
def test_farneback_wide_images(eng, lib, W, winsize):
    """7700 px are 65 strips of k_flow_iter_ws at winsize 5 and 67 at 9; 8200 px are 65 strips of k_flow_iter (winsize
    7); 12000 px are 94 of them."""
    from flowdenoising_b200.engine import FlowParams
    H, n = 16, 1
    imgs = images((H, W), n + 1, W + winsize)
    init = np.zeros((n, H, W, 2), np.float32)
    got, names = farneback_and_log(eng, lib, imgs[:n], imgs[1:], init, FlowParams(3, winsize, 3, 5, 1.2, True))
    assert sorted(x for x in names if x.startswith("k_flow_iter")) == expected_flow_kernels(H, W, 3, winsize, 3)
    ref = O.farneback_c(imgs[0], imgs[1], None, 3, winsize, 3, 5, 1.2)
    assert np.array_equal(got[0].view(np.int32), ref.view(np.int32)), f"bit-equal fraction {np.mean(got[0] == ref):.5f}"


@gpu
def test_pass_over_wide_slices(eng, lib):
    """A default Z pass over slices of 16 x 8200 px (69 strips of k_flow_iter_ws)."""
    from flowdenoising_b200.engine import FlowParams
    vol = O.synthetic_volume((6, 16, 8200), seed=71, noise_sigma=8.0)
    k = O.get_gaussian_kernel(1.0)
    d_in = dev(vol)
    out = torch.empty_like(d_in)
    with LaunchLog(lib) as log:
        eng.filter_along_axis(d_in, out, 0, k, FlowParams())
    assert "k_flow_iter_ws" in log.names and "k_flow_iter" not in log.names
    assert np.array_equal(out.cpu().numpy(), O.flow_axis_c(vol, 0, k))
