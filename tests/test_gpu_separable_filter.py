"""The 1-D filter a pass applies, over every kernel length the C ABI accepts, with asymmetric taps.

With a Gaussian k[r - d] == k[r + d], so a kernel that swaps the two sides of the window, or is off by one slot, passes
every test that uses Gaussian taps. Here the taps are drawn from a seeded generator (positive; with negative taps; with
a zero tap and a tap of 3.0, outside the range in which the exact no-OF kernels round with float64 instructions) and
each case is compared with a plain restatement of the reference's arithmetic:

* no optical flow, float32, exact mode: NumPy's `tmp_slice += slice * kernel[i]` (float64 product and sum, rounded to
  float32 after every tap, periodic), bit for bit, for klen 1 .. 257 along Z, Y (strided views) and X (rows), on
  output counts around the 128-slice segment of k_gauss_axis_ring, volumes shorter than the kernel, windows with a
  halo and more than 65535 rows;
* the fast mode against a float64 convolution, within the rounding of the float32 taps and of the FMA chain;
* integer volumes (generic kernels, truncation toward zero at the store);
* the optical-flow pass (k_warp_pair, k_acc_finish) against the C oracle, r = 0 .. 128, chunk remainders with and
  without the whole-axis cache, halo windows, integer volumes and a batch of more than 65535 image pairs;
* fdn_warp_accumulate with a non-Gaussian weight.

Every case asserts from the launch log which kernel ran; the vector width each kernel picks is not in the log, so the
rules of launch_gauss_axis_ring and launch_warp_pair are restated below and a CPU test checks that the shapes reach
every width."""
import numpy as np
import pytest

from oracle import fd_oracle as O

torch = pytest.importorskip("torch")
gpu = pytest.mark.gpu

KLENS = [1, 3, 5, 7, 9, 11, 13, 17, 21, 25, 33, 35, 41, 65, 129, 257]
RING = {5, 9, 13, 17, 21, 25, 33}          # the specialised lengths of csrc/noof.cu
TAP_KINDS = ["positive", "negative", "zero_and_3"]


@pytest.fixture(scope="module")
def eng():
    from flowdenoising_b200.engine import DeviceEngine
    return DeviceEngine()


@pytest.fixture(scope="module")
def lib():
    from flowdenoising_b200 import _lib
    return _lib.load()


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


# ---- taps ----
def taps(klen, kind, seed=0):
    """Asymmetric taps (klen > 1) from a seeded generator."""
    rng = np.random.default_rng(1000 * klen + 7 * TAP_KINDS.index(kind) + seed)
    if kind == "positive":
        k = rng.uniform(0.05, 1.0, klen)
        k /= k.sum()
    elif kind == "negative":
        k = rng.standard_normal(klen)
        k /= np.abs(k).sum()
    else:
        k = rng.uniform(0.05, 1.0, klen) / klen
        k[rng.integers(klen)] = 3.0
        if klen > 1:
            k[(np.argmax(k) + 1 + rng.integers(klen - 1)) % klen] = 0.0
    if klen > 1:
        assert not np.array_equal(k, k[::-1])
    return k


def integer_taps(klen, seed=0):
    """Nonnegative asymmetric taps summing to less than 1 (an integer result stays in range), one of them zero."""
    rng = np.random.default_rng(5000 + klen + seed)
    k = rng.uniform(0.05, 1.0, klen)
    if klen > 2:
        k[rng.integers(klen)] = 0.0
    return k / k.sum() * 0.999


# ---- the reference's arithmetic, restated ----
def filter0(inp, n_out, halo, periodic, k):
    """out[s] = fold_i f32(f64(acc) + f64(inp[s + halo + i - r]) * k[i]) along axis 0 of inp (n_in slices)."""
    n_in = inp.shape[0]
    r = k.size // 2
    s = np.arange(n_out)
    x = inp.astype(np.float32).astype(np.float64)
    acc = np.zeros((n_out,) + inp.shape[1:], np.float32)
    with np.errstate(all="ignore"):
        for i in range(k.size):
            j = s + halo + i - r
            if periodic:
                j = j % n_in
            acc = (acc.astype(np.float64) + x[j] * k[i]).astype(np.float32)
    return acc


def numpy_axis_filter(vol, axis, k):
    """Periodic pass along `axis` (src/flowdenoising.py:133-158 under NumPy >= 2)."""
    v = np.moveaxis(vol, axis, 0)
    return np.ascontiguousarray(np.moveaxis(filter0(v, v.shape[0], 0, True, k), 0, axis))


def conv0(inp, n_out, halo, periodic, k):
    """sum_i k[i] v[s + halo + i - r] and sum_i |k[i]| |v[s + halo + i - r]| in float64, along axis 0."""
    v = inp.astype(np.float64)
    r = k.size // 2
    s = np.arange(n_out)
    e = np.zeros((n_out,) + v.shape[1:])
    a = np.zeros_like(e)
    for i in range(k.size):
        j = s + halo + i - r
        if periodic:
            j = j % v.shape[0]
        e += k[i] * v[j]
        a += abs(k[i]) * np.abs(v[j])
    return e, a


def conv64(vol, axis, k):
    v = np.moveaxis(vol, axis, 0)
    e, a = conv0(v, v.shape[0], 0, True, k)
    return np.moveaxis(e, 0, axis), np.moveaxis(a, 0, axis)


def fma_bound(klen, a):
    """Rounding the taps to float32 and the FMA chain: (klen + 2) 2^-24 sum |k_i| |v_i|."""
    return (klen + 2) * 2.0 ** -24 * a


# ---- dispatch rules, restated ----
def ring_vec(klen, exact, W, strides, ptrs):
    """launch_gauss_axis_ring: the widest vector every address of the view is aligned for; the exact mode keeps its
    window in float64 and stops at 2; four columns only up to 17 taps. strides: the view's four strides (elements);
    ptrs: the input and output addresses (bytes)."""
    def aligned(n):
        return W % n == 0 and all(s % n == 0 for s in strides) and all(p % (4 * n) == 0 for p in ptrs)
    vec = 2 if aligned(2) else 1
    if not exact and klen <= 17 and aligned(4):
        vec = 4
    return vec


def axis_kernel(klen):
    return "k_gauss_axis_ring" if klen in RING else "k_gauss_axis"


def rows_kernel(klen, exact, W, ptrs):
    if klen in RING and W % 4 == 0 and all(p % 16 == 0 for p in ptrs):
        return "k_gauss_rows_tile" if exact else "k_gauss_rows_direct"
    return "k_gauss_rows"


def warp_vec(W, strides, ptrs):
    """launch_warp_pair / launch_acc_finish / launch_warp_acc: four pixels per thread iff W % 4 == 0 and every stride
    and address allows 16-byte float accesses."""
    return 4 if W % 4 == 0 and all(s % 4 == 0 for s in strides) and all(p % 16 == 0 for p in ptrs) else 1


def view_strides(shape, axis):
    Z, Y, X = shape
    if axis == 0:
        return (X, Y * X, X, Y * X)     # in_row, in_slice, out_row, out_slice
    return (Y * X, X, Y * X, X)


# (shape, axis, element offset of the input and output tensors). The offset moves the base pointer off the 8- and
# 16-byte boundaries (1) or off the 16-byte boundary only (2). Filtered-axis lengths 127, 128, 129, 257 sit around
# the 128-slice segment of k_gauss_axis_ring; 2, 3, 5, 7 are shorter than most kernels (the wrap applies repeatedly).
STRIDED_CASES = [
    ((129, 6, 20), 0, 0),      # W % 4 == 0
    ((128, 5, 22), 0, 0),      # W % 2 == 0, W % 4 != 0
    ((127, 4, 19), 0, 0),      # odd W
    ((257, 3, 12), 0, 1),      # misaligned base pointer
    ((3, 128, 24), 1, 2),      # Y pass, 8- but not 16-byte aligned
    ((4, 129, 18), 1, 0),
    ((5, 3, 16), 0, 0),
    ((2, 7, 12), 1, 0),
]
ROWS_CASES = [
    ((5, 7, 132), 0),          # W % 4 == 0: the specialised row kernels for the RING lengths
    ((4, 6, 130), 0),
    ((3, 5, 131), 0),
    ((4, 5, 132), 1),          # misaligned: generic kernel
    ((6, 5, 8), 0),            # rows shorter than most kernels
]


def ptr_of(t):
    return t.data_ptr()


def device_volume(vol, offset):
    """A contiguous CUDA tensor holding vol whose data starts `offset` elements into its allocation."""
    src = torch.from_numpy(np.ascontiguousarray(vol))
    buf = torch.empty(src.numel() + offset, dtype=src.dtype, device="cuda")
    t = buf[offset:].view(src.shape)
    t.copy_(src)
    return t


def empty_like_offset(t, offset):
    buf = torch.empty(t.numel() + offset, dtype=t.dtype, device=t.device)
    return buf[offset:].view(t.shape)


def test_shapes_reach_every_vector_width():
    """CPU: the STRIDED_CASES reach vector widths 1 and 2 of the exact ring kernel and 1, 2 and 4 of the fast one; the
    row cases reach the specialised and the generic row kernels; the OF cases reach both warp widths."""
    seen = set()
    for shape, axis, off in STRIDED_CASES:
        W = shape[2]
        ptrs = (256 + 4 * off, 512 + 4 * off)
        for klen in RING:
            for exact in (True, False):
                seen.add((exact, ring_vec(klen, exact, W, view_strides(shape, axis), ptrs)))
    assert seen == {(True, 1), (True, 2), (False, 1), (False, 2), (False, 4)}
    kinds = {rows_kernel(klen, ex, s[2], (256 + 4 * o,)) for s, o in ROWS_CASES for klen in KLENS for ex in (1, 0)}
    assert kinds == {"k_gauss_rows", "k_gauss_rows_tile", "k_gauss_rows_direct"}
    assert {warp_vec(shape[2], view_strides(shape, axis), (256,)) for _i, shape, axis, _k, _c in OF_CASES} == {1, 4}


def random_volume(shape, seed):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal(shape) * 60 + 40).astype(np.float32)


# ------------------------------------------------------------------------------------------------
# No optical flow, float32
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("klen", KLENS)
def test_noof_exact_strided_axes(eng, lib, klen):
    for ci, (shape, axis, off) in enumerate(STRIDED_CASES):
        vol = random_volume(shape, seed=klen + 31 * ci)
        d_in = device_volume(vol, off)
        out = empty_like_offset(d_in, off)
        for kind in TAP_KINDS:
            k = taps(klen, kind)
            with LaunchLog(lib) as log:
                eng.filter_along_axis(d_in, out, axis, k, None, exact=True)
            assert log.names == [axis_kernel(klen)], (shape, axis, log.names)
            want = numpy_axis_filter(vol, axis, k)
            got = out.cpu().numpy()
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), \
                (shape, axis, off, kind, f"vec {ring_vec(klen, True, shape[2], view_strides(shape, axis), (ptr_of(d_in), ptr_of(out)))}",
                 f"equal {np.mean(got == want):.5f}")


@gpu
@pytest.mark.parametrize("klen", KLENS)
def test_noof_exact_rows(eng, lib, klen):
    for ci, (shape, off) in enumerate(ROWS_CASES):
        vol = random_volume(shape, seed=klen + 17 * ci)
        d_in = device_volume(vol, off)
        out = empty_like_offset(d_in, off)
        for kind in TAP_KINDS:
            k = taps(klen, kind)
            with LaunchLog(lib) as log:
                eng.filter_along_axis(d_in, out, 2, k, None, exact=True)
            assert log.names == [rows_kernel(klen, True, shape[2], (ptr_of(d_in), ptr_of(out)))], (shape, log.names)
            want = numpy_axis_filter(vol, 2, k)
            assert np.array_equal(out.cpu().numpy().view(np.uint32), want.view(np.uint32)), (shape, off, kind)


@gpu
@pytest.mark.parametrize("klen", KLENS)
def test_noof_exact_halo_window(eng, lib, klen):
    """A non-periodic view (the multi-GPU slab): output slice s is centred on input slice s + halo; one slice more than
    needed on each side, so that reading one slot too far or too near changes the result."""
    from flowdenoising_b200._lib import View
    r = klen // 2
    n_out, halo = 9, r + 1
    n_in = n_out + 2 * halo
    Y, X = 5, 20
    inp = random_volume((n_in, Y, X), seed=klen)
    d_in = device_volume(inp, 0)
    out = torch.empty((n_out, Y, X), dtype=torch.float32, device="cuda")
    for kind in TAP_KINDS:
        k = taps(klen, kind)
        for exact in (True, False):
            with LaunchLog(lib) as log:
                eng.filter_view(d_in, out, View(n_in, n_out, halo, 0, Y, X, Y * X, X, Y * X, X), k, None, exact=exact)
            assert log.names == [axis_kernel(klen)]
            got = out.cpu().numpy()
            if exact:
                want = filter0(inp, n_out, halo, False, k)
                assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), kind
            else:
                e, a = conv0(inp, n_out, halo, False, k)
                assert np.all(np.abs(got - e) <= fma_bound(klen, a)), kind


@gpu
@pytest.mark.parametrize("klen", [3, 5, 33, 35])
def test_noof_rows_more_than_65535(eng, lib, klen):
    """300 x 300 x 8: 90000 rows. The generic row kernel runs in batches of 65535 rows, the specialised ones put the
    rest in gridDim.z."""
    vol = random_volume((300, 300, 8), seed=klen)
    d_in = device_volume(vol, 0)
    out = torch.empty_like(d_in)
    k = taps(klen, "zero_and_3")
    with LaunchLog(lib) as log:
        eng.filter_along_axis(d_in, out, 2, k, None, exact=True)
    name = rows_kernel(klen, True, 8, (16, 16))
    assert log.names == [name] * (1 if name != "k_gauss_rows" else 2), log.names
    want = numpy_axis_filter(vol, 2, k)
    assert np.array_equal(out.cpu().numpy().view(np.uint32), want.view(np.uint32))
    with LaunchLog(lib) as log:
        eng.filter_along_axis(d_in, out, 2, k, None, exact=False)
    assert log.names == [rows_kernel(klen, False, 8, (16, 16))] * len(log.names) and len(log.names) in (1, 2)
    e, a = conv64(vol, 2, k)
    assert np.all(np.abs(out.cpu().numpy() - e) <= fma_bound(klen, a))


@gpu
@pytest.mark.parametrize("klen", KLENS)
def test_noof_fast_within_the_fma_bound(eng, lib, klen):
    """|fast - sum k_i v_i| <= (klen + 2) 2^-24 sum |k_i| |v_i|: the float32 rounding of the taps and of the FMA chain."""
    cases = [(s, a, o) for s, a, o in STRIDED_CASES] + [(s, 2, o) for s, o in ROWS_CASES]
    for ci, (shape, axis, off) in enumerate(cases):
        vol = random_volume(shape, seed=7 * klen + ci)
        d_in = device_volume(vol, off)
        out = empty_like_offset(d_in, off)
        for kind in TAP_KINDS:
            k = taps(klen, kind)
            with LaunchLog(lib) as log:
                eng.filter_along_axis(d_in, out, axis, k, None, exact=False)
            ptrs = (ptr_of(d_in), ptr_of(out))
            want_name = rows_kernel(klen, False, shape[2], ptrs) if axis == 2 else axis_kernel(klen)
            assert log.names == [want_name], (shape, axis, log.names)
            e, a = conv64(vol, axis, k)
            err = np.abs(out.cpu().numpy().astype(np.float64) - e)
            bound = fma_bound(klen, a)
            assert np.all(err <= bound), (shape, axis, kind, float((err / np.maximum(bound, 1e-300)).max()))


@gpu
def test_noof_fast_mode_ulps_from_exact(eng, lib):
    """The fast mode's largest distance from the exact mode, in float32 ulps, for Gaussian taps of every length on a
    volume of 8-bit-like values (the documented accuracy of the fast mode). Printed per length; asserted against the
    bound of the test above (2 klen + 2 ulp for a positive sum)."""
    from flowdenoising_b200.engine import gaussian_kernel
    vol = O.synthetic_volume((40, 48, 132), seed=3, noise_sigma=10.0)
    d_in = device_volume(vol, 0)
    a = torch.empty_like(d_in)
    b = torch.empty_like(d_in)
    rows = []
    for klen in KLENS:
        k = gaussian_kernel((klen - 1) / 8) if klen > 1 else np.ones(1)
        assert k.size == klen
        worst = 0
        for axis in range(3):
            eng.filter_along_axis(d_in, a, axis, k, None, exact=True)
            eng.filter_along_axis(d_in, b, axis, k, None, exact=False)
            x = a.cpu().numpy().view(np.int32).astype(np.int64)
            y = b.cpu().numpy().view(np.int32).astype(np.int64)
            worst = max(worst, int(np.abs(x - y).max()))
        rows.append((klen, worst))
        assert worst <= 2 * klen + 2, (klen, worst)
    print("fast mode, largest distance from the exact mode (float32 ulps) per kernel length: " +
          ", ".join(f"{kl}: {w}" for kl, w in rows))


# ------------------------------------------------------------------------------------------------
# No optical flow, integer volumes (generic kernels, exact mode)
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.int8, np.uint16, np.int16], ids=["uint8", "int8", "uint16", "int16"])
@pytest.mark.parametrize("klen", KLENS)
def test_noof_typed(eng, lib, klen, dtype):
    from oracle import fd_oracle_int as I
    for ci, (shape, axis) in enumerate([((9, 6, 20), 0), ((5, 7, 19), 1), ((4, 5, 21), 2), ((3, 4, 132), 2)]):
        vol = I.integer_volume(shape, dtype, seed=klen + ci)
        d_in = torch.from_numpy(vol).cuda()
        out = torch.empty_like(d_in)
        k = integer_taps(klen, ci)
        with LaunchLog(lib) as log:
            eng.filter_along_axis(d_in, out, axis, k, None)
        assert log.names == ["k_gauss_rows" if axis == 2 else "k_gauss_axis"], log.names
        want = numpy_axis_filter(vol, axis, k).astype(dtype)     # truncation toward zero
        got = out.cpu().numpy()
        assert np.array_equal(got, want), (shape, axis, f"equal {np.mean(got == want):.5f}")


# ------------------------------------------------------------------------------------------------
# Optical flow: stage 4 (k_warp_pair, k_acc_finish) with asymmetric taps
# ------------------------------------------------------------------------------------------------
# (id, shape, axis, klen, chunk). Pass images are H x W = (Y, X) for axis 0 and (Z, X) for axis 1.
OF_CASES = [
    ("k1", (5, 40, 48), 0, 1, None),               # r = 0: no flows, only the centre tap
    ("k3_w45", (7, 40, 45), 0, 3, None),           # W % 4 != 0: k_warp_pair<T, 1>
    ("k7_Y_w48", (40, 9, 48), 1, 7, None),         # Y pass, W % 4 == 0: k_warp_pair<T, 4>
    ("k33_short", (6, 36, 44), 0, 33, None),       # 32 neighbours on 6 slices: the wrap applies repeatedly
    ("k257", (6, 40, 48), 0, 257, None),           # r = 128, the largest radius
    ("k3_chunk4", (11, 40, 48), 0, 3, 4),          # chunks 4 + 4 + 3, slices cached per chunk
    ("k7_chunk5_full_wrap", (11, 40, 46), 0, 7, 5),  # chunk + 2r >= n: the whole axis cached once; chunks 5 + 5 + 1
]


@gpu
@pytest.mark.parametrize("case", OF_CASES, ids=lambda c: c[0])
def test_of_pass_asymmetric_taps(eng, lib, case):
    from flowdenoising_b200.engine import FlowParams
    _id, shape, axis, klen, chunk = case
    r = klen // 2
    vol = O.synthetic_volume(shape, seed=40 + klen, noise_sigma=8.0)
    k = taps(klen, "positive", seed=1)
    d_in = torch.from_numpy(vol).cuda()
    out = torch.empty_like(d_in)
    with LaunchLog(lib) as log:
        eng.filter_along_axis(d_in, out, axis, k, FlowParams(), chunk=chunk)
    n = shape[axis]
    nchunks = -(-n // (chunk or n))
    assert log.names.count("k_warp_pair") == r * nchunks, log.names.count("k_warp_pair")
    assert log.names.count("k_acc_finish") == nchunks
    if r == 0:      # no neighbours: no flow is computed, the centre tap alone (the slices' pyramids are still built)
        assert not [x for x in log.names if x.startswith("k_flow") or x.startswith("k_warp")], log.names
    ref = O.flow_axis_c(vol, axis, k)
    got = out.cpu().numpy()
    assert np.array_equal(got, ref), f"bit-equal fraction {np.mean(got == ref):.6f}"


@gpu
def test_of_pass_halo_window(eng, lib):
    """Non-periodic view: output slice s of the slab is centred on slab slice s + halo, with one spare slice on each
    side."""
    from flowdenoising_b200.engine import FlowParams
    from flowdenoising_b200._lib import View
    vol = O.synthetic_volume((12, 40, 44), seed=77, noise_sigma=8.0)
    Z, Y, X = vol.shape
    k = taps(5, "positive", seed=2)
    r = 2
    s0, n_out, halo = 3, 6, r + 1
    idx = [(s0 - halo + q) % Z for q in range(n_out + 2 * halo)]
    slab = torch.from_numpy(np.ascontiguousarray(vol[idx])).cuda()
    out = torch.empty((n_out, Y, X), dtype=torch.float32, device="cuda")
    eng.filter_view(slab, out, View(len(idx), n_out, halo, 0, Y, X, Y * X, X, Y * X, X), k, FlowParams())
    ref = O.flow_axis_c(vol, 0, k, s0=s0, s1=s0 + n_out)
    assert np.array_equal(out.cpu().numpy(), ref[s0:s0 + n_out])


@gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.int16], ids=["uint8", "int16"])
@pytest.mark.parametrize("shape,axis,klen", [((6, 40, 44), 0, 5), ((36, 7, 45), 1, 3)], ids=["Z_w44_k5", "Y_w45_k3"])
def test_of_pass_typed_asymmetric_taps(eng, lib, dtype, shape, axis, klen):
    from oracle import fd_oracle_int as I
    from flowdenoising_b200.engine import FlowParams
    vol = I.integer_volume(shape, dtype, seed=90 + klen)
    k = integer_taps(klen, seed=3)
    d_in = torch.from_numpy(vol).cuda()
    out = torch.empty_like(d_in)
    with LaunchLog(lib) as log:
        eng.filter_along_axis(d_in, out, axis, k, FlowParams())
    assert log.names.count("k_warp_pair") == klen // 2 and log.names.count("k_acc_finish") == 1
    o = I.IntegerDenoiser(8, vol.copy(), True, 3, 5, backend="c")
    o.filter_along_axis(axis, k)
    got = out.cpu().numpy()
    assert np.array_equal(got, o.filtered_vol), f"equal fraction {np.mean(got == o.filtered_vol):.5f}"


@gpu
def test_of_pass_more_than_65535_image_pairs(eng, lib):
    """Y pass of 8 x 32768 x 8 with chunk = 32768: both chain directions together are 65536 image pairs, so
    launch_warp_pair splits the batch."""
    from flowdenoising_b200.engine import FlowParams
    vol = O.synthetic_volume((8, 32768, 8), seed=5, noise_sigma=8.0)
    k = taps(3, "positive", seed=4)
    d_in = torch.from_numpy(vol).cuda()
    out = torch.empty_like(d_in)
    with LaunchLog(lib) as log:
        eng.filter_along_axis(d_in, out, 1, k, FlowParams(), chunk=32768)
    assert log.names.count("k_warp_pair") == 2 and log.names.count("k_acc_finish") == 1, \
        (log.names.count("k_warp_pair"), log.names.count("k_acc_finish"))
    ref = O.flow_axis_c(vol, 1, k)
    got = out.cpu().numpy()
    assert np.array_equal(got, ref), f"bit-equal fraction {np.mean(got == ref):.6f}"
    del d_in, out
    eng.release_workspace()
    torch.cuda.empty_cache()


@gpu
@pytest.mark.parametrize("W", [24, 23])
@pytest.mark.parametrize("with_flow", [True, False], ids=["flow", "identity"])
def test_warp_accumulate(eng, lib, W, with_flow):
    """fdn_warp_accumulate: acc = f32(f64(acc) + f64(remap(neigh, flow)) * weight), k_warp_acc4 for W % 4 == 0."""
    n, H = 3, 20
    rng = np.random.default_rng(W)
    neigh = (rng.standard_normal((n, H, W)) * 50 + 100).astype(np.float32)
    flow = rng.uniform(-3.5, 3.5, (n, H, W, 2)).astype(np.float32)
    acc0 = (rng.standard_normal((n, H, W)) * 10).astype(np.float32)
    weight = -0.3712345678901234
    acc = torch.from_numpy(acc0.copy()).cuda()
    with LaunchLog(lib) as log:
        eng.warp_accumulate(torch.from_numpy(neigh).cuda(), torch.from_numpy(flow).cuda() if with_flow else None,
                            weight, acc)
    assert log.names == ["k_warp_acc4" if W % 4 == 0 else "k_warp_acc"], log.names
    for b in range(n):
        w = O.warp_slice_c(neigh[b], flow[b]) if with_flow else neigh[b]
        want = (acc0[b].astype(np.float64) + w.astype(np.float64) * weight).astype(np.float32)
        assert np.array_equal(acc[b].cpu().numpy(), want), b
