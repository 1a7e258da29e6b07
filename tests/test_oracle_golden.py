"""Pins the CPU oracle (oracle/) against outputs of the UNMODIFIED reference (tests/golden, made by
oracle/gen_golden.py from /root/reference/src/flowdenoising.py) and against live cv2 calls.

The reference itself has no tests or golden vectors (SURVEY.md §4), so these fixtures are the pin."""
import hashlib

import numpy as np
import pytest

from oracle import fd_oracle as O

cv2 = pytest.importorskip("cv2")


def test_gaussian_kernel_matches_reference(golden):
    g = golden("kernels.npz")
    for s in g["sigmas"]:
        ref = g[f"k_{s}"]
        got = O.get_gaussian_kernel(float(s))
        assert got.size == ref.size == 2 * int(4 * s + 0.5) + 1
        assert np.array_equal(got, ref), s


@pytest.mark.parametrize("case", ["a", "b", "d"])
def test_c_farneback_and_warp_bit_exact_vs_reference(golden, case):
    """C restatement of cv2.calcOpticalFlowFarneback / cv2.remap vs the reference's get_flow / warp_slice
    (src/flowdenoising.py:55-114): bit-exact on the fixtures (zero-init, chained, --recompute_flow)."""
    g = golden("flows.npz")
    v = g[f"{case}_vol"].astype(np.float32)
    l, w = (int(x) for x in g[f"{case}_lw"])
    centre = v[0]
    prev = np.zeros(centre.shape + (2,), np.float32)
    for j in (1, 2, 3):
        prev = O.farneback_c(centre, v[j], prev, l, w, flags=4)
        if j != 2:
            ref = g[f"{case}_flow_chain{j}"]
            assert np.array_equal(prev, ref), f"chain{j}: max diff {np.abs(prev - ref).max()}"
    assert np.array_equal(O.warp_slice_c(v[3], prev), g[f"{case}_warp_chain3"])
    f2 = O.farneback_c(centre, v[2], None, l, w, flags=0)
    assert np.array_equal(f2, g[f"{case}_flow_noprev2"])


def test_c_farneback_vs_live_cv2_odd_shapes():
    for shape, l, w, seed in [((100, 100), 3, 5, 5), ((77, 131), 3, 5, 6), ((260, 300), 3, 7, 7)]:
        v = O.synthetic_volume((2,) + shape, seed=seed)
        ref = cv2.calcOpticalFlowFarneback(v[0], v[1], None, 0.5, l, w, 3, 5, 1.2, 0)
        got = O.farneback_c(v[0], v[1], None, l, w)
        epe = np.sqrt(((ref - got) ** 2).sum(-1))
        # bit-exact on the AVX2 build host; other hosts may differ in OpenCV's SIMD tails (1 ulp of the blur)
        assert epe.mean() < 1e-5 and epe.max() < 1e-3


@pytest.mark.parametrize("backend", ["cv2", "c"])
def test_oracle_driver_of_matches_reference(golden, backend):
    g = golden("toy_of.npz")
    vol = g["vol"].astype(np.float32)
    kernels = [O.get_gaussian_kernel(float(s)) for s in g["sigmas"]]
    o = O.OracleDenoiser(3, vol.copy(), True, int(g["l"]), int(g["w"]), backend=backend)
    o.filter_along_Z(kernels[0]); assert np.array_equal(o.filtered_vol, g["Z"])
    o.vol[...] = o.filtered_vol
    o.filter_along_Y(kernels[1]); assert np.array_equal(o.filtered_vol, g["ZY"])
    o.vol[...] = o.filtered_vol
    o.filter_along_X(kernels[2]); assert np.array_equal(o.filtered_vol, g["ZYX"])


def test_oracle_c_pass_matches_reference(golden):
    g = golden("toy_of.npz")
    vol = g["vol"].astype(np.float32)
    k = O.get_gaussian_kernel(float(g["sigmas"][0]))
    assert np.array_equal(O.flow_axis_c(vol, 0, k), g["Z"])
    k = O.get_gaussian_kernel(float(g["sigmas"][1]))
    assert np.array_equal(O.flow_axis_c(g["Z"], 1, k), g["ZY"])
    k = O.get_gaussian_kernel(float(g["sigmas"][2]))
    assert np.array_equal(O.flow_axis_c(g["ZY"], 2, k), g["ZYX"])


def test_oracle_recompute_flow_matches_reference(golden):
    g = golden("toy_of_recompute.npz")
    vol = g["vol"].astype(np.float32)
    k = O.get_gaussian_kernel(float(g["sigmas"][0]))
    assert np.array_equal(O.flow_axis_c(vol, 0, k, use_prev_flow=False), g["Z"])
    o = O.OracleDenoiser(2, vol.copy(), True, recompute_flow=True)
    o.filter_along_Z(k)
    assert np.array_equal(o.filtered_vol, g["Z"])


@pytest.mark.parametrize("name", ["toy_noof.npz", "toy_noof_float.npz"])
def test_oracle_noof_matches_reference(golden, name):
    g = golden(name)
    vol = g["vol"].astype(np.float32)
    kernels = [O.get_gaussian_kernel(float(s)) for s in g["sigmas"]]
    o = O.OracleDenoiser(2, vol.copy(), use_OF=False)
    out = o.filter(kernels)
    assert np.array_equal(out, g["ZYX"]) and np.array_equal(o.vol, g["ZY"])
    a = O.gauss_axis_c(vol, 0, kernels[0]); assert np.array_equal(a, g["Z"])
    b = O.gauss_axis_c(a, 1, kernels[1]); assert np.array_equal(b, g["ZY"])
    c = O.gauss_axis_c(b, 2, kernels[2]); assert np.array_equal(c, g["ZYX"])


def test_synthetic_volume_reproducible_and_cfg1_slice(golden):
    """cfg 1 input regenerates bit-identically; one Z-pass slice of the C oracle equals the reference's."""
    g = golden("cfg1_slices.npz")
    vol = O.synthetic_volume((64, 256, 256), seed=0, noise_sigma=20.0)
    assert hashlib.sha256(vol.tobytes()).hexdigest() == str(g["input_sha256"])
    k = O.get_gaussian_kernel(2.0)
    out = np.zeros_like(vol)
    O.flow_axis_c(vol, 0, k, s0=37, s1=38, out=out)
    assert np.array_equal(out[37], g["Z"][1])


def test_veltkamp_split_is_round_to_nearest_even_float32():
    """The exact no-OF kernels (csrc/noof.cu) round a float64 sum to float32 precision with Veltkamp's splitting
    (p = s * (2^29 + 1); hi = (s - p) + p) instead of a double -> float -> double conversion pair. The two must agree
    for every zero / float32-normal value, exact ties (round half to even) and mantissa carries included."""
    rng = np.random.default_rng(1)
    n = 3_000_000
    expo = rng.integers(1023 - 112, 1023 + 127, n, dtype=np.uint64)
    mant_hi = rng.integers(0, 2 ** 20, n, dtype=np.uint64)
    top3 = rng.integers(0, 8, n, dtype=np.uint64)
    kind = rng.integers(0, 6, n)
    mant_hi = np.where(kind >= 4, np.uint64(0xFFFFF), mant_hi)          # all ones above the rounding position
    top3 = np.where(kind >= 4, np.uint64(7), top3)
    low29 = np.where(kind % 2 == 0, np.uint64(0x10000000), rng.integers(0, 2 ** 29, n, dtype=np.uint64))   # exact ties
    low29 = np.where(kind == 3, np.uint64(0x10000000) + rng.integers(-1, 2, n).astype(np.int64).astype(np.uint64),
                     low29) & np.uint64(0x1FFFFFFF)
    bits = (expo << np.uint64(52)) | (mant_hi << np.uint64(32)) | (top3 << np.uint64(29)) | low29
    s = bits.view(np.float64)
    s = np.where(rng.integers(0, 2, n) == 1, -s, s)
    # (-0.0 is the one value the two forms disagree on -- Veltkamp returns +0.0 -- and it cannot occur: the kernels'
    # sums start from +0.0, and x + y is -0.0 under round-to-nearest only when both operands are -0.0)
    s[:3] = [0.0, 2.0 ** -112, -(2.0 ** 127)]
    with np.errstate(over="ignore"):
        ref = s.astype(np.float32).astype(np.float64)
    ok = np.isfinite(ref)                                               # (values that round up to 2^128 overflow)
    p = s * (2.0 ** 29 + 1)
    hi = (s - p) + p
    assert np.count_nonzero(low29 == 0x10000000) > 1_000_000
    assert np.array_equal(hi[ok].view(np.uint64), ref[ok].view(np.uint64))
