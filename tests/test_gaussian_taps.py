"""The Gaussian taps the package filters with are the reference's taps, bit for bit (CPU only).

The reference builds its kernel by filtering a growing delta with scipy.ndimage.gaussian_filter1d
(src/flowdenoising.py:34-45). That is SciPy's kernel, exp(-x^2 / 2 sigma^2) / sum, computed with NumPy's exp and
NumPy's pairwise sum. The C library's exp differs from NumPy's in the last bit for some arguments (exp(-0.125): taps 7
and 9 of sigma = 2), so a restatement in C is close but not equal; an `allclose` at rtol 4e-16 lets that through.
Every test here compares bits."""
import ctypes as C

import numpy as np
import pytest

from flowdenoising_b200 import _lib, engine
from flowdenoising_b200 import flowdenoising as fd
from oracle import fd_oracle as O

scipy_ndimage = pytest.importorskip("scipy.ndimage")


def reference_taps(sigma):
    """src/flowdenoising.py:34-45, restated: grow a delta from 3 coefficients until gaussian_filter1d leaves at least
    two exact zeros, return the response without its two ends."""
    n = 3
    zeros = 0
    while zeros < 2:
        delta = np.zeros(n)
        delta[n // 2] = 1
        coeffs = scipy_ndimage.gaussian_filter1d(delta, sigma=sigma)
        zeros = coeffs.size - np.count_nonzero(coeffs)
        n += 1
    return coeffs[1:-1]


def sigma_grid():
    """0.05 .. 32.1 in steps of 1/16; every radius boundary (k - 0.5) / 4 (where int(4 sigma + 0.5) steps to k) and
    its neighbours at +-1 ulp; the sigmas of the benchmark configurations and a few that are not dyadic."""
    s = [0.05 + i / 16 for i in range(int((32.1 - 0.05) * 16) + 1)]
    for k in range(1, 130):
        b = (k - 0.5) / 4
        s += [np.nextafter(b, 0.0), b, np.nextafter(b, np.inf)]
    s += [0.5, 1.0, 1.5, 2.0, 2.5, 3.0, 4.0, 0.7, 1.3, 2.2, 0.3, 5.9, 12.345]
    return sorted(set(float(x) for x in s))


SIGMAS = sigma_grid()


@pytest.fixture(scope="module")
def ref():
    return {s: reference_taps(s) for s in SIGMAS}


def mismatches(fn, ref):
    bad = []
    for s, want in ref.items():
        got = np.asarray(fn(s))
        if got.dtype != np.float64 or not np.array_equal(got, want):
            bad.append(s)
    return bad


def test_restatement_equals_the_reference_fixtures(golden):
    """tests/golden/kernels.npz was written by the unmodified reference."""
    g = golden("kernels.npz")
    for s in g["sigmas"]:
        want = g[f"k_{s}"]
        assert np.array_equal(reference_taps(float(s)), want), s
        assert want.size == 2 * int(4 * s + 0.5) + 1


def test_grid_covers_every_radius():
    radii = {int(4 * s + 0.5) for s in SIGMAS}
    assert radii >= set(range(0, 129)), sorted(set(range(0, 129)) - radii)
    assert 2.0 in SIGMAS and 4.0 in SIGMAS


def test_radius_follows_the_reference(ref):
    """The loop stops at radius int(4 sigma + 0.5), rounded in float64 like SciPy rounds it (just below a boundary
    4 sigma + 0.5 may still round up to k)."""
    for s, taps in ref.items():
        assert taps.size == 2 * int(4 * s + 0.5) + 1, s
    for k in range(1, 130):
        assert ref[(k - 0.5) / 4].size == 2 * k + 1


@pytest.mark.parametrize("name,fn", [("engine.gaussian_kernel", engine.gaussian_kernel),
                                     ("flowdenoising.get_gaussian_kernel", fd.get_gaussian_kernel),
                                     ("oracle get_gaussian_kernel", O.get_gaussian_kernel)])
def test_taps_equal_the_reference_bit_for_bit(ref, name, fn):
    bad = mismatches(fn, ref)
    assert not bad, (f"{name}: the taps of {len(bad)} of {len(ref)} sigmas differ from the reference's "
                     f"(sigma 2: {'differs' if 2.0 in bad else 'equal'}, sigma 4: {'differs' if 4.0 in bad else 'equal'}): "
                     + " ".join(f"{s:.17g}" for s in bad))


def test_known_last_bit_cases(ref):
    """sigma = 2 (cfg 1, 2, 3, 5) and 4 (the Z kernel of cfg 4): the sigmas where the C library's exp loses a bit."""
    for s in (2.0, 4.0):
        assert np.array_equal(engine.gaussian_kernel(s), ref[s]), s


@pytest.mark.parametrize("sigma", [0.0, -1.0, -0.0, float("nan"), float("inf"), float("-inf"), 1e6])
def test_bad_sigma_raises(sigma):
    with pytest.raises(ValueError):
        engine.gaussian_kernel(sigma)


def test_c_abi_taps_are_close_and_same_length(ref):
    """fdn_gaussian_kernel stays in the C ABI for C callers: SciPy's formula with the C library's exp. Same length,
    within a few ulp of the reference (include/fdn_b200.h says so)."""
    lib = _lib.load()
    buf = (C.c_double * 512)()
    worst = 0.0
    for s, want in ref.items():
        n = lib.fdn_gaussian_kernel(s, buf, 512)
        assert n == want.size, s
        got = np.frombuffer(buf, dtype=np.float64, count=n)
        worst = max(worst, float(np.max(np.abs(got - want) / np.spacing(want))))
    assert worst <= 8, worst
    for bad in (0.0, -1.0, float("nan"), float("inf"), 1e300):
        assert lib.fdn_gaussian_kernel(bad, buf, 512) == 0, bad


def asymmetric_taps(klen, seed):
    rng = np.random.default_rng(seed)
    k = rng.uniform(0.05, 1.0, klen)
    return k / k.sum()


def test_oracle_tap_order_with_an_asymmetric_kernel():
    """The C pass (O.flow_axis_c) applies kernel[i] to neighbour s + i - r exactly like the reference's loop around live
    cv2 (OracleDenoiser(backend="cv2")): with k[r - d] != k[r + d] a swapped side or a shifted index shows."""
    pytest.importorskip("cv2")
    vol = O.synthetic_volume((6, 40, 48), seed=11, noise_sigma=8.0)
    k = asymmetric_taps(7, seed=5)
    assert not np.array_equal(k, k[::-1])
    o = O.OracleDenoiser(1, vol.copy(), True, backend="cv2")
    o.filter_along_Z(k)
    ref = o.filtered_vol
    assert np.array_equal(O.flow_axis_c(vol, 0, k), ref)
    # the mirrored kernel gives another result: the check above does depend on the order
    assert not np.array_equal(O.flow_axis_c(vol, 0, k[::-1].copy()), ref)
