"""CPU checks of the box-window Farneback oracle (``O.farneback_c``) against live cv2 over every parameter the C ABI
accepts: winsize 1..31, even winsizes with and without an initial flow, poly_n 1..7 with any poly_sigma (0 included),
iterations 1..5, levels 0..5, degenerate image shapes and images wider than 8192 px. tests/test_gpu_flow_params.py
compares the kernels bit for bit with this oracle at the same points, so the oracle has to hold at every one of them.
No GPU needed."""
import numpy as np
import pytest

from oracle import fd_oracle as O

cv2 = pytest.importorskip("cv2")


def image_pair(H, W, seed, drift=(0.7, -0.4)):
    """A smooth textured image and the same scene moved by a sub-pixel drift, plus independent noise: a pair with a
    real flow at any shape, 1 x N and N x 1 included."""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:H, 0:W].astype(np.float64)
    comps = [(rng.uniform(0.03, 0.35), rng.uniform(0.03, 0.35), rng.uniform(0, 2 * np.pi), rng.uniform(10, 40))
             for _ in range(6)]

    def scene(dy, dx):
        v = np.full((H, W), 120.0)
        for fy, fx, ph, a in comps:
            v += a * np.sin(fy * (y + dy) + fx * (x + dx) + ph)
        return v

    prev = scene(0.0, 0.0) + rng.normal(0, 2.0, (H, W))
    nxt = scene(*drift) + rng.normal(0, 2.0, (H, W))
    return np.clip(prev, 0, 255).astype(np.float32), np.clip(nxt, 0, 255).astype(np.float32)


def init_flow(H, W, seed):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((H, W, 2)) * 0.8 + np.float32(0.3)).astype(np.float32)


def check(H, W, levels, winsize, iters=3, poly_n=5, poly_sigma=1.2, use_init=False, seed=0):
    prev, nxt = image_pair(H, W, seed)
    flags = cv2.OPTFLOW_USE_INITIAL_FLOW if use_init else 0
    init = init_flow(H, W, seed + 1) if use_init else None
    ref = cv2.calcOpticalFlowFarneback(prev, nxt, None if init is None else init.copy(), 0.5, levels, winsize, iters,
                                       poly_n, poly_sigma, flags)
    got = O.farneback_c(prev, nxt, None if init is None else init.copy(), levels, winsize, iters, poly_n, poly_sigma,
                        flags=flags)
    assert np.array_equal(got.view(np.int32), ref.view(np.int32)), \
        f"{H}x{W} l{levels} w{winsize} it{iters} poly {poly_n}/{poly_sigma} init {use_init}: " \
        f"bit-equal {np.mean(got == ref):.5f}"


# 40 x 52 and 9 x 130: smaller than the window in one direction for the large winsizes; 70 x 97: larger in both
@pytest.mark.parametrize("shape", [(40, 52), (9, 130), (70, 97)])
@pytest.mark.parametrize("winsize", range(1, 32))
def test_every_winsize(shape, winsize):
    check(*shape, 3, winsize, seed=winsize)
    if winsize % 2 == 0:     # an even window is not the next odd one: the box mean divides by winsize^2
        check(*shape, 3, winsize, use_init=True, seed=winsize)


@pytest.mark.parametrize("poly_n", range(1, 8))
@pytest.mark.parametrize("poly_sigma", [0.0, 0.6, 1.1, 1.5])
def test_poly_n_and_sigma(poly_n, poly_sigma):
    """poly_sigma 0 is n * 0.3 in cv2's FarnebackPrepareGaussian."""
    check(48, 70, 2, 5, poly_n=poly_n, poly_sigma=poly_sigma, seed=poly_n)


@pytest.mark.parametrize("iters", range(1, 6))
def test_iterations(iters):
    check(66, 130, 3, 9, iters=iters, seed=iters)
    check(33, 64, 1, 4, iters=iters, use_init=True, seed=iters)


@pytest.mark.parametrize("levels", range(0, 6))
def test_levels_on_a_large_image(levels):
    """Levels 4 and 5 of a >= 1024 px image: 39- and 79-tap pyramid blurs, flow resizes by 16 and 32."""
    check(1024, 1036, levels, 5, iters=2, use_init=levels % 2 == 1, seed=levels)


@pytest.mark.parametrize("shape", [(1, 40), (2, 40), (40, 1), (3, 3), (5, 200), (200, 5)])
@pytest.mark.parametrize("winsize", [1, 5, 15, 31])
def test_degenerate_shapes(shape, winsize):
    check(*shape, 3, winsize, seed=7)
    check(*shape, 3, winsize, use_init=True, seed=8)


@pytest.mark.parametrize("W", [7700, 8192, 8200, 12000])
@pytest.mark.parametrize("winsize", [5, 7, 9])
def test_wide_images(W, winsize):
    """Wider than the 64 strips the box kernels once accepted (7424 / 7680 / 8192 px)."""
    check(24, W, 2, winsize, iters=2, seed=W + winsize)
