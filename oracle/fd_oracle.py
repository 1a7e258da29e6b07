"""CPU ORACLE -- test infrastructure only (never imported by the product package).

Two layers:

1. ctypes bindings of ``oracle/fd_oracle.c`` (plain-C restatement of the OpenCV / SciPy numerics the
   reference calls; stage-addressable: pyramid level, polyexp, update-matrices, blur-solve, remap).
2. A restatement of the reference's own driver code -- ``GaussianDenoising`` / ``FlowDenoising``
   slice loops of ``/root/reference/src/flowdenoising.py:133-158, 306-373`` and ``filter``
   ``:285-290`` -- with a selectable numerics backend:
     backend="cv2": calls ``cv2.calcOpticalFlowFarneback`` / ``cv2.remap`` exactly like the reference
                    does (``:55-63``, ``:65-114``); cv2 is the reference's real third-party dependency
                    (opencv-python-headless 4.13.0.92 in this image) -- the authoritative arm.
     backend="c"  : uses the C restatement (no cv2 needed).

Parity pinning: the reference ships no golden vectors (SURVEY.md §4). This oracle is pinned against
outputs of the UNMODIFIED reference executed in the build container (``tests/golden/*.npz``, written by
``oracle/gen_golden.py``) and against live cv2 calls (``tests/test_oracle_*.py``).

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference`` legs
may import this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libfd_oracle.so")
_lib = None

# Reference constants (src/flowdenoising.py:47-53)
OF_LEVELS = 3
OF_WINDOW_SIZE = 5
OF_ITERS = 3
OF_POLY_N = 5
OF_POLY_SIGMA = 1.2
SIGMA = 2.0

_f32p = C.POINTER(C.c_float)
_f64p = C.POINTER(C.c_double)
_i32p = C.POINTER(C.c_int)


def build(force: bool = False) -> str:
    """Compile oracle/fd_oracle.c -> oracle/libfd_oracle.so (gcc, see oracle/Makefile)."""
    src = os.path.join(_HERE, "fd_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-B", "libfd_oracle.so"], stdout=subprocess.DEVNULL)
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB_PATH)
        _lib.fdo_level_geometry.restype = C.c_int
        _lib.fdo_farneback.restype = C.c_int
    return _lib


def _p(a, t=_f32p):
    return a.ctypes.data_as(t)


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


# ----------------------------------------------------------------------------------------------
# Layer 1: C restatement, stage by stage
# ----------------------------------------------------------------------------------------------
def gauss_blur(img, ksz, sigma):
    img = _f32(img)
    out = np.empty_like(img)
    lib().fdo_gauss_blur(_p(img), img.shape[0], img.shape[1], int(ksz), C.c_double(sigma), _p(out))
    return out


def resize_linear(img, h, w, ipp=None):
    """cv2.resize INTER_LINEAR; ipp=None picks what cv2 itself uses (IPP for 1 channel, native for 2)."""
    img = _f32(img)
    if ipp is None:
        ipp = img.ndim == 2
    cn = 1 if img.ndim == 2 else img.shape[2]
    out = np.empty((h, w) if img.ndim == 2 else (h, w, cn), np.float32)
    lib().fdo_resize_linear(_p(img), img.shape[0], img.shape[1], cn, _p(out), h, w, int(bool(ipp)))
    return out


def resize_area(img, h, w):
    img = _f32(img)
    cn = 1 if img.ndim == 2 else img.shape[2]
    out = np.empty((h, w) if img.ndim == 2 else (h, w, cn), np.float32)
    lib().fdo_resize_area(_p(img), img.shape[0], img.shape[1], cn, _p(out), h, w)
    return out


def level_geometry(H, W, levels):
    """Returns list of (h, w, ksz, sigma) for k = 0..n_extra_levels (SURVEY App. A.0)."""
    hs = np.zeros(32, np.int32); ws = np.zeros(32, np.int32); ks = np.zeros(32, np.int32)
    sg = np.zeros(32, np.float64)
    nl = lib().fdo_level_geometry(H, W, int(min(levels, 30)), _p(hs, _i32p), _p(ws, _i32p), _p(ks, _i32p),
                                  _p(sg, _f64p))
    return [(int(hs[k]), int(ws[k]), int(ks[k]), float(sg[k])) for k in range(nl + 1)]


def pyramid_level(img, ksz, sigma, h, w):
    img = _f32(img)
    out = np.empty((h, w), np.float32)
    lib().fdo_pyramid_level(_p(img), img.shape[0], img.shape[1], int(ksz), C.c_double(sigma), h, w, _p(out))
    return out


def polyexp_consts(n=OF_POLY_N, sigma=OF_POLY_SIGMA):
    g = np.zeros(n + 1, np.float32); xg = np.zeros(n + 1, np.float32); xxg = np.zeros(n + 1, np.float32)
    ig = np.zeros(4, np.float64)
    lib().fdo_polyexp_consts(int(n), C.c_double(sigma), _p(g), _p(xg), _p(xxg), _p(ig, _f64p))
    return g, xg, xxg, ig


def polyexp(img, n=OF_POLY_N, sigma=OF_POLY_SIGMA):
    """(H, W) -> R (H, W, 5)  (SURVEY App. A.2)."""
    img = _f32(img)
    out = np.empty(img.shape + (5,), np.float32)
    lib().fdo_polyexp(_p(img), img.shape[0], img.shape[1], int(n), C.c_double(sigma), _p(out))
    return out


def update_matrices(R0, R1, flow):
    R0 = _f32(R0); R1 = _f32(R1); flow = _f32(flow)
    H, W = flow.shape[:2]
    M = np.empty((H, W, 5), np.float32)
    lib().fdo_update_matrices(_p(R0), _p(R1), _p(flow), H, W, _p(M), 0, H)
    return M


def blur_solve(M, win):
    M = _f32(M)
    H, W = M.shape[:2]
    flow = np.empty((H, W, 2), np.float32)
    lib().fdo_blur_solve(_p(M), H, W, int(win), _p(flow))
    return flow


def farneback_c(prev, nxt, flow, levels=OF_LEVELS, winsize=OF_WINDOW_SIZE, iters=OF_ITERS,
                poly_n=OF_POLY_N, poly_sigma=OF_POLY_SIGMA, flags=0):
    """C restatement of cv2.calcOpticalFlowFarneback(prev, next, flow, 0.5, ...). flow updated in place."""
    prev = _f32(prev); nxt = _f32(nxt)
    H, W = prev.shape
    if flow is None:
        flow = np.zeros((H, W, 2), np.float32)
    assert flow.dtype == np.float32 and flow.flags.c_contiguous and flow.shape == (H, W, 2)
    lib().fdo_farneback(_p(prev), _p(nxt), _p(flow), H, W, int(levels), int(winsize), int(iters), int(poly_n),
                        C.c_double(poly_sigma), int(flags))
    return flow


def warp_slice_c(reference, flow):
    reference = _f32(reference); flow = _f32(flow)
    H, W = reference.shape
    out = np.empty((H, W), np.float32)
    lib().fdo_warp_slice(_p(reference), H, W, _p(flow), _p(out))
    return out


def gauss_axis_c(vol, axis, kernel):
    """a5, whole pass, C (OpenMP)."""
    vol = _f32(vol)
    out = np.empty_like(vol)
    k = np.ascontiguousarray(kernel, np.float64)
    Z, Y, X = vol.shape
    lib().fdo_gauss_axis(_p(vol), _p(out), Z, Y, X, int(axis), _p(k, _f64p), int(k.size))
    return out


def flow_axis_c(vol, axis, kernel, levels=OF_LEVELS, winsize=OF_WINDOW_SIZE, iters=OF_ITERS,
                poly_n=OF_POLY_N, poly_sigma=OF_POLY_SIGMA, use_prev_flow=True, s0=0, s1=None, out=None):
    """a6, whole pass (or slices [s0, s1)), C restatement end to end (OpenMP over slices)."""
    vol = _f32(vol)
    if out is None:
        out = np.zeros_like(vol)
    k = np.ascontiguousarray(kernel, np.float64)
    Z, Y, X = vol.shape
    if s1 is None:
        s1 = vol.shape[axis]
    lib().fdo_flow_axis(_p(vol), _p(out), Z, Y, X, int(axis), _p(k, _f64p), int(k.size), int(levels),
                        int(winsize), int(iters), int(poly_n), C.c_double(poly_sigma), int(bool(use_prev_flow)),
                        int(s0), int(s1))
    return out


# ----------------------------------------------------------------------------------------------
# Layer 2: the reference's driver, restated (cv2 backend = what the reference executes)
# ----------------------------------------------------------------------------------------------
def get_gaussian_kernel(sigma=1.0):
    """src/flowdenoising.py:34-45, the reference's own loop: grow a delta until scipy.ndimage.gaussian_filter1d
    leaves at least two exact zeros, return the response without its two ends (SciPy's kernel, computed by SciPy)."""
    import scipy.ndimage
    number_of_coeffs = 3
    number_of_zeros = 0
    while number_of_zeros < 2:
        delta = np.zeros(number_of_coeffs)
        delta[delta.size // 2] = 1
        coeffs = scipy.ndimage.gaussian_filter1d(delta, sigma=sigma)
        number_of_zeros = coeffs.size - np.count_nonzero(coeffs)
        number_of_coeffs += 1
    return coeffs[1:-1]


def warp_slice(reference, flow):
    """src/flowdenoising.py:55-63."""
    import cv2
    height, width = flow.shape[:2]
    map_x = np.tile(np.arange(width), (height, 1))
    map_y = np.swapaxes(np.tile(np.arange(height), (width, 1)), 0, 1)
    map_xy = (flow + np.dstack((map_x, map_y))).astype("float32")
    return cv2.remap(reference, map_xy, None, interpolation=cv2.INTER_LINEAR, borderMode=cv2.BORDER_REPLICATE)


def get_flow_with_prev_flow(reference, target, l=OF_LEVELS, w=OF_WINDOW_SIZE, prev_flow=None,
                            iters=OF_ITERS, poly_n=OF_POLY_N, poly_sigma=OF_POLY_SIGMA):
    """src/flowdenoising.py:65-87."""
    import cv2
    return cv2.calcOpticalFlowFarneback(prev=target, next=reference, flow=prev_flow, pyr_scale=0.5, levels=l,
                                        winsize=w, iterations=iters, poly_n=poly_n, poly_sigma=poly_sigma,
                                        flags=cv2.OPTFLOW_USE_INITIAL_FLOW)


def get_flow_without_prev_flow(reference, target, l=OF_LEVELS, w=OF_WINDOW_SIZE, prev_flow=None,
                               iters=OF_ITERS, poly_n=OF_POLY_N, poly_sigma=OF_POLY_SIGMA):
    """src/flowdenoising.py:89-114."""
    import cv2
    return cv2.calcOpticalFlowFarneback(prev=target, next=reference, flow=None, pyr_scale=0.5, levels=l,
                                        winsize=w, iterations=iters, poly_n=poly_n, poly_sigma=poly_sigma, flags=0)


def _slice_view(vol, axis, idx):
    if axis == 0:
        return vol[idx, :, :]
    if axis == 1:
        return vol[:, idx, :]
    return vol[:, :, idx]


class OracleDenoiser:
    """Restatement of GaussianDenoising (:116-295) and FlowDenoising (:297-373) of the reference.

    ``filter(kernels)`` follows :285-290: Z pass, copy back into vol, Y pass, copy back, X pass; the ZYX
    result is ``filtered_vol`` and ``vol`` ends up holding the ZY intermediate (SURVEY App. B Q1).
    """

    def __init__(self, number_of_processes, vol, use_OF=True, l=OF_LEVELS, w=OF_WINDOW_SIZE,
                 iters=OF_ITERS, poly_n=OF_POLY_N, poly_sigma=OF_POLY_SIGMA, recompute_flow=False,
                 backend="cv2"):
        self.number_of_processes = max(1, int(number_of_processes))
        self.vol = vol
        self.filtered_vol = np.zeros_like(vol)
        self.use_OF = use_OF
        self.l, self.w, self.iters, self.poly_n, self.poly_sigma = l, w, iters, poly_n, poly_sigma
        self.recompute_flow = recompute_flow
        self.backend = backend

    # -- numerics seam (reference: injected get_flow / warp_slice callables, :299-304) --
    def _flow(self, reference, target, prev_flow):
        if self.backend == "cv2":
            f = get_flow_without_prev_flow if self.recompute_flow else get_flow_with_prev_flow
            return f(reference, target, self.l, self.w, prev_flow, self.iters, self.poly_n, self.poly_sigma)
        if self.recompute_flow:
            return farneback_c(target, reference, None, self.l, self.w, self.iters, self.poly_n,
                               self.poly_sigma, flags=0)
        return farneback_c(target, reference, prev_flow, self.l, self.w, self.iters, self.poly_n,
                           self.poly_sigma, flags=4)

    def _warp(self, reference, flow):
        if self.backend == "cv2":
            return warp_slice(reference, flow)
        return warp_slice_c(reference, flow)

    # -- per-slice filters --
    def filter_slice(self, axis, idx, kernel):
        vol = self.vol
        n = vol.shape[axis]
        ks2 = kernel.size // 2
        centre = _slice_view(vol, axis, idx)
        tmp_slice = np.zeros(centre.shape, dtype=np.float32)
        if not self.use_OF:
            # :133-158
            for i in range(kernel.size):
                tmp_slice += _slice_view(vol, axis, (idx + i - ks2) % n) * kernel[i]
        else:
            # :306-373
            assert kernel.size % 2 != 0
            prev_flow = np.zeros(centre.shape + (2,), dtype=np.float32)
            for i in range(ks2 - 1, -1, -1):
                neigh = _slice_view(vol, axis, (idx + i - ks2) % n)
                flow = self._flow(neigh, centre, prev_flow)
                prev_flow = flow
                tmp_slice += self._warp(neigh, flow) * kernel[i]
            tmp_slice += centre * kernel[ks2]
            prev_flow = np.zeros(centre.shape + (2,), dtype=np.float32)
            for i in range(ks2 + 1, kernel.size):
                neigh = _slice_view(vol, axis, (idx + i - ks2) % n)
                flow = self._flow(neigh, centre, prev_flow)
                prev_flow = flow
                tmp_slice += self._warp(neigh, flow) * kernel[i]
        if axis == 0:
            self.filtered_vol[idx, :, :] = tmp_slice
        elif axis == 1:
            self.filtered_vol[:, idx, :] = tmp_slice
        else:
            self.filtered_vol[:, :, idx] = tmp_slice

    def filter_along_axis(self, axis, kernel, indices=None):
        """:175-283 -- slices of a pass are independent; spread over a thread pool (:187-206)."""
        kernel = np.asarray(kernel, np.float64)
        idxs = list(range(self.vol.shape[axis])) if indices is None else list(indices)
        if self.number_of_processes == 1:
            for i in idxs:
                self.filter_slice(axis, i, kernel)
        else:
            with ThreadPoolExecutor(max_workers=self.number_of_processes) as ex:
                list(ex.map(lambda i: self.filter_slice(axis, i, kernel), idxs))

    def filter_along_Z(self, kernel): self.filter_along_axis(0, kernel)
    def filter_along_Y(self, kernel): self.filter_along_axis(1, kernel)
    def filter_along_X(self, kernel): self.filter_along_axis(2, kernel)

    def filter(self, kernels):
        self.filter_along_Z(kernels[0])
        self.vol[...] = self.filtered_vol[...]
        self.filter_along_Y(kernels[1])
        self.vol[...] = self.filtered_vol[...]
        self.filter_along_X(kernels[2])
        return self.filtered_vol


# ----------------------------------------------------------------------------------------------
# Synthetic volumes (SURVEY §8d: 8-bit-like amplitude or the flows collapse to zero)
# ----------------------------------------------------------------------------------------------
def synthetic_volume(shape, seed=0, noise_sigma=10.0, dtype=np.float32, quantise=True, chunk=32):
    """Smooth drifting structure + blobs + Gaussian noise, clipped to [0, 255] (SURVEY §8d).

    Computed in float64 and (by default) rounded to integers 0..255, so the volume is bit-reproducible on
    any host (no dependence on libm / SIMD ulps) -- the golden fixtures store only its SHA-256.
    """
    Z, Y, X = shape
    rng = np.random.default_rng(seed)
    nb = int(min(64, max(4, (Z * Y * X) // 60000)))
    cz = rng.uniform(0, Z, nb); cy = rng.uniform(0, Y, nb); cx = rng.uniform(0, X, nb)
    rad = rng.uniform(3.0, 9.0, nb); amp = rng.uniform(-70, 70, nb)
    drift = rng.uniform(-1.2, 1.2, (nb, 2))
    out = np.empty(shape, dtype)
    y = np.arange(Y, dtype=np.float64)[None, :, None]
    x = np.arange(X, dtype=np.float64)[None, None, :]
    for z0 in range(0, Z, chunk):
        z1 = min(Z, z0 + chunk)
        z = np.arange(z0, z1, dtype=np.float64)[:, None, None]
        v = 128.0 + 60.0 * np.sin(x / 9.0 + z / 13.0) * np.cos(y / 7.0 - z / 17.0) + 30.0 * np.sin((x + y) / 23.0)
        for b in range(nb):
            zz = np.arange(z0, z1, dtype=np.float64)
            dzv = zz - cz[b]
            sel = np.nonzero(np.abs(dzv) < 8 * rad[b])[0]      # exp(-(8/2)^2/2) ~ 3e-4 relative cut-off
            if sel.size == 0:
                continue
            R = 4 * rad[b] + 1.2 * 8 * rad[b]
            ya, yb = int(max(0, cy[b] - R)), int(min(Y, cy[b] + R + 1))
            xa, xb = int(max(0, cx[b] - R)), int(min(X, cx[b] + R + 1))
            if ya >= yb or xa >= xb:
                continue
            dz = dzv[sel][:, None, None]
            yy = np.arange(ya, yb, dtype=np.float64)[None, :, None]
            xx = np.arange(xa, xb, dtype=np.float64)[None, None, :]
            d2 = (dz / 2.0) ** 2 + (yy - cy[b] - drift[b, 0] * dz) ** 2 + (xx - cx[b] - drift[b, 1] * dz) ** 2
            v[sel[0]:sel[-1] + 1, ya:yb, xa:xb] += amp[b] * np.exp(-d2 / (2.0 * rad[b] ** 2))
        if noise_sigma > 0:
            v = v + rng.normal(0.0, noise_sigma, size=v.shape)
        v = np.clip(v, 0, 255)
        if quantise or np.issubdtype(np.dtype(dtype), np.integer):
            v = np.rint(v)
        out[z0:z1] = v.astype(dtype)
    return out
