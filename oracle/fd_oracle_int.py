"""CPU ORACLE of integer volumes -- test infrastructure only, like fd_oracle.py.

The reference keeps an integer volume's dtype through every pass (SURVEY App. B Q3): ``filtered_vol = zeros_like(vol)``
is integer, ``cv2.remap`` of an integer neighbour returns an integer image, ``tmp_slice += warped * kernel[i]``
accumulates in float32 and ``filtered_vol[z] = tmp_slice`` truncates toward zero; the Y and X passes read the truncated
result of the pass before. ``fd_oracle.OracleDenoiser(backend="cv2")`` already does all of that (it keeps
``zeros_like(vol)`` and calls cv2 like the reference). This module adds

  * ctypes bindings of ``oracle/fd_oracle_int.c``: cv2.remap of 8U / 16U / 16S images, restated in C;
  * ``IntegerDenoiser`` / ``IntegerGaussianWindowDenoiser``: the oracle drivers whose C backend warps integer slices
    with that restatement (the flows are the C Farneback of float32(slice), which is what cv2 computes: it converts
    integer images to float32 before the pyramid);
  * the seeded integer test volumes of ``tests/golden/integer_volumes.npz``.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from . import fd_oracle as O
from . import fd_oracle_gw as GW

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libfd_oracle_int.so")
_SOURCE = os.path.join(_HERE, "fd_oracle_int.c")
_CFLAGS = ["-O2", "-ffp-contract=off", "-fPIC", "-shared", "-fvisibility=hidden"]
_lib = None

# FDN_DTYPE_* (include/fdn_b200.h)
DTYPE_CODES = {np.dtype(np.float32): 0, np.dtype(np.uint8): 1, np.dtype(np.int8): 2, np.dtype(np.uint16): 3,
               np.dtype(np.int16): 4}


def build(force: bool = False) -> str:
    """Compile oracle/fd_oracle_int.c -> oracle/libfd_oracle_int.so (gcc)."""
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(_SOURCE):
        subprocess.check_call(["gcc", *_CFLAGS, "-o", _LIB_PATH, _SOURCE, "-lm"], cwd=_HERE)
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB_PATH)
        _lib.fdo_remap_typed.restype = C.c_int
    return _lib


def remap_table_8u() -> np.ndarray:
    """OpenCV's fixed-point bilinear table: (1024, 4) int16, entry (sy & 31) * 32 + (sx & 31)."""
    out = np.empty((1024, 4), np.int16)
    lib().fdo_remap_table_8u(out.ctypes.data_as(C.c_void_p))
    return out


def remap(src, map_xy) -> np.ndarray:
    """cv2.remap(src, map_xy, None, INTER_LINEAR, BORDER_REPLICATE) for uint8 / uint16 / int16 src (H, W) and a
    float32 (H, W, 2) map."""
    src = np.ascontiguousarray(src)
    map_xy = np.ascontiguousarray(map_xy, np.float32)
    H, W = src.shape
    if map_xy.shape != (H, W, 2):
        raise ValueError("map must have shape src.shape + (2,)")
    code = DTYPE_CODES.get(src.dtype)
    out = np.empty_like(src)
    if code is None or lib().fdo_remap_typed(src.ctypes.data_as(C.c_void_p), code, H, W,
                                             map_xy.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p)) != 0:
        raise ValueError(f"cv2.remap does not take {src.dtype} images")
    return out


def warp_slice(reference, flow) -> np.ndarray:
    """src/flowdenoising.py:55-63 for an integer slice, C restatement (same map as the reference builds)."""
    height, width = flow.shape[:2]
    map_x = np.tile(np.arange(width), (height, 1))
    map_y = np.swapaxes(np.tile(np.arange(height), (width, 1)), 0, 1)
    map_xy = (flow + np.dstack((map_x, map_y))).astype("float32")
    return remap(reference, map_xy)


class _IntegerWarp:
    def _warp(self, reference, flow):
        if self.backend == "c" and reference.dtype != np.float32:
            return warp_slice(reference, flow)
        return super()._warp(reference, flow)


class IntegerDenoiser(_IntegerWarp, O.OracleDenoiser):
    """fd_oracle.OracleDenoiser; its C backend warps integer slices in their own type like cv2."""


class IntegerGaussianWindowDenoiser(_IntegerWarp, GW.GaussianWindowDenoiser):
    """fd_oracle_gw.GaussianWindowDenoiser with the integer warp of IntegerDenoiser."""


# ----------------------------------------------------------------------------------------------
# seeded test volumes (tests/golden/integer_volumes.npz stores their seeds and digests only)
# ----------------------------------------------------------------------------------------------
def integer_volume(shape, dtype, seed, noise_sigma=10.0) -> np.ndarray:
    """fd_oracle.synthetic_volume (integers 0..255) mapped onto the dtype:
    uint8 as is; uint16 * 17 + 1000 (1000..5335); int16 * 12 - 1536 (-1536..1524, truncation toward zero of negative
    sums is exercised); int8 - 128 (-128..127)."""
    v = O.synthetic_volume(shape, seed=seed, noise_sigma=noise_sigma).astype(np.int32)
    dtype = np.dtype(dtype)
    if dtype == np.uint8:
        return v.astype(np.uint8)
    if dtype == np.uint16:
        return (v * 17 + 1000).astype(np.uint16)
    if dtype == np.int16:
        return (v * 12 - 1536).astype(np.int16)
    if dtype == np.int8:
        return (v - 128).astype(np.int8)
    raise ValueError(f"no integer test volume of dtype {dtype}")
