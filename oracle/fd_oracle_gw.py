"""CPU ORACLE of the Gaussian window (OPTFLOW_FARNEBACK_GAUSSIAN) -- test infrastructure only, like fd_oracle.py.

ctypes bindings of ``oracle/fd_oracle_gw.c`` (fd_oracle.c plus the Gaussian blur-solve and flag-aware level / pass
drivers) and a variant of ``fd_oracle.OracleDenoiser`` whose cv2 and C backends pass the window flag. Everything else
(stages, synthetic volumes, kernels) is fd_oracle's.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from . import fd_oracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libfd_oracle_gw.so")
_SOURCES = [os.path.join(_HERE, "fd_oracle_gw.c"), os.path.join(_HERE, "fd_oracle.c")]
# the flags of oracle/Makefile (no FMA contraction: OpenCV's scalar code has none here)
_CFLAGS = ["-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", "-fvisibility=hidden", "-Wno-comment"]
_lib = None

USE_INITIAL_FLOW = 4        # cv2.OPTFLOW_USE_INITIAL_FLOW
FARNEBACK_GAUSSIAN = 256    # cv2.OPTFLOW_FARNEBACK_GAUSSIAN


def build(force: bool = False) -> str:
    """Compile oracle/fd_oracle_gw.c -> oracle/libfd_oracle_gw.so (gcc)."""
    if force or not os.path.exists(_LIB_PATH) or \
            os.path.getmtime(_LIB_PATH) < max(os.path.getmtime(s) for s in _SOURCES):
        subprocess.check_call(["gcc", *_CFLAGS, "-o", _LIB_PATH, _SOURCES[0], "-lm"], cwd=_HERE)
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB_PATH)
        _lib.fdo_farneback_gw.restype = C.c_int
    return _lib


def gauss_blur_solve(M, win):
    """FarnebackUpdateFlow_GaussianBlur: separable float32 Gaussian window of M (H, W, 5), then the 2x2 solve."""
    M = O._f32(M)
    H, W = M.shape[:2]
    flow = np.empty((H, W, 2), np.float32)
    lib().fdo_gauss_blur_solve(O._p(M), H, W, int(win), O._p(flow))
    return flow


def farneback_c(prev, nxt, flow, levels=O.OF_LEVELS, winsize=O.OF_WINDOW_SIZE, iters=O.OF_ITERS,
                poly_n=O.OF_POLY_N, poly_sigma=O.OF_POLY_SIGMA, flags=FARNEBACK_GAUSSIAN):
    """cv2.calcOpticalFlowFarneback(prev, next, flow, 0.5, ..., flags) restated; flow updated in place."""
    prev = O._f32(prev); nxt = O._f32(nxt)
    H, W = prev.shape
    if flow is None:
        flow = np.zeros((H, W, 2), np.float32)
    assert flow.dtype == np.float32 and flow.flags.c_contiguous and flow.shape == (H, W, 2)
    lib().fdo_farneback_gw(O._p(prev), O._p(nxt), O._p(flow), H, W, int(levels), int(winsize), int(iters),
                           int(poly_n), C.c_double(poly_sigma), int(flags))
    return flow


def flow_axis_c(vol, axis, kernel, levels=O.OF_LEVELS, winsize=O.OF_WINDOW_SIZE, iters=O.OF_ITERS,
                poly_n=O.OF_POLY_N, poly_sigma=O.OF_POLY_SIGMA, use_prev_flow=True, s0=0, s1=None, out=None,
                flags=FARNEBACK_GAUSSIAN):
    """fd_oracle.flow_axis_c with the window flag (the initial-flow bit follows use_prev_flow)."""
    vol = O._f32(vol)
    if out is None:
        out = np.zeros_like(vol)
    k = np.ascontiguousarray(kernel, np.float64)
    Z, Y, X = vol.shape
    if s1 is None:
        s1 = vol.shape[axis]
    lib().fdo_flow_axis_gw(O._p(vol), O._p(out), Z, Y, X, int(axis), O._p(k, O._f64p), int(k.size), int(levels),
                           int(winsize), int(iters), int(poly_n), C.c_double(poly_sigma), int(bool(use_prev_flow)),
                           int(s0), int(s1), int(flags))
    return out


class GaussianWindowDenoiser(O.OracleDenoiser):
    """fd_oracle.OracleDenoiser with every flow computed with the Gaussian window, on either backend."""

    def _flow(self, reference, target, prev_flow):
        init = 0 if self.recompute_flow else USE_INITIAL_FLOW
        if self.backend == "cv2":
            import cv2
            return cv2.calcOpticalFlowFarneback(prev=target, next=reference, flow=None if init == 0 else prev_flow,
                                                pyr_scale=0.5, levels=self.l, winsize=self.w, iterations=self.iters,
                                                poly_n=self.poly_n, poly_sigma=self.poly_sigma,
                                                flags=init | FARNEBACK_GAUSSIAN)
        return farneback_c(target, reference, None if init == 0 else prev_flow, self.l, self.w, self.iters,
                           self.poly_n, self.poly_sigma, flags=init | FARNEBACK_GAUSSIAN)
