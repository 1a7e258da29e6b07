"""ctypes binding of libfdn_b200.so (C ABI declared in include/fdn_b200.h).

There is NO CPU fallback: if the CUDA library cannot be loaded, or no CUDA device is present, every compute
entry point raises. PyTorch is used by callers only to own device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os

from . import _build

_lib = None

c_f32p = C.c_void_p      # device pointers travel as plain addresses
c_i64 = C.c_int64


class OfParams(C.Structure):
    """struct fdn_of_params (reference constants: src/flowdenoising.py:47-53)."""
    _fields_ = [("levels", C.c_int), ("winsize", C.c_int), ("iterations", C.c_int), ("poly_n", C.c_int),
                ("poly_sigma", C.c_double), ("use_prev_flow", C.c_int), ("flags", C.c_int)]


FARNEBACK_GAUSSIAN = 256   # FDN_OF_FARNEBACK_GAUSSIAN (= cv2.OPTFLOW_FARNEBACK_GAUSSIAN)

# FDN_DTYPE_*: element types of typed volumes (the reference's integer semantics, opt-in)
DTYPE_F32, DTYPE_U8, DTYPE_I8, DTYPE_U16, DTYPE_I16 = 0, 1, 2, 3, 4

# FDN_BORDER_*: the border along a pass's axis (fdn_view.periodic, fdn_gauss_rows_border)
BORDER_WRAP, BORDER_REFLECT, BORDER_MIRROR, BORDER_NEAREST = 1, 2, 3, 4


class View(C.Structure):
    """struct fdn_view."""
    _fields_ = [("n_in", C.c_int), ("n_out", C.c_int), ("halo", C.c_int), ("periodic", C.c_int),
                ("H", C.c_int), ("W", C.c_int),
                ("in_slice_stride", c_i64), ("in_row_stride", c_i64),
                ("out_slice_stride", c_i64), ("out_row_stride", c_i64)]


# name -> (restype, argtypes); every symbol of include/fdn_b200.h
SIGNATURES = {
    "fdn_version": (C.c_int, []),
    "fdn_last_error": (C.c_char_p, []),
    "fdn_launch_count": (c_i64, []),
    "fdn_reset_launch_count": (None, []),
    "fdn_launch_log_enable": (None, [C.c_int]),
    "fdn_launch_log_count": (C.c_int, []),
    "fdn_launch_log_name": (C.c_char_p, [C.c_int]),
    "fdn_progress_milli": (c_i64, []),
    "fdn_progress_reset": (None, []),
    "fdn_profile_enable": (None, [C.c_int]),
    "fdn_profile_reset": (None, []),
    "fdn_profile_kernel_count": (C.c_int, []),
    "fdn_profile_kernel_name": (C.c_char_p, [C.c_int]),
    "fdn_profile_read": (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(c_i64), C.POINTER(C.c_double)]),
    "fdn_profile_record_count": (C.c_int, []),
    "fdn_profile_record": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                     C.POINTER(C.c_int), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "fdn_gaussian_kernel": (C.c_int, [C.c_double, C.POINTER(C.c_double), C.c_int]),
    "fdn_level_geometry": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                     C.POINTER(C.c_int), C.POINTER(C.c_double)]),
    "fdn_workspace_bytes": (C.c_size_t, [C.POINTER(View), C.c_int, C.POINTER(OfParams), C.c_int]),
    "fdn_filter_axis": (C.c_int, [c_f32p, c_f32p, C.POINTER(View), C.POINTER(C.c_double), C.c_int,
                                  C.POINTER(OfParams), C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "fdn_gauss_axis": (C.c_int, [c_f32p, c_f32p, C.POINTER(View), C.POINTER(C.c_double), C.c_int, C.c_int,
                                 C.c_void_p]),
    "fdn_gauss_rows": (C.c_int, [c_f32p, c_f32p, c_i64, C.c_int, C.POINTER(C.c_double), C.c_int, C.c_int,
                                 C.c_void_p]),
    "fdn_transpose_yx": (C.c_int, [c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "fdn_workspace_bytes_batch": (C.c_size_t, [C.POINTER(View), C.c_int, C.c_int, C.POINTER(OfParams)]),
    "fdn_filter_axis_batch": (C.c_int, [c_f32p, c_f32p, C.POINTER(View), C.c_int, c_i64, c_i64, C.POINTER(C.c_double),
                                        C.c_int, C.POINTER(OfParams), C.c_void_p, C.c_size_t, C.c_void_p]),
    "fdn_gauss_axis_batch": (C.c_int, [c_f32p, c_f32p, C.POINTER(View), C.c_int, c_i64, c_i64, C.POINTER(C.c_double),
                                       C.c_int, C.c_int, C.c_void_p]),
    "fdn_transpose_strided": (C.c_int, [c_f32p, c_i64, c_i64, c_f32p, c_i64, c_i64, C.c_int, C.c_int, C.c_int,
                                        C.c_void_p]),
    "fdn_copy3d": (C.c_int, [c_f32p, c_i64, c_i64, C.c_int, C.c_int, C.c_int, C.c_int, c_f32p, c_i64, c_i64, C.c_int,
                             C.c_int, C.c_int, C.c_void_p]),
    "fdn_copy2d_async": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int,
                                   C.c_void_p]),
    "fdn_pyramid_level": (C.c_int, [c_f32p, C.c_int, C.c_int, C.c_int, c_i64, c_i64, C.c_int, C.c_double, C.c_int,
                                    C.c_int, c_f32p, c_f32p, C.c_void_p]),
    "fdn_polyexp": (C.c_int, [c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, c_f32p, C.c_void_p]),
    "fdn_polyexp_floats": (C.c_size_t, [C.c_int, C.c_int]),
    "fdn_flow_iteration_scratch_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "fdn_flow_iteration": (C.c_int, [c_f32p, c_f32p, c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_void_p, C.c_size_t, C.c_void_p]),
    "fdn_flow_iterations": (C.c_int, [c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.POINTER(C.c_void_p)]),
    "fdn_flow_iterations_gaussian": (C.c_int, [c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, C.c_int, C.c_int, C.c_int,
                                               C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "fdn_set_flow_iter_variant": (None, [C.c_int]),
    "fdn_flow_area_down": (C.c_int, [c_f32p, C.c_int, C.c_int, C.c_int, c_f32p, C.c_int, C.c_int, C.c_float,
                                     C.c_void_p]),
    "fdn_flow_upsample": (C.c_int, [c_f32p, C.c_int, C.c_int, C.c_int, c_f32p, C.c_int, C.c_int, C.c_void_p]),
    "fdn_farneback_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.POINTER(OfParams)]),
    "fdn_farneback": (C.c_int, [c_f32p, c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, C.POINTER(OfParams), C.c_void_p,
                                C.c_size_t, C.c_void_p]),
    "fdn_workspace_bytes_typed": (C.c_size_t, [C.POINTER(View), C.c_int, C.POINTER(OfParams), C.c_int, C.c_int]),
    "fdn_filter_axis_typed": (C.c_int, [c_f32p, c_f32p, C.c_int, C.POINTER(View), C.POINTER(C.c_double), C.c_int,
                                        C.POINTER(OfParams), C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]),
    "fdn_gauss_axis_typed": (C.c_int, [c_f32p, c_f32p, C.c_int, C.POINTER(View), C.POINTER(C.c_double), C.c_int,
                                       C.c_int, C.c_void_p]),
    "fdn_gauss_rows_typed": (C.c_int, [c_f32p, c_f32p, C.c_int, c_i64, C.c_int, C.POINTER(C.c_double), C.c_int,
                                       C.c_int, C.c_void_p]),
    "fdn_gauss_rows_border": (C.c_int, [c_f32p, c_f32p, C.c_int, c_i64, C.c_int, C.POINTER(C.c_double), C.c_int,
                                        C.c_int, C.c_int, C.c_void_p]),
    "fdn_transpose_yx_typed": (C.c_int, [c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "fdn_remap_typed": (C.c_int, [c_f32p, c_f32p, c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "fdn_transpose_strided_typed": (C.c_int, [c_f32p, C.c_int, c_i64, c_i64, c_f32p, c_i64, c_i64, C.c_int, C.c_int,
                                              C.c_int, C.c_void_p]),
    "fdn_copy3d_typed": (C.c_int, [c_f32p, C.c_int, c_i64, c_i64, C.c_int, C.c_int, C.c_int, C.c_int, c_f32p, c_i64,
                                   c_i64, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "fdn_warp_accumulate": (C.c_int, [c_f32p, c_i64, c_i64, c_f32p, C.c_double, c_f32p, c_i64, c_i64, C.c_int,
                                      C.c_int, C.c_int, C.c_void_p]),
}


class FdnError(RuntimeError):
    pass


def lib_path() -> str:
    return _build.LIB


def load():
    """Load (building first if the sources are newer) libfdn_b200.so. Raises if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("FDN_LIB_PATH")   # development: a build variant (tools/build_variant.py)
    lab = path is not None
    if not lab:
        path = _build.LIB
        if _build.needs_build():
            try:
                _build.build_locked()
            except Exception as e:  # no nvcc, compile error ...
                if not os.path.exists(path):
                    raise FdnError(f"libfdn_b200.so is missing and could not be built ({e}); there is no CPU "
                                   f"fallback. Run `python -m flowdenoising_b200._build`.") from e
                # a stale library must never be used silently: its ABI or numerics may not match the sources
                raise FdnError(f"libfdn_b200.so is older than its sources and the rebuild failed ({e})") from e
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name, None)
        if fn is None:
            if lab:
                continue   # an older build variant under comparison
            raise AttributeError(f"{name} is declared in include/fdn_b200.h but not exported by {path}")
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        msg = load().fdn_last_error().decode("utf-8", "replace")
        raise (ValueError if rc == 1 else FdnError)(f"libfdn_b200: {msg} (status {rc})")


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise FdnError("flowdenoising_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch
