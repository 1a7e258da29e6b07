"""Device-side pass engine: thin Python over the C ABI (include/fdn_b200.h).

PyTorch tensors own every device buffer (volume, output, workspace); the C library only receives raw pointers.
Nothing here computes on the CPU.

Mirrors the reference's pass driver `GaussianDenoising.filter` / `filter_along_{Z,Y,X}`
(/root/reference/src/flowdenoising.py:175-290) for a device-resident float32 volume [Z, Y, X]. A uint8, int8, uint16 or
int16 volume runs the reference's integer semantics in its own dtype (typed passes, fdn_*_typed: integer remap,
float32 accumulation, truncating store); int8 without optical flow only, like cv2.remap.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from . import _lib
from ._lib import FARNEBACK_GAUSSIAN, OfParams, View

# reference defaults, src/flowdenoising.py:47-53
OF_LEVELS = 3
OF_WINDOW_SIZE = 5
OF_ITERS = 3
OF_POLY_N = 5
OF_POLY_SIGMA = 1.2
SIGMA = 2.0


@dataclass
class FlowParams:
    levels: int = OF_LEVELS
    winsize: int = OF_WINDOW_SIZE
    iterations: int = OF_ITERS
    poly_n: int = OF_POLY_N
    poly_sigma: float = OF_POLY_SIGMA
    use_prev_flow: bool = True
    # OPTFLOW_FARNEBACK_GAUSSIAN: Gaussian window instead of the box mean (a different flow estimate)
    gaussian_window: bool = False

    def c_struct(self) -> OfParams:
        return OfParams(int(self.levels), int(self.winsize), int(self.iterations), int(self.poly_n),
                        float(self.poly_sigma), int(bool(self.use_prev_flow)),
                        FARNEBACK_GAUSSIAN if self.gaussian_window else 0)


def gaussian_kernel(sigma: float) -> np.ndarray:
    """get_gaussian_kernel (src/flowdenoising.py:34-45): float64 taps, length 2*int(4*sigma+0.5)+1."""
    lib = _lib.load()
    buf = (C.c_double * 4096)()
    n = lib.fdn_gaussian_kernel(float(sigma), buf, 4096)
    if n <= 0:
        raise ValueError(f"cannot build a Gaussian kernel for sigma={sigma}")
    return np.frombuffer(buf, dtype=np.float64, count=n).copy()


def level_geometry(H: int, W: int, levels: int):
    lib = _lib.load()
    hs = (C.c_int * 32)(); ws = (C.c_int * 32)(); ks = (C.c_int * 32)(); sg = (C.c_double * 32)()
    nl = lib.fdn_level_geometry(H, W, levels, hs, ws, ks, sg)
    return [(hs[k], ws[k], ks[k], sg[k]) for k in range(nl + 1)]


def _taps(kernel) -> tuple:
    k = np.ascontiguousarray(kernel, dtype=np.float64)
    if k.ndim != 1 or k.size % 2 == 0:
        raise ValueError("kernel.size must be odd")  # src/flowdenoising.py:309
    return k, k.ctypes.data_as(C.POINTER(C.c_double))


def _stream_ptr(torch):
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def dtype_code(t) -> int:
    """FDN_DTYPE_* of a tensor's dtype (ValueError for any other dtype)."""
    import torch
    codes = {torch.float32: _lib.DTYPE_F32, torch.uint8: _lib.DTYPE_U8, torch.int8: _lib.DTYPE_I8,
             torch.uint16: _lib.DTYPE_U16, torch.int16: _lib.DTYPE_I16}
    if t.dtype not in codes:
        raise ValueError(f"unsupported volume dtype {t.dtype} (float32, uint8, int8, uint16 or int16)")
    return codes[t.dtype]


class DeviceEngine:
    """Runs passes on device-resident float32 volumes. One engine per GPU / process."""

    def __init__(self, device=None, workspace_limit_bytes: Optional[int] = None):
        self.torch = _lib.require_cuda()
        self.lib = _lib.load()
        torch = self.torch
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.workspace_limit_bytes = workspace_limit_bytes
        self._ws = None

    # ---- workspace ----
    def _workspace(self, nbytes: int):
        torch = self.torch
        if self._ws is None or self._ws.numel() < nbytes:
            self._ws = None
            self._ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=self.device)
        return self._ws

    def release_workspace(self):
        self._ws = None

    def _workspace_bytes(self, view: View, klen: int, ofp: OfParams, chunk: int, dtype: int) -> int:
        if dtype == _lib.DTYPE_F32:
            return self.lib.fdn_workspace_bytes(C.byref(view), klen, C.byref(ofp), chunk)
        return self.lib.fdn_workspace_bytes_typed(C.byref(view), klen, C.byref(ofp), chunk, dtype)

    def _pick_chunk(self, view: View, klen: int, ofp: OfParams, dtype: int = _lib.DTYPE_F32) -> int:
        """Largest chunk of output slices whose workspace fits the limit (default: 85 % of free HBM)."""
        torch = self.torch
        need = lambda c: self._workspace_bytes(view, klen, ofp, c, dtype)
        full = need(view.n_out)
        if full == 0:
            _lib.check(1)
        limit = self.workspace_limit_bytes
        if limit is None:
            have = self._ws.numel() if self._ws is not None else 0
            if full <= have:
                # the workspace this engine already holds is enough: no driver query (cudaMemGetInfo blocks for
                # milliseconds while a large host <-> device copy is in flight, tools/host_stall_lab.py)
                return view.n_out
            free, _total = torch.cuda.mem_get_info(self.device)
            limit = int((free + have) * 0.85)
        if full <= limit:
            return view.n_out
        lo, hi = 1, view.n_out
        if need(1) > limit:
            raise _lib.FdnError(f"not enough device memory for a single-slice chunk ({need(1)} bytes needed)")
        while lo < hi:
            mid = (lo + hi + 1) // 2
            if need(mid) <= limit:
                lo = mid
            else:
                hi = mid - 1
        return lo

    def reserve_workspace(self, view: View, klen: int, flow: Optional[FlowParams]):
        """Sizes the workspace for a later filter_view(view) now, so that a smaller call issued first (the head of a
        pass that overlaps the upload) does not allocate a workspace the next call has to replace."""
        if flow is None:
            return
        with self.torch.cuda.device(self.device):
            ofp = flow.c_struct()
            chunk = self._pick_chunk(view, klen, ofp)
            nbytes = self.lib.fdn_workspace_bytes(C.byref(view), klen, C.byref(ofp), int(chunk))
            if nbytes == 0:
                _lib.check(1)
            self._workspace(nbytes)

    # ---- one pass over an explicit view ----
    def filter_view(self, d_in, d_out, view: View, kernel, flow: Optional[FlowParams], chunk: Optional[int] = None,
                    exact: bool = True):
        """out[s] = sum_i k[i] * warp(in[s+halo+i-r]) for the slices of `view` (see fdn_view). Integer tensors run the
        typed pass (exact arithmetic only)."""
        torch = self.torch
        k, kp = _taps(kernel)
        if d_in.dtype != torch.float32:
            return self._filter_view_typed(d_in, d_out, view, k, kp, flow, chunk, exact)
        with torch.cuda.device(self.device):
            if flow is None:
                _lib.check(self.lib.fdn_gauss_axis(d_in.data_ptr(), d_out.data_ptr(), C.byref(view), kp, k.size,
                                                   int(bool(exact)), _stream_ptr(torch)))
                return
            ofp = flow.c_struct()
            if chunk is None:
                chunk = self._pick_chunk(view, k.size, ofp)
            nbytes = self.lib.fdn_workspace_bytes(C.byref(view), k.size, C.byref(ofp), int(chunk))
            if nbytes == 0:
                _lib.check(1)
            ws = self._workspace(nbytes)
            _lib.check(self.lib.fdn_filter_axis(d_in.data_ptr(), d_out.data_ptr(), C.byref(view), kp, k.size,
                                                C.byref(ofp), int(chunk), ws.data_ptr(), ws.numel(),
                                                _stream_ptr(torch)))

    def _filter_view_typed(self, d_in, d_out, view: View, k, kp, flow: Optional[FlowParams], chunk, exact):
        torch = self.torch
        dt = dtype_code(d_in)
        if d_out.dtype != d_in.dtype:
            raise ValueError("a typed pass writes the dtype it reads")
        with torch.cuda.device(self.device):
            if flow is None:
                _lib.check(self.lib.fdn_gauss_axis_typed(d_in.data_ptr(), d_out.data_ptr(), dt, C.byref(view), kp,
                                                         k.size, int(bool(exact)), _stream_ptr(torch)))
                return
            ofp = flow.c_struct()
            if chunk is None:
                chunk = self._pick_chunk(view, k.size, ofp, dt)
            nbytes = self._workspace_bytes(view, k.size, ofp, int(chunk), dt)
            if nbytes == 0:
                _lib.check(1)
            ws = self._workspace(nbytes)
            _lib.check(self.lib.fdn_filter_axis_typed(d_in.data_ptr(), d_out.data_ptr(), dt, C.byref(view), kp,
                                                      k.size, C.byref(ofp), int(chunk), ws.data_ptr(), ws.numel(),
                                                      _stream_ptr(torch)))

    # ---- passes over a dense [Z, Y, X] volume (single GPU, periodic along the filtered axis) ----
    def _check_vol(self, t):
        torch = self.torch
        if not (t.is_cuda and t.dim() == 3 and t.is_contiguous()):
            raise ValueError("expected a contiguous CUDA tensor [Z, Y, X]")
        if t.dtype != torch.float32:
            dtype_code(t)

    def transpose_yx(self, src, dst=None):
        """[n, A, B] -> [n, B, A] with the library's transpose kernel (any dtype of a typed volume)."""
        torch = self.torch
        n, A, B = src.shape
        if dst is None:
            dst = torch.empty((n, B, A), dtype=src.dtype, device=src.device)
        with torch.cuda.device(self.device):
            if src.dtype == torch.float32:
                _lib.check(self.lib.fdn_transpose_yx(src.data_ptr(), dst.data_ptr(), n, A, B, _stream_ptr(torch)))
            else:
                if dst.dtype != src.dtype:
                    raise ValueError("transpose_yx keeps the dtype")
                _lib.check(self.lib.fdn_transpose_yx_typed(src.data_ptr(), dst.data_ptr(), dtype_code(src), n, A, B,
                                                           _stream_ptr(torch)))
        return dst

    def empty(self, shape, dtype=None):
        dtype = self.torch.float32 if dtype is None else dtype
        return self.torch.empty(tuple(int(s) for s in shape), dtype=dtype, device=self.device)

    @staticmethod
    def _same_dtype(src, dst, what):
        if dst.dtype != src.dtype:
            raise ValueError(f"{what} keeps the dtype ({src.dtype} -> {dst.dtype})")

    def copy3d(self, src, src_off, in_sa, in_sb, b0, bw, c0, cw, dst, dst_off, out_sa, out_sb, A, B, C):
        """dst[a*out_sa + b*out_sb + c] = src[a*in_sa + ((b0+b) % bw)*in_sb + (c0+c) % cw]  (element offsets/strides
        into flat buffers of one dtype) -- the packing kernel of the multi-GPU re-slab."""
        torch = self.torch
        self._same_dtype(src, dst, "copy3d")
        es = src.element_size()
        with torch.cuda.device(self.device):
            if src.dtype == torch.float32:
                _lib.check(self.lib.fdn_copy3d(src.data_ptr() + es * int(src_off), int(in_sa), int(in_sb), int(b0),
                                               int(bw), int(c0), int(cw), dst.data_ptr() + es * int(dst_off),
                                               int(out_sa), int(out_sb), int(A), int(B), int(C), _stream_ptr(torch)))
            else:
                _lib.check(self.lib.fdn_copy3d_typed(src.data_ptr() + es * int(src_off), dtype_code(src), int(in_sa),
                                                     int(in_sb), int(b0), int(bw), int(c0), int(cw),
                                                     dst.data_ptr() + es * int(dst_off), int(out_sa), int(out_sb),
                                                     int(A), int(B), int(C), _stream_ptr(torch)))

    def copy2d_async(self, dst_ptr, dst_pitch, src_ptr, src_pitch, width_bytes, rows, direction, stream):
        """fdn_copy2d_async on a torch stream: direction 0 = host to device, 1 = device to host, 2 = on the device."""
        with self.torch.cuda.device(self.device):
            _lib.check(self.lib.fdn_copy2d_async(int(dst_ptr), int(dst_pitch), int(src_ptr), int(src_pitch),
                                                 int(width_bytes), int(rows), int(direction), stream.cuda_stream))

    def transpose_strided(self, src, src_off, in_sn, in_sa, dst, dst_off, out_sn, out_sb, n, A, B):
        """dst[i*out_sn + b*out_sb + a] = src[i*in_sn + a*in_sa + b] -- the transposing unpack of the re-slab."""
        torch = self.torch
        self._same_dtype(src, dst, "transpose_strided")
        es = src.element_size()
        with torch.cuda.device(self.device):
            if src.dtype == torch.float32:
                _lib.check(self.lib.fdn_transpose_strided(src.data_ptr() + es * int(src_off), int(in_sn), int(in_sa),
                                                          dst.data_ptr() + es * int(dst_off), int(out_sn), int(out_sb),
                                                          int(n), int(A), int(B), _stream_ptr(torch)))
            else:
                _lib.check(self.lib.fdn_transpose_strided_typed(src.data_ptr() + es * int(src_off), dtype_code(src),
                                                                int(in_sn), int(in_sa),
                                                                dst.data_ptr() + es * int(dst_off), int(out_sn),
                                                                int(out_sb), int(n), int(A), int(B), _stream_ptr(torch)))

    def filter_along_axis(self, vol, out, axis: int, kernel, flow: Optional[FlowParams], chunk: Optional[int] = None,
                          exact: bool = True, scratch=None):
        """One pass of the reference's filter_along_{Z,Y,X} (src/flowdenoising.py:175-283) on the device."""
        torch = self.torch
        self._check_vol(vol); self._check_vol(out)
        if vol.data_ptr() == out.data_ptr():
            raise ValueError("in-place passes are not supported")
        if vol.dtype != out.dtype:
            raise ValueError("a pass writes the dtype it reads")
        Z, Y, X = vol.shape
        if axis == 0:
            v = View(Z, Z, 0, 1, Y, X, Y * X, X, Y * X, X)
            self.filter_view(vol, out, v, kernel, flow, chunk, exact)
        elif axis == 1:
            v = View(Y, Y, 0, 1, Z, X, X, Y * X, X, Y * X)
            self.filter_view(vol, out, v, kernel, flow, chunk, exact)
        elif axis == 2:
            if flow is None:
                k, kp = _taps(kernel)
                with torch.cuda.device(self.device):
                    if vol.dtype == torch.float32:
                        _lib.check(self.lib.fdn_gauss_rows(vol.data_ptr(), out.data_ptr(), Z * Y, X, kp, k.size,
                                                           int(bool(exact)), _stream_ptr(torch)))
                    else:
                        _lib.check(self.lib.fdn_gauss_rows_typed(vol.data_ptr(), out.data_ptr(), dtype_code(vol), Z * Y,
                                                                 X, kp, k.size, int(bool(exact)), _stream_ptr(torch)))
                return
            # slices vol[:, :, x] are (Z, Y) images with element-strided columns: run on the [Z, X, Y] transpose
            vt = self.transpose_yx(vol, scratch[0] if scratch else None)
            ot = scratch[1] if scratch else torch.empty_like(vt)
            v = View(X, X, 0, 1, Z, Y, Y, X * Y, Y, X * Y)
            self.filter_view(vt, ot, v, kernel, flow, chunk, exact)
            self.transpose_yx(ot.view(Z, X, Y), out)
        else:
            raise ValueError("axis must be 0, 1 or 2")

    def filter(self, vol, kernels: Sequence, flow: Optional[FlowParams], chunk: Optional[int] = None,
               exact: bool = True):
        """Z, Y, X passes (src/flowdenoising.py:285-290). Returns (zy, zyx): the reference leaves the Z+Y
        intermediate in `vol` and the final result in `filtered_vol`; `vol` itself is not modified here."""
        torch = self.torch
        self._check_vol(vol)
        Z, Y, X = vol.shape
        # every volume-sized buffer exists before the first pass sizes its workspace from the free memory
        a = torch.empty_like(vol)
        b = torch.empty_like(vol)
        ot = torch.empty((Z, X, Y), dtype=vol.dtype, device=vol.device) if flow is not None else torch.empty_like(vol)
        self.filter_along_axis(vol, a, 0, kernels[0], flow, chunk, exact)
        self.filter_along_axis(a, b, 1, kernels[1], flow, chunk, exact)      # b = ZY
        if flow is None:
            self.filter_along_axis(b, ot, 2, kernels[2], flow, chunk, exact)
            return b, ot
        # X pass on the [Z, X, Y] transpose: `a` (the Z result) is dead now and holds first the transposed input,
        # then -- once the pass has written `ot` -- the final result
        vt = self.transpose_yx(b, a.view(Z, X, Y))
        v = View(X, X, 0, 1, Z, Y, Y, X * Y, Y, X * Y)
        self.filter_view(vt, ot, v, kernels[2], flow, chunk, exact)
        out = self.transpose_yx(ot, a.view(Z, Y, X))
        return b, out

    # ---- building blocks exposed for the module-level functions and the parity tests ----
    def farneback(self, prev, nxt, flow_init, params: FlowParams):
        """cv2.calcOpticalFlowFarneback(prev, next, flow, 0.5, ...) for a batch: prev/next [n,H,W], flow [n,H,W,2]
        (read as initial flow when params.use_prev_flow, overwritten with the result)."""
        torch = self.torch
        n, H, W = prev.shape
        ofp = params.c_struct()
        nbytes = self.lib.fdn_farneback_workspace_bytes(n, H, W, C.byref(ofp))
        if nbytes == 0:
            _lib.check(1)
        ws = self._workspace(nbytes)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.fdn_farneback(prev.data_ptr(), nxt.data_ptr(), flow_init.data_ptr(), n, H, W,
                                              C.byref(ofp), ws.data_ptr(), ws.numel(), _stream_ptr(torch)))
        return flow_init

    def warp_accumulate(self, neigh, flow, weight: float, acc):
        """acc = f32(f64(acc) + f64(remap(neigh, flow)) * weight); neigh/acc [n,H,W], flow [n,H,W,2] or None."""
        torch = self.torch
        n, H, W = neigh.shape
        with torch.cuda.device(self.device):
            _lib.check(self.lib.fdn_warp_accumulate(neigh.data_ptr(), H * W, W,
                                                    None if flow is None else flow.data_ptr(), float(weight),
                                                    acc.data_ptr(), H * W, W, n, H, W, _stream_ptr(torch)))
        return acc
