"""Out-of-core / multi-device passes: the volume stays on the HOST (an ndarray or an np.memmap) and streams through
one or several GPUs slab by slab.

Covers what the reference offers for volumes that do not fit the device: `-m/--memory_map`
(/root/reference/src/flowdenoising.py:407-409, live in src/flowdenoising_sequential.py:510-512) and, as an option, the
sequential variant's mean-padding border (src/flowdenoising_sequential.py:88-89) instead of the periodic one
(src/flowdenoising.py:312).

Within a pass every output slice depends only on its 2r neighbour slices, so a pass is cut into slabs along the
FILTERED axis, each uploaded with an r-slice halo (periodic wrap or the volume's mean), filtered on a non-periodic
view (the same `fdn_view` the multi-GPU path uses) and downloaded:

    Z pass   slab = vol[z0-r : z1+r]            device [zl+2r][Y][X]            slices = planes
    Y pass   slab = vol[:, y0-r : y1+r, :]      device [Z][yl+2r][X]            slice stride X, row stride (yl+2r) X
    X pass   slab = vol[:, :, x0-r : x1+r]      device [Z][Y][xl+2r] -> transposed to [Z][xl+2r][Y] (y contiguous)

Slabs are independent: with several devices they are dealt round-robin, one host thread drives all of them (every
library call only enqueues work). Per device two slabs are in flight -- while slab k computes, slab k+1 is gathered
into pinned staging memory and uploaded on a copy stream and slab k-1 is downloaded and scattered -- so host copies,
PCIe transfers and kernels overlap. Results are bit-identical to the in-core passes (same kernels, same inputs per
slice); tests/test_gpu_streaming.py forces small slabs on toy volumes and demands equality.

Typed mode (keep_dtype=True, an integer volume: uint8, int8, uint16 or int16): staging buffers, device slabs and the
X pass's transposes are in the volume's dtype T, so nothing is cast while gathering and every transfer carries
1 or 2 B/voxel. Each pass truncates into T (the reference's integer `filtered_vol`), so the intermediates of filter()
are T arrays; the last pass may scatter into a float32 array, which holds integers of up to 16 bits exactly.

Nothing here computes on the CPU: the host side only copies slabs.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, List, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import View
from .engine import DeviceEngine, FlowParams


_TYPED = tuple(np.dtype(t) for t in (np.uint8, np.int8, np.uint16, np.int16))


def _torch_dtype(torch, dt):
    return {np.dtype(np.uint8): torch.uint8, np.dtype(np.int8): torch.int8, np.dtype(np.uint16): torch.uint16,
            np.dtype(np.int16): torch.int16}[np.dtype(dt)]


def _lib_dtype(dt):
    return {np.dtype(np.uint8): _lib.DTYPE_U8, np.dtype(np.int8): _lib.DTYPE_I8, np.dtype(np.uint16): _lib.DTYPE_U16,
            np.dtype(np.int16): _lib.DTYPE_I16}[np.dtype(dt)]


def _runs(lo: int, hi: int, n: int):
    """[lo, hi) as (dst offset, src start, length, inside) runs: indices outside [0, n) wrap periodically."""
    out = []
    i = lo
    while i < hi:
        j = i % n
        length = min(hi - i, n - j)
        out.append((i - lo, j, length, 0 <= i < n))
        i += length
    return out


class _DeviceLane:
    """Per-device state: engine, streams, double-buffered pinned staging and device slabs."""

    def __init__(self, device, workspace_limit_bytes):
        torch = _lib.require_cuda()
        self.torch = torch
        self.device = torch.device(device)
        with torch.cuda.device(self.device):
            self.engine = DeviceEngine(self.device, workspace_limit_bytes=workspace_limit_bytes)
            self.compute = torch.cuda.Stream(device=self.device)
            self.copy_in = torch.cuda.Stream(device=self.device)
            self.copy_out = torch.cuda.Stream(device=self.device)
        self.pin_in = [None, None]
        self.pin_out = [None, None]
        self.dev_in = [None, None]
        self.dev_out = [None, None]
        self.dev_tmp = [None, None]     # X pass: transposed input / output
        self.jobs: List[dict] = []      # slabs in flight, oldest first

    def buffers(self, slot, n_in_elems, n_out_elems, need_tmp, dtype=None):
        torch = self.torch
        dtype = torch.float32 if dtype is None else dtype

        def stale(t, n):
            return t is None or t.numel() < n or t.dtype != dtype

        def grow(lst, n, pinned):
            if stale(lst[slot], n):
                lst[slot] = None
                lst[slot] = (torch.empty(n, dtype=dtype, pin_memory=True) if pinned else
                             torch.empty(n, dtype=dtype, device=self.device))
            return lst[slot]
        grow(self.pin_in, n_in_elems, True)
        grow(self.pin_out, n_out_elems, True)
        grow(self.dev_in, n_in_elems, False)
        grow(self.dev_out, n_out_elems, False)
        if need_tmp:
            if stale(self.dev_tmp[0], n_in_elems):
                self.dev_tmp[0] = torch.empty(n_in_elems, dtype=dtype, device=self.device)
            if stale(self.dev_tmp[1], n_out_elems):
                self.dev_tmp[1] = torch.empty(n_out_elems, dtype=dtype, device=self.device)


class StreamingDenoiser:
    """Three-pass filter of a host-resident volume (see the module docstring).

    border: "wrap" (the reference, src/flowdenoising.py:312) or "mean" (the sequential variant's padding).
    slab_slices: output slices per slab (None: sized from `device_budget_bytes` / the free device memory).
    devices: CUDA device indices to spread the slabs over (default: the current device).
    keep_dtype: an integer volume runs the typed passes in its own dtype (see the module docstring); otherwise every
    volume is filtered as float32."""

    def __init__(self, flow: Optional[FlowParams], exact: bool = True, border: str = "wrap",
                 slab_slices: Optional[int] = None, devices: Optional[Sequence[int]] = None,
                 device_budget_bytes: Optional[int] = None, progress: Optional[Callable[[float], None]] = None,
                 keep_dtype: bool = False):
        if border not in ("wrap", "mean"):
            raise ValueError("border must be 'wrap' or 'mean'")
        self.keep_dtype = bool(keep_dtype)
        torch = _lib.require_cuda()
        self.torch = torch
        self.flow = flow
        self.exact = exact
        self.border = border
        self.slab_slices = slab_slices
        self.device_budget_bytes = device_budget_bytes
        self.progress = progress
        devs = list(devices) if devices else [torch.cuda.current_device()]
        self.lanes = [_DeviceLane(f"cuda:{d}", None) for d in devs]

    def pass_dtype(self, src):
        """NumPy dtype the passes over `src` run in: its own for an integer volume in typed mode, float32 otherwise."""
        dt = np.dtype(src.dtype)
        if not self.keep_dtype or dt not in _TYPED:
            return np.dtype(np.float32)
        if self.border != "wrap":
            raise ValueError("keep_dtype: streaming with --border mean is not supported for integer volumes (the "
                             "reference defines no integer mean padding)")
        return dt

    # ---------------------------------------------------------------------------------------------- slab sizing
    def _slab_len(self, shape, axis, r, dtype=np.float32):
        if self.slab_slices:
            return max(1, int(self.slab_slices))
        torch = self.torch
        n = shape[axis]
        budget = self.device_budget_bytes
        if budget is None:
            free = min(torch.cuda.mem_get_info(l.device)[0] for l in self.lanes)
            budget = int(free * 0.8)
        if np.dtype(dtype) != np.float32:
            cost, fixed = self._typed_slice_cost(shape, axis, r, np.dtype(dtype))
        else:
            per_slice = int(np.prod(shape)) // n * 4                 # bytes of one slice
            # per output slice: 2 x (input + output) slabs (+ transposes on the X pass) and the pass workspace (cached
            # polynomial expansions 26.6 B/px, three flow buffers for both chain directions 48 B/px, stash 4 r B/px)
            ws = (27 + 48 + 4 * r) / 4.0 if self.flow is not None else 0.0
            cost = per_slice * (2 * 2 + (2 if axis == 2 else 0) + ws)
            fixed = per_slice * 2 * r * (2 + 27 / 4.0)               # halo slices: input copies + their expansions
        length = int((budget - fixed) // cost)
        if length < 1:
            raise _lib.FdnError("device budget too small for a one-slice slab of this volume")
        # balance the slabs over the devices
        parts = max(len(self.lanes), -(-n // length))
        parts = -(-parts // len(self.lanes)) * len(self.lanes) if n >= len(self.lanes) else parts
        return max(1, -(-n // parts))

    def _typed_slice_cost(self, shape, axis, r, dt):
        """(bytes per output slice, fixed bytes) of a typed slab: 2 x (input + output) slabs in T (+ transposes on the
        X pass) and the typed pass workspace, fdn_workspace_bytes_typed (stash in T, float32 chunk accumulator) at one
        and two output slices."""
        n = shape[axis]
        px = int(np.prod(shape)) // n
        per_slice = px * dt.itemsize
        cost, fixed = per_slice * (2 * 2 + (2 if axis == 2 else 0)), per_slice * 2 * r * 2
        if self.flow is not None:
            H, W = [s for i, s in enumerate(shape) if i != axis]
            ofp = self.flow.c_struct()
            lib = _lib.load()

            def ws(k):
                v = View(k + 2 * r, k, r, 0, H, W, H * W, W, H * W, W)
                nbytes = lib.fdn_workspace_bytes_typed(C.byref(v), 2 * r + 1, C.byref(ofp), k, _lib_dtype(dt))
                if nbytes == 0:
                    _lib.check(1)
                return nbytes
            w1, w2 = ws(1), ws(2)
            cost += w2 - w1
            fixed += max(0, 2 * w1 - w2)
        return cost, fixed

    # ---------------------------------------------------------------------------------------------- host <-> staging
    def _gather(self, src, axis, lo, hi, dst, mean):
        """dst[...] = src[lo:hi along axis] with indices outside [0, n) wrapped or replaced by the mean."""
        n = src.shape[axis]
        for off, start, length, inside in _runs(lo, hi, n):
            sl_d = [slice(None)] * 3
            sl_s = [slice(None)] * 3
            sl_d[axis] = slice(off, off + length)
            sl_s[axis] = slice(start, start + length)
            if inside or self.border == "wrap":
                np.copyto(dst[tuple(sl_d)], src[tuple(sl_s)], casting="unsafe")
            else:
                dst[tuple(sl_d)] = mean

    # ---------------------------------------------------------------------------------------------- one pass
    def filter_axis(self, src, dst, axis: int, kernel, mean: Optional[float] = None):
        """dst = one pass of the reference's filter_along_{Z,Y,X} over the host volume `src` ([Z, Y, X], any dtype
        NumPy can cast to float32; np.memmap welcome). `dst`: float32 host array / memmap of the same shape, != src.
        Typed mode on an integer `src`: the pass runs in src's dtype T and truncates into T; `dst` is a T array, or
        float32 (exact for these integers)."""
        torch = self.torch
        pd = self.pass_dtype(src)
        if pd != np.float32 and np.dtype(dst.dtype) not in (pd, np.dtype(np.float32)):
            raise ValueError(f"a typed pass over a {pd} volume writes {pd} or float32, not {dst.dtype}")
        kernel = np.ascontiguousarray(kernel, dtype=np.float64)
        if kernel.ndim != 1 or kernel.size % 2 == 0:
            raise ValueError("kernel.size must be odd")
        if src.ndim != 3 or tuple(dst.shape) != tuple(src.shape):
            raise ValueError("src and dst must be 3-D arrays of the same shape")
        if np.shares_memory(src, dst):
            raise ValueError("in-place passes are not supported")
        r = kernel.size // 2
        shape = tuple(int(s) for s in src.shape)
        Z, Y, X = shape
        n = shape[axis]
        if self.border == "mean" and mean is None:
            mean = float(np.float32(np.mean(src)))
        L = self._slab_len(shape, axis, r, pd)
        slabs = [(a, min(a + L, n)) for a in range(0, n, L)]
        done = 0
        for k, (a, b) in enumerate(slabs):
            lane = self.lanes[k % len(self.lanes)]
            if len(lane.jobs) == 2:
                done += self._finish(lane, lane.jobs.pop(0), dst, axis)
                self._report(done, n)
            self._start(lane, src, axis, a, b, r, kernel, mean, pd)
        for lane in self.lanes:
            while lane.jobs:
                done += self._finish(lane, lane.jobs.pop(0), dst, axis)
                self._report(done, n)

    def _report(self, done, n):
        if self.progress is not None:
            self.progress(done)

    def _start(self, lane: _DeviceLane, src, axis, a, b, r, kernel, mean, pd=np.float32):
        torch = self.torch
        Z, Y, X = (int(s) for s in src.shape)
        nl = b - a
        ne = nl + 2 * r
        in_shape = {0: (ne, Y, X), 1: (Z, ne, X), 2: (Z, Y, ne)}[axis]
        out_shape = {0: (nl, Y, X), 1: (Z, nl, X), 2: (Z, Y, nl)}[axis]
        n_in, n_out = int(np.prod(in_shape)), int(np.prod(out_shape))
        slot = 0 if not lane.jobs else 1 - lane.jobs[-1]["slot"]
        with torch.cuda.device(lane.device):
            lane.buffers(slot, n_in, n_out, axis == 2, None if pd == np.float32 else _torch_dtype(torch, pd))
            pin = lane.pin_in[slot][:n_in].view(in_shape)
            # the staging buffer may still be the source of the previous upload from this slot
            prev = getattr(lane, f"h2d_done_{slot}", None)
            if prev is not None:
                prev.synchronize()
            self._gather(src, axis, a - r, b + r, pin.numpy(), mean)
            d_in = lane.dev_in[slot][:n_in].view(in_shape)
            d_out = lane.dev_out[slot][:n_out].view(out_shape)
            # (the job that used this slot before has been finished -- downloaded -- by the caller, so its device
            # slabs are free; the other slot's job may still be computing: that is the overlap)
            with torch.cuda.stream(lane.copy_in):
                d_in.copy_(pin, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(lane.copy_in)
                setattr(lane, f"h2d_done_{slot}", ev)
            with torch.cuda.stream(lane.compute):
                lane.compute.wait_event(ev)
                eng = lane.engine
                if axis == 0:
                    v = View(ne, nl, r, 0, Y, X, Y * X, X, Y * X, X)
                    eng.filter_view(d_in, d_out, v, kernel, self.flow, exact=self.exact)
                elif axis == 1:
                    v = View(ne, nl, r, 0, Z, X, X, ne * X, X, nl * X)
                    eng.filter_view(d_in, d_out, v, kernel, self.flow, exact=self.exact)
                else:
                    t_in = eng.transpose_yx(d_in, lane.dev_tmp[0][:n_in].view(Z, ne, Y))
                    t_out = lane.dev_tmp[1][:n_out].view(Z, nl, Y)
                    v = View(ne, nl, r, 0, Z, Y, Y, ne * Y, Y, nl * Y)
                    eng.filter_view(t_in, t_out, v, kernel, self.flow, exact=self.exact)
                    eng.transpose_yx(t_out, d_out)
                done_ev = torch.cuda.Event()
                done_ev.record(lane.compute)
            with torch.cuda.stream(lane.copy_out):
                lane.copy_out.wait_event(done_ev)
                pout = lane.pin_out[slot][:n_out].view(out_shape)
                pout.copy_(d_out, non_blocking=True)
                out_ev = torch.cuda.Event()
                out_ev.record(lane.copy_out)
        lane.jobs.append({"slot": slot, "a": a, "b": b, "out_shape": out_shape, "event": out_ev})

    def _finish(self, lane: _DeviceLane, job, dst, axis):
        job["event"].synchronize()
        n_out = int(np.prod(job["out_shape"]))
        res = lane.pin_out[job["slot"]][:n_out].view(job["out_shape"]).numpy()
        sl = [slice(None)] * 3
        sl[axis] = slice(job["a"], job["b"])
        np.copyto(dst[tuple(sl)], res, casting="unsafe")
        return job["b"] - job["a"]

    # ---------------------------------------------------------------------------------------------- three passes
    def filter(self, vol, kernels, filtered_vol=None, scratch=None):
        """Z, Y, X passes (src/flowdenoising.py:285-290) of the host volume `vol`. Like the reference, `vol` ends up
        holding the Z+Y intermediate and `filtered_vol` the Z+Y+X result; `scratch` (an array / memmap of the volume's
        shape in the pass dtype) holds the Z result in between. `vol` must be writable and of the pass dtype (float32;
        in typed mode the integer volume's own) for the in-place semantics; otherwise a copy of the Z+Y result in the
        pass dtype is returned as the first element. In typed mode `filtered_vol` may be float32."""
        shape = tuple(vol.shape)
        pd = self.pass_dtype(vol)
        if scratch is None:
            scratch = np.empty(shape, pd)
        if filtered_vol is None:
            filtered_vol = np.empty(shape, pd)
        # the sequential variant pads all three passes with the mean of the ORIGINAL volume (vol.mean(), :420-430)
        mean = float(np.float32(np.mean(vol))) if self.border == "mean" else None
        self.filter_axis(vol, scratch, 0, kernels[0], mean)
        writable = isinstance(vol, np.ndarray) and vol.dtype == pd and vol.flags.writeable
        zy = vol if writable else np.empty(shape, pd)
        self.filter_axis(scratch, zy, 1, kernels[1], mean)
        self.filter_axis(zy, filtered_vol, 2, kernels[2], mean)
        return zy, filtered_vol

    def release(self):
        for lane in self.lanes:
            lane.engine.release_workspace()
            lane.pin_in = [None, None]; lane.pin_out = [None, None]
            lane.dev_in = [None, None]; lane.dev_out = [None, None]; lane.dev_tmp = [None, None]
