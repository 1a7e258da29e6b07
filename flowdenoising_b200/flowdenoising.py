#!/usr/bin/env python
'''3D Gaussian filtering controlled by the optical flow -- B200 (sm_100a) implementation.

Drop-in for the module / CLI surface of the reference's ``src/flowdenoising.py`` (same function and class
names, argument meaning and error behaviour; file:line citations below are into /root/reference). The hot
path -- ``filter_along_Z/Y/X`` and everything under it -- runs as hand-written CUDA kernels reached through the
C ABI of ``libfdn_b200.so``; there is no CPU fallback.

Differences from the reference that are deliberate (SURVEY.md App. B):
  * ``filter()`` returns ``filtered_vol`` (the reference returns None, Q1); like the reference it leaves the
    Z+Y intermediate in ``vol`` and the Z+Y+X result in ``filtered_vol``.
  * Volumes are processed as float32; integer inputs are converted (Q3). With ``keep_dtype=True`` (CLI
    ``--keep_dtype``) a uint8, uint16 or int16 volume (int8 without OF) keeps its dtype through every pass with the
    reference's integer arithmetic instead, bit for bit.
  * ``l``/``w`` are instance state, not module globals (Q5); iterations / poly_n / poly_sigma are parameters.
  * ``number_of_processes`` is accepted and ignored: slices are batched on the GPU.
'''
from __future__ import annotations

import argparse
import hashlib
import logging
import multiprocessing
import os
import sys
import threading
import time

import numpy as np

from . import engine as _engine
from .engine import FlowParams, OF_LEVELS, OF_WINDOW_SIZE, OF_ITERS, OF_POLY_N, OF_POLY_SIGMA, SIGMA

LOGGING_FORMAT = "[%(asctime)s] (%(levelname)s) %(message)s"
OFCA_EXTENSION_MODE = 1  # cv2.BORDER_REPLICATE (src/flowdenoising.py:47); the only mode implemented

_ENGINE = None


def _get_engine():
    global _ENGINE
    if _ENGINE is None:
        _ENGINE = _engine.DeviceEngine()
    return _ENGINE


def release_device_memory():
    '''Frees the pass workspace the module-level engine keeps between calls (not part of the reference's surface).'''
    if _ENGINE is not None:
        _ENGINE.release_workspace()
        _ENGINE.torch.cuda.empty_cache()


def get_gaussian_kernel(sigma=1):
    '''src/flowdenoising.py:34-45 -- same taps (SciPy's truncated Gaussian, radius int(4*sigma+0.5)).'''
    logging.info(f"Computing gaussian kernel with sigma={sigma}")
    return _engine.gaussian_kernel(float(sigma))


def _to_dev(a, torch, dev):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev, non_blocking=False)


_STAGE_BYTES = 64 << 20
_PINNED = {}


_COPY_POOL = None
_COPY_THREADS = 4


def _pcopy(dst, src):
    """np.copyto(dst, src, casting="unsafe") for the staging copies, large ones split over a few host threads along
    the first axis (NumPy releases the GIL inside the copy loop; one core moves ~5 GB/s, a PCIe 5 link 50)."""
    global _COPY_POOL
    n = dst.shape[0] if dst.ndim else 0
    if n < 2 or dst.nbytes < (8 << 20) or _COPY_THREADS < 2:
        np.copyto(dst, src, casting="unsafe")
        return
    if _COPY_POOL is None:
        from concurrent.futures import ThreadPoolExecutor
        _COPY_POOL = ThreadPoolExecutor(max_workers=_COPY_THREADS, thread_name_prefix="fdn-copy")
    step = -(-n // min(n, _COPY_THREADS))
    jobs = [_COPY_POOL.submit(np.copyto, dst[i:i + step], src[i:i + step], "unsafe") for i in range(0, n, step)]
    for j in jobs:
        j.result()


def _pinned_pair(torch):
    """Two pinned staging buffers per process (page-locking is expensive: they are kept)."""
    if "bufs" not in _PINNED:
        _PINNED["bufs"] = [torch.empty(_STAGE_BYTES // 4, dtype=torch.float32, pin_memory=True) for _ in range(2)]
    return _PINNED["bufs"]


def _is_pinned_f32(a, torch):
    if not (isinstance(a, np.ndarray) and a.dtype == np.float32 and a.flags.c_contiguous and a.flags.writeable):
        return False
    try:
        return bool(torch.from_numpy(a).is_pinned())
    except Exception:
        return False


def _upload_volume(vol, torch, dev):
    """Host volume (any dtype / layout NumPy can cast to float32, pageable or pinned) -> float32 device tensor.
    A pinned float32 array is copied directly; anything else goes through two pinned staging buffers, the host-side
    cast/copy of chunk k+1 overlapping the DMA of chunk k (a pageable cudaMemcpy would serialise the two)."""
    shape = tuple(int(s) for s in vol.shape)
    d = torch.empty(shape, dtype=torch.float32, device=dev)
    if _is_pinned_f32(vol, torch):
        d.copy_(torch.from_numpy(vol), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return d
    bufs = _pinned_pair(torch)
    plane = int(np.prod(shape[1:]))
    step = max(1, (_STAGE_BYTES // 4) // plane)
    if plane > _STAGE_BYTES // 4:      # a single plane larger than the staging buffer: plain copy
        d.copy_(torch.from_numpy(np.ascontiguousarray(vol, dtype=np.float32)))
        return d
    evs = [None, None]
    for i, z0 in enumerate(range(0, shape[0], step)):
        z1 = min(shape[0], z0 + step)
        b = bufs[i & 1][:(z1 - z0) * plane].view((z1 - z0,) + shape[1:])
        if evs[i & 1] is not None:
            evs[i & 1].synchronize()
        _pcopy(b.numpy(), vol[z0:z1])
        d[z0:z1].copy_(b, non_blocking=True)
        evs[i & 1] = torch.cuda.Event()
        evs[i & 1].record()
    torch.cuda.current_stream().synchronize()
    return d


class _Download:
    """Device tensor -> caller's array on a side stream (and, for pageable / non-float32 destinations, a host thread
    that drains pinned staging chunks), so that the copy overlaps whatever the main stream does next."""

    def __init__(self, t, dst, torch):
        self.torch = torch
        self.t = t
        self.dst = dst
        self.stream = torch.cuda.Stream(device=t.device)
        self.ready = torch.cuda.Event()
        self.ready.record()                      # on the current stream: `t` is complete after this point
        self.thread = None
        if _is_pinned_f32(dst, torch):
            with torch.cuda.stream(self.stream):
                self.stream.wait_event(self.ready)
                torch.from_numpy(dst).copy_(t, non_blocking=True)
        else:
            self.thread = threading.Thread(target=self._drain, daemon=True)
            self.thread.start()

    def _drain(self):
        torch = self.torch
        t, dst = self.t, self.dst
        shape = tuple(t.shape)
        plane = int(np.prod(shape[1:]))
        if plane > _STAGE_BYTES // 4:
            self.ready.synchronize()
            dst[...] = t.cpu().numpy()
            return
        step = max(1, (_STAGE_BYTES // 4) // plane)
        bufs = [torch.empty(_STAGE_BYTES // 4, dtype=torch.float32, pin_memory=True) for _ in range(2)]
        with torch.cuda.device(t.device), torch.cuda.stream(self.stream):
            self.stream.wait_event(self.ready)
            chunks = [(z0, min(shape[0], z0 + step)) for z0 in range(0, shape[0], step)]
            evs = []
            def issue(i):
                z0, z1 = chunks[i]
                b = bufs[i & 1][:(z1 - z0) * plane].view((z1 - z0,) + shape[1:])
                b.copy_(t[z0:z1], non_blocking=True)
                e = torch.cuda.Event(); e.record(self.stream)
                evs.append((e, b))
            if chunks:
                issue(0)
            for i, (z0, z1) in enumerate(chunks):
                e, b = evs[i]
                e.synchronize()
                if i + 1 < len(chunks):
                    # the other buffer is free: its previous contents were copied out in the previous iteration
                    issue(i + 1)
                _pcopy(dst[z0:z1], b.numpy())

    def wait(self):
        if self.thread is not None:
            self.thread.join()
        self.stream.synchronize()


def _to_host(t, dst, torch):
    '''Device tensor -> caller's ndarray; straight into its memory when it is a writable float32 C array (a pinned
    array then gets a pinned-speed copy), through a cast otherwise (integer volumes, quirk Q3).'''
    if isinstance(dst, np.ndarray) and dst.dtype == np.float32 and dst.flags.c_contiguous and dst.flags.writeable:
        torch.from_numpy(dst).copy_(t)
    else:
        dst[...] = t.cpu().numpy()


# In-core volumes of at least this many bytes run the first slices of the Z pass and the last columns of the X pass
# as device calls of their own (windows of the periodic view, include/fdn_b200.h), so that the rest of the upload and
# most of the download overlap the passes. Smaller volumes are not worth the two extra calls.
_OVERLAP_MIN_BYTES = 256 << 20
_TRACE = None   # development (tools/overlap_lab.py): a list that receives (label, CUDA event) stamps of filter()


def _mark(torch, label):
    if _TRACE is not None:
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        _TRACE.append((label, e, time.perf_counter()))


class _Upload:
    """Host volume -> float32 device tensor `d` on a side stream, the Z ranges in the given order. ready(k) makes the
    current stream wait until ranges 0..k are on the device. A pinned float32 array is copied directly; anything else
    goes through the two pinned staging buffers on a host thread (cast + copy of one piece overlapping the DMA of
    the previous one)."""

    def __init__(self, vol, torch, dev, ranges):
        self.torch = torch
        self.vol = vol
        self.ranges = list(ranges)
        shape = tuple(int(s) for s in vol.shape)
        self.d = torch.empty(shape, dtype=torch.float32, device=dev)
        self.stream = torch.cuda.Stream(device=dev)
        self.events = [torch.cuda.Event() for _ in self.ranges]
        self.flags = [threading.Event() for _ in self.ranges]
        self.error = None
        self.thread = None
        self.started = False

    def start(self):
        """Issues the copies. Called after the caller's other allocations and workspace sizing: cudaMemGetInfo
        blocks for milliseconds while a large copy is in flight (tools/host_stall_lab.py), which would hold back
        the launches the copy is supposed to hide behind."""
        torch, vol = self.torch, self.vol
        self.started = True
        self.stream.wait_stream(torch.cuda.current_stream())   # earlier users of this memory are done first
        if _is_pinned_f32(vol, torch):
            src = torch.from_numpy(vol)
            with torch.cuda.stream(self.stream):
                for k, (z0, z1) in enumerate(self.ranges):
                    if z1 > z0:
                        self.d[z0:z1].copy_(src[z0:z1], non_blocking=True)
                    self.events[k].record(self.stream)
                    self.flags[k].set()
        else:
            self.thread = threading.Thread(target=self._feed, args=(vol, self.ranges), daemon=True)
            self.thread.start()

    def _feed(self, vol, ranges):
        torch = self.torch
        try:
            shape = tuple(self.d.shape)
            plane = int(np.prod(shape[1:]))
            step = max(1, (_STAGE_BYTES // 4) // plane)
            bufs = _pinned_pair(torch)
            evs = [None, None]
            i = 0
            with torch.cuda.device(self.d.device), torch.cuda.stream(self.stream):
                for k, (a, b) in enumerate(ranges):
                    for z0 in range(a, b, step):
                        z1 = min(b, z0 + step)
                        buf = bufs[i & 1][:(z1 - z0) * plane].view((z1 - z0,) + shape[1:])
                        if evs[i & 1] is not None:
                            evs[i & 1].synchronize()
                        _pcopy(buf.numpy(), vol[z0:z1])
                        self.d[z0:z1].copy_(buf, non_blocking=True)
                        evs[i & 1] = torch.cuda.Event()
                        evs[i & 1].record(self.stream)
                        i += 1
                    self.events[k].record(self.stream)
                    self.flags[k].set()
                for e in evs:                  # the staging buffers belong to the next caller after this
                    if e is not None:
                        e.synchronize()
        except BaseException as e:             # surfaces in ready() / close() on the calling thread
            self.error = e
            for f in self.flags:
                f.set()

    def ready(self, k):
        if not self.started:
            raise RuntimeError("_Upload.ready() before start()")
        self.flags[k].wait()
        if self.error is not None:
            raise self.error
        self.torch.cuda.current_stream().wait_event(self.events[k])

    def close(self):
        if self.thread is not None:
            self.thread.join()
        if self.error is not None:
            raise self.error


def _prefault(a):
    """Touches every page of a freshly allocated (np.zeros_like: still unmapped) result array on a host thread while
    the device computes, so that the download's host copy does not pay the page faults. Values are unchanged."""
    def touch():
        try:
            flat = a.reshape(-1)
            step = max(1, 4096 // a.itemsize)
            for i in range(0, flat.size, step << 14):      # 64 MB at a time: short slices keep the GIL available
                seg = flat[i:i + (step << 14):step]
                seg[...] = seg.copy()                      # (NumPy skips a plain self-assignment)
        except Exception:
            pass                                            # an optimisation only
    if not (isinstance(a, np.ndarray) and a.flags.c_contiguous and a.flags.writeable):
        return None
    th = threading.Thread(target=touch, daemon=True)
    th.start()
    return th


class _DownloadCols:
    """Columns [x0, x1) of a device volume [Z, Y, X] -> the same columns of the caller's array, on a side stream
    (pitched copies, fdn_copy2d_async), while the main stream goes on with the other columns."""

    def __init__(self, t, dst, x0, x1, torch):
        self.torch = torch
        self.t, self.dst, self.x0, self.x1 = t, dst, int(x0), int(x1)
        self.stream = torch.cuda.Stream(device=t.device)
        self.ready = torch.cuda.Event()
        self.ready.record()                      # on the current stream: the columns are complete after this point
        self.thread = None
        self.error = None
        Z, Y, X = (int(v) for v in t.shape)
        if _is_pinned_f32(dst, torch):
            lib = _engine._lib.load()
            with torch.cuda.device(t.device):
                self.stream.wait_event(self.ready)
                _engine._lib.check(lib.fdn_copy2d_async(
                    dst.ctypes.data + 4 * self.x0, 4 * X, t.data_ptr() + 4 * self.x0, 4 * X, 4 * (self.x1 - self.x0),
                    Z * Y, 1, self.stream.cuda_stream))
        else:
            self.thread = threading.Thread(target=self._drain, daemon=True)
            self.thread.start()

    def _drain(self):
        torch = self.torch
        try:
            lib = _engine._lib.load()
            t, dst, x0, x1 = self.t, self.dst, self.x0, self.x1
            Z, Y, X = (int(v) for v in t.shape)
            w = x1 - x0
            step = max(1, (_STAGE_BYTES // 4) // (Y * w))
            bufs = [torch.empty(_STAGE_BYTES // 4, dtype=torch.float32, pin_memory=True) for _ in range(2)]
            chunks = [(z0, min(Z, z0 + step)) for z0 in range(0, Z, step)]
            evs = []
            with torch.cuda.device(t.device):
                self.stream.wait_event(self.ready)

                def issue(i):
                    z0, z1 = chunks[i]
                    b = bufs[i & 1][:(z1 - z0) * Y * w]
                    _engine._lib.check(lib.fdn_copy2d_async(
                        b.data_ptr(), 4 * w, t.data_ptr() + 4 * (z0 * Y * X + x0), 4 * X, 4 * w, (z1 - z0) * Y, 1,
                        self.stream.cuda_stream))
                    e = torch.cuda.Event()
                    e.record(self.stream)
                    evs.append((e, b))
                issue(0)
                for i, (z0, z1) in enumerate(chunks):
                    e, b = evs[i]
                    e.synchronize()
                    if i + 1 < len(chunks):
                        issue(i + 1)
                    _pcopy(dst[z0:z1, :, x0:x1], b.numpy().reshape(z1 - z0, Y, w))
        except BaseException as e:
            self.error = e

    def wait(self):
        if self.thread is not None:
            self.thread.join()
        self.stream.synchronize()
        if self.error is not None:
            raise self.error


def warp_slice(reference, flow):
    '''src/flowdenoising.py:55-63 -- bilinear remap, replicate border, OpenCV's 1/32-px map quantiser.'''
    eng = _get_engine()
    torch = eng.torch
    ref = _to_dev(reference, torch, eng.device)[None]
    fl = _to_dev(flow, torch, eng.device)[None]
    if fl.shape != ref.shape + (2,):
        raise ValueError("flow must have shape reference.shape + (2,)")
    acc = torch.zeros_like(ref)
    eng.warp_accumulate(ref, fl, 1.0, acc)  # f32(0 + f64(v) * 1.0) == v
    return acc[0].cpu().numpy()


def _get_flow(reference, target, l, w, prev_flow, use_prev, iterations, poly_n, poly_sigma, gaussian_window):
    eng = _get_engine()
    torch = eng.torch
    ref = _to_dev(reference, torch, eng.device)[None]
    tgt = _to_dev(target, torch, eng.device)[None]
    if ref.shape != tgt.shape or ref.dim() != 3:
        raise ValueError("reference and target must be 2-D arrays of the same shape")
    if use_prev and prev_flow is not None:
        fl = _to_dev(prev_flow, torch, eng.device)[None].contiguous()
    else:
        fl = torch.zeros(ref.shape + (2,), dtype=torch.float32, device=eng.device)
    p = FlowParams(int(l), int(w), int(iterations), int(poly_n), float(poly_sigma), bool(use_prev),
                   bool(gaussian_window))
    # cv2.calcOpticalFlowFarneback(prev=target, next=reference, ...)
    eng.farneback(tgt, ref, fl, p)
    out = fl[0].cpu().numpy()
    if use_prev and isinstance(prev_flow, np.ndarray) and prev_flow.dtype == np.float32 \
            and prev_flow.shape == out.shape:
        prev_flow[...] = out  # cv2 updates the initial-flow array in place and returns it (SURVEY §8a a7)
        return prev_flow
    return out


def get_flow_with_prev_flow(reference, target, l=OF_LEVELS, w=OF_WINDOW_SIZE, prev_flow=None,
                            iterations=OF_ITERS, poly_n=OF_POLY_N, poly_sigma=OF_POLY_SIGMA, gaussian_window=False):
    '''src/flowdenoising.py:65-87 (OPTFLOW_USE_INITIAL_FLOW); gaussian_window adds OPTFLOW_FARNEBACK_GAUSSIAN.'''
    return _get_flow(reference, target, l, w, prev_flow, True, iterations, poly_n, poly_sigma, gaussian_window)


def get_flow_without_prev_flow(reference, target, l=OF_LEVELS, w=OF_WINDOW_SIZE, prev_flow=None,
                               iterations=OF_ITERS, poly_n=OF_POLY_N, poly_sigma=OF_POLY_SIGMA, gaussian_window=False):
    '''src/flowdenoising.py:89-114 (--recompute_flow); gaussian_window adds OPTFLOW_FARNEBACK_GAUSSIAN.'''
    return _get_flow(reference, target, l, w, None, False, iterations, poly_n, poly_sigma, gaussian_window)


_TYPED_DTYPES = (np.dtype(np.uint8), np.dtype(np.int8), np.dtype(np.uint16), np.dtype(np.int16))


class GaussianDenoising():
    '''src/flowdenoising.py:116-295.

    keep_dtype=True: an integer volume is filtered in its own dtype with the reference's integer semantics (integer
    remap of each neighbour, float32 accumulation, truncation toward zero at every pass's store, the next pass reading
    the truncated result), bit for bit. Without it (the default), or for a float32 volume, the passes run in float32.'''

    def __init__(self, number_of_processes, vol, keep_dtype=False):
        self._progress_done = 0.0
        self._progress_mark = None      # library counter at the start of the device call in flight
        self.number_of_processes = number_of_processes
        self.vol = vol
        vol_size = vol.dtype.itemsize * vol.size
        logging.info(f"shape of the input volume (Z, Y, X) = {vol.shape}")
        logging.info(f"type of the volume = {vol.dtype}")
        logging.info(f"vol requires {vol_size/(1024*1024):.1f} MB")
        if vol.ndim != 3:
            raise ValueError("vol must be a 3-D array (Z, Y, X)")
        self.filtered_vol = np.zeros_like(vol)
        self._flow_params = None  # no OF
        self.exact = True         # no-OF arithmetic: bit-exact NumPy emulation (False: float32 FMA)
        # beyond the reference's surface (set after construction; the CLI maps --border / --gpus / --slab_slices):
        # "wrap": the reference's periodic axis; "reflect", "mirror", "nearest": SciPy's modes, in core or streamed;
        # "mean": the sequential variant's padding (src/flowdenoising_sequential.py:88-89), streamed, float32 only
        self.border = "wrap"
        self.devices = None       # CUDA devices to spread slabs over (None: the current one)
        self.slab_slices = None   # output slices per streamed slab (None: sized from the free device memory)
        self.streaming = None     # None: stream slab by slab only when needed (memory map, > device memory, ...)
        self.keep_dtype = bool(keep_dtype)

    # The reference bumps `progress` once per finished slice (:139-140) and feedback() prints it (:292-295). Here the
    # count of the device call in flight comes from the library (host functions in the stream after every chain step).
    @property
    def progress(self):
        live = 0.0
        if self._progress_mark is not None:
            live = _engine._lib.load().fdn_progress_milli() / 1000.0 - self._progress_mark
        return self._progress_done + live

    @progress.setter
    def progress(self, value):
        self._progress_done = float(value)

    def _begin_device_call(self):
        self._progress_mark = _engine._lib.load().fdn_progress_milli() / 1000.0

    def _end_device_call(self, slices_done):
        self._progress_mark = None
        self._progress_done += slices_done

    # -- device plumbing --
    def _flow(self):
        return self._flow_params

    def _typed(self):
        """True when the passes run in the volume's integer dtype (keep_dtype), in core or streamed (memory maps,
        several devices, volumes larger than the device); raises ValueError for a combination that is not supported
        rather than converting silently."""
        dt = self.vol.dtype
        if not self.keep_dtype or (dt.kind == "f" and dt.itemsize >= 4):
            return False
        if dt not in _TYPED_DTYPES or not dt.isnative:
            raise ValueError(f"keep_dtype: {dt} volumes are not supported (native uint8, int8, uint16 or int16; "
                             f"float16 is out of scope)")
        if dt == np.int8 and self._flow() is not None:
            raise ValueError("keep_dtype: int8 volumes are supported without optical flow only (cv2.remap, which the "
                             "reference calls, rejects int8 images)")
        if self.border == "mean":
            raise ValueError("keep_dtype: streaming with --border mean is not supported for integer volumes (the "
                             "reference defines no integer mean padding)")
        return True

    def _streaming_needed(self):
        if self.streaming is not None:
            return bool(self.streaming)
        if isinstance(self.vol, np.memmap) or self.border == "mean" or (self.devices and len(self.devices) > 1):
            return True
        eng = _get_engine()
        free, _total = eng.torch.cuda.mem_get_info(eng.device)
        # in core: the volume, two intermediates and the result in the pass dtype (float32, or the integer dtype of a
        # typed volume, whose float32 chunk accumulator lives in the workspace), plus a workspace worth having
        itemsize = self.vol.dtype.itemsize if self._typed() else 4
        return 4 * itemsize * self.vol.size + (2 << 30) > 0.9 * free

    def _streamer(self):
        from .streaming import StreamingDenoiser
        done0 = [self._progress_done]

        def report(slices):
            self._progress_done = done0[0] + slices
        sd = StreamingDenoiser(self._flow(), exact=self.exact, border=self.border, slab_slices=self.slab_slices,
                               devices=self.devices, progress=report, keep_dtype=self._typed())
        return sd, done0

    def _pass(self, axis, kernel):
        eng = _get_engine()
        torch = eng.torch
        kernel = np.asarray(kernel, dtype=np.float64)
        assert kernel.size % 2 != 0  # kernel.size must be odd (src/flowdenoising.py:309)
        typed = self._typed()
        if typed and not self._streaming_needed():
            d_in = torch.from_numpy(np.ascontiguousarray(self.vol)).to(eng.device)
            d_out = torch.empty_like(d_in)
            self._begin_device_call()
            eng.filter_along_axis(d_in, d_out, axis, kernel, self._flow(), exact=self.exact, border=self.border)
            self.filtered_vol[...] = d_out.cpu().numpy()
            self._end_device_call(self.vol.shape[axis])
            return
        if self._streaming_needed():
            sd, done0 = self._streamer()
            # the pass dtype (float32, or the typed volume's own), or float32: exact for the integers of a typed pass
            pd = self.vol.dtype if typed else np.dtype(np.float32)
            ok = self.filtered_vol.dtype in (pd, np.dtype(np.float32))
            dst = self.filtered_vol if ok else np.empty(self.vol.shape, pd)
            sd.filter_axis(self.vol, dst, axis, kernel)
            if dst is not self.filtered_vol:
                self.filtered_vol[...] = dst
            sd.release()
            self._progress_done = done0[0] + self.vol.shape[axis]
            return
        d_in = _upload_volume(self.vol, torch, eng.device)
        d_out = torch.empty_like(d_in)
        self._begin_device_call()
        eng.filter_along_axis(d_in, d_out, axis, kernel, self._flow(), exact=self.exact, border=self.border)
        dl = _Download(d_out, self.filtered_vol, torch)
        dl.wait()
        self._end_device_call(self.vol.shape[axis])

    def filter_along_Z(self, kernel):
        logging.info(f"Filtering along Z with kernel length={kernel.size}")
        self._pass(0, kernel)

    def filter_along_Y(self, kernel):
        logging.info(f"Filtering along Y with kernel length={kernel.size}")
        self._pass(1, kernel)

    def filter_along_X(self, kernel):
        logging.info(f"Filtering along X with kernel length={kernel.size}")
        self._pass(2, kernel)

    # The reference's per-slice / per-chunk entry points (:133-173). A slice is not a useful unit of GPU work,
    # but they are kept so that code driving the reference slice by slice still runs. The neighbours of a slice are
    # the slices the border maps to (the reference's `% n` for wrap and, as before, for mean).
    def _slice(self, axis, idx, kernel):
        eng = _get_engine()
        torch = eng.torch
        kernel = np.asarray(kernel, dtype=np.float64)
        assert kernel.size % 2 != 0
        r = kernel.size // 2
        n = self.vol.shape[axis]
        idxs = _engine.border_indices(np.arange(idx - r, idx + r + 1), n, self.border)
        typed = self._typed()
        slab = np.ascontiguousarray(np.moveaxis(np.take(self.vol, idxs, axis=axis), axis, 0),
                                    dtype=self.vol.dtype if typed else np.float32)
        d_in = torch.from_numpy(slab).to(eng.device)
        H, W = slab.shape[1:]
        d_out = torch.empty((1, H, W), dtype=d_in.dtype, device=eng.device)
        v = _engine.View(2 * r + 1, 1, r, 0, H, W, H * W, W, H * W, W)
        eng.filter_view(d_in, d_out, v, kernel, self._flow(), exact=self.exact)
        res = d_out[0].cpu().numpy()
        if axis == 0:
            self.filtered_vol[idx, :, :] = res
        elif axis == 1:
            self.filtered_vol[:, idx, :] = res
        else:
            self.filtered_vol[:, :, idx] = res
        self.progress += 1

    def filter_along_Z_slice(self, z, kernel): self._slice(0, z, kernel)
    def filter_along_Y_slice(self, y, kernel): self._slice(1, y, kernel)
    def filter_along_X_slice(self, x, kernel): self._slice(2, x, kernel)

    def _chunk(self, axis, start, count, kernel):
        '''The reference's unit of parallel work (:160-173) as ONE device call: the chunk's slices plus an r-slice
        halo (the slices the border maps to) go up as a slab, one non-periodic view filters them, the result comes back. Same bits as
        slice-by-slice calls (every output slice sees the same inputs).'''
        if count <= 0:
            return
        eng = _get_engine()
        torch = eng.torch
        kernel = np.asarray(kernel, dtype=np.float64)
        assert kernel.size % 2 != 0
        r = kernel.size // 2
        n = self.vol.shape[axis]
        idxs = _engine.border_indices(np.arange(start - r, start + count + r), n, self.border)
        typed = self._typed()
        slab = np.ascontiguousarray(np.moveaxis(np.take(self.vol, idxs, axis=axis), axis, 0),
                                    dtype=self.vol.dtype if typed else np.float32)
        d_in = torch.from_numpy(slab).to(eng.device)
        H, W = slab.shape[1:]
        d_out = torch.empty((count, H, W), dtype=d_in.dtype, device=eng.device)
        v = _engine.View(count + 2 * r, count, r, 0, H, W, H * W, W, H * W, W)
        eng.filter_view(d_in, d_out, v, kernel, self._flow(), exact=self.exact)
        res = d_out.cpu().numpy()
        out_idx = [(start + d) % n for d in range(count)]
        if axis == 0:
            self.filtered_vol[out_idx, :, :] = res
        elif axis == 1:
            self.filtered_vol[:, out_idx, :] = np.moveaxis(res, 0, 1)
        else:
            self.filtered_vol[:, :, out_idx] = np.moveaxis(res, 0, 2)
        self.progress += count

    def filter_along_Z_chunk(self, chunk_index, chunk_size, chunk_offset, kernel):
        self._chunk(0, chunk_index*chunk_size + chunk_offset, chunk_size, kernel)
        return chunk_index

    def filter_along_Y_chunk(self, chunk_index, chunk_size, chunk_offset, kernel):
        self._chunk(1, chunk_index*chunk_size + chunk_offset, chunk_size, kernel)
        return chunk_index

    def filter_along_X_chunk(self, chunk_index, chunk_size, chunk_offset, kernel):
        self._chunk(2, chunk_index*chunk_size + chunk_offset, chunk_size, kernel)
        return chunk_index

    def filter(self, kernels):
        '''src/flowdenoising.py:285-290: Z, Y, X passes; vol ends as the Z+Y intermediate, filtered_vol as the
        Z+Y+X result. In core: one upload (pinned staging), three device passes, the download of the Z+Y
        intermediate overlapping the X pass. Volumes that are memory-mapped, larger than the device, spread over
        several devices or mean-padded stream through the device(s) slab by slab (streaming.py).'''
        eng = _get_engine()
        torch = eng.torch
        for k in kernels:
            assert np.asarray(k).size % 2 != 0
        ks = [np.asarray(k, np.float64) for k in kernels]
        Z, Y, X = (int(v) for v in self.vol.shape)
        typed = self._typed()
        if typed and not self._streaming_needed():
            # the plain sequence: upload in the dtype, three typed passes, the ZY intermediate and the result home
            d_in = torch.from_numpy(np.ascontiguousarray(self.vol)).to(eng.device)
            self._begin_device_call()
            zy, zyx = eng.filter(d_in, ks, self._flow(), exact=self.exact, border=self.border)
            self.vol[...] = zy.cpu().numpy()
            self.filtered_vol[...] = zyx.cpu().numpy()
            self._end_device_call(Z + Y + X)
            return self.filtered_vol
        if self._streaming_needed():
            sd, done0 = self._streamer()
            # typed: every pass truncates into the volume's dtype, so the intermediates are arrays of that dtype; the
            # result may land in a float32 array (an output map), which holds these integers exactly
            pd = self.vol.dtype if typed else np.dtype(np.float32)
            ok = self.filtered_vol.dtype in (pd, np.dtype(np.float32))
            fv = self.filtered_vol if ok else np.empty(self.vol.shape, pd)
            base = done0[0]
            zy, zyx = None, None
            # three passes with the reference's buffer roles: vol -> scratch -> vol (Z+Y) -> filtered_vol
            writable = isinstance(self.vol, np.ndarray) and self.vol.dtype == pd and self.vol.flags.writeable
            scratch = np.empty(self.vol.shape, pd)
            mean = float(np.float32(np.mean(self.vol))) if self.border == "mean" else None
            sd.filter_axis(self.vol, scratch, 0, ks[0], mean)
            done0[0] = base + Z
            zy = self.vol if writable else np.empty(self.vol.shape, pd)
            sd.filter_axis(scratch, zy, 1, ks[1], mean)
            done0[0] = base + Z + Y
            del scratch
            sd.filter_axis(zy, fv, 2, ks[2], mean)
            sd.release()
            if not writable:
                try:
                    self.vol[...] = zy      # integer volumes: truncation, like the reference (Q3); read-only maps: skip
                except (ValueError, TypeError):
                    pass
            if fv is not self.filtered_vol:
                self.filtered_vol[...] = fv
            self._progress_done = base + Z + Y + X
            return self.filtered_vol
        flow = self._flow()
        plan = self._overlap_plan(torch, ks)
        if plan is not None:
            return self._filter_overlapped(eng, ks, flow, *plan)
        d_in = _upload_volume(self.vol, torch, eng.device)
        a = torch.empty_like(d_in)
        b = torch.empty_like(d_in)
        ot = torch.empty((Z, X, Y), dtype=torch.float32, device=d_in.device) if flow is not None else torch.empty_like(d_in)
        self._begin_device_call()
        bd = self.border
        eng.filter_along_axis(d_in, a, 0, ks[0], flow, exact=self.exact, border=bd)
        eng.filter_along_axis(a, b, 1, ks[1], flow, exact=self.exact, border=bd)          # b = Z+Y
        dl_zy = _Download(b, self.vol, torch)                                   # ... goes home while X runs
        if flow is None:
            eng.filter_along_axis(b, ot, 2, ks[2], None, exact=self.exact, border=bd)
            out = ot
        else:
            vt = eng.transpose_yx(b, a.view(Z, X, Y))
            v = _engine.View(X, X, 0, _engine.border_code(bd), Z, Y, Y, X * Y, Y, X * Y)
            eng.filter_view(vt, ot, v, ks[2], flow, exact=self.exact)
            out = eng.transpose_yx(ot, a.view(Z, Y, X))
        dl = _Download(out, self.filtered_vol, torch)
        dl.wait()
        dl_zy.wait()
        self._end_device_call(Z + Y + X)
        return self.filtered_vol

    def _overlap_plan(self, torch, ks):
        """(head, tail): output slices of the Z pass that run before the whole volume is on the device and columns
        of the X pass whose download stays exposed; None = the plain sequence upload, passes, download."""
        Z, Y, X = (int(v) for v in self.vol.shape)
        if self._flow() is None or 4 * Z * Y * X < _OVERLAP_MIN_BYTES:
            return None     # no-OF passes take a few milliseconds: nothing to hide a transfer behind
        if 4 * Y * X > _STAGE_BYTES or 4 * Z * Y > _STAGE_BYTES:
            return None     # a plane larger than a staging buffer
        # pageable / non-float32 arrays move at the speed of a host copy: larger pieces keep the transfers hidden
        # (pinned: about 256 MB of slices, 8 .. 64 of them -- the head's upload is the part that stays exposed)
        head = min(Z // 2, max(8, min(64, (256 << 20) // (4 * Y * X)))) if _is_pinned_f32(self.vol, torch) else Z // 4
        tail = min(128, X // 2) if _is_pinned_f32(self.filtered_vol, torch) else X // 4
        if head < 1 or tail < 1:
            return None
        return head, tail

    def _filter_overlapped(self, eng, ks, flow, head, tail):
        '''filter() for an in-core volume with the transfers hidden: the Z pass starts on its first `head` slices as
        soon as they and their periodic neighbours are on the device, the last `tail` columns of the X pass run
        while the other columns already travel home. Every slice still sees the same inputs: same bits.'''
        torch = eng.torch
        View = _engine.View
        Z, Y, X = (int(v) for v in self.vol.shape)
        rz = ks[0].size // 2
        pc = _engine.border_code(self.border)    # fdn_view.periodic of every whole-axis view and window below
        if head <= 0 or head + 2 * rz >= Z:      # (head 0: tools/overlap_lab3.py measures the download split alone)
            ranges, head_key, head = [(0, Z)], 0, 0
        else:   # what the head needs first: its periodic neighbours at the far end (the other borders map the head's
            # neighbours below 0 into slices 0 .. r), then slices 0 .. head + r
            ranges, head_key = [(Z - rz, Z), (0, head + rz), (head + rz, Z - rz)], 1
        up = _Upload(self.vol, torch, eng.device, ranges)
        d_in = up.d
        a = torch.empty_like(d_in)
        b = torch.empty_like(d_in)
        ot = torch.empty((Z, X, Y), dtype=torch.float32, device=d_in.device)
        # one workspace for all three passes, sized after every volume-sized buffer exists
        for v, k in ((View(Z, Z, 0, pc, Y, X, Y * X, X, Y * X, X), ks[0]),
                     (View(Y, Y, 0, pc, Z, X, X, Y * X, X, Y * X), ks[1]),
                     (View(X, X, 0, pc, Z, Y, Y, X * Y, Y, X * Y), ks[2])):
            eng.reserve_workspace(v, k.size, flow)
        # a pageable result array is usually untouched memory: map its pages while the passes run
        pre = None if _is_pinned_f32(self.filtered_vol, torch) else _prefault(self.filtered_vol)
        up.start()
        self._begin_device_call()
        _mark(torch, "start")
        try:
            up.ready(head_key)
            _mark(torch, "head uploaded")
            if head > 0:
                eng.filter_view(d_in, a, View(Z, head, 0, pc, Y, X, Y * X, X, Y * X, X), ks[0], flow, exact=self.exact)
            _mark(torch, "Z head")
            up.ready(len(ranges) - 1)
            _mark(torch, "all uploaded")
            eng.filter_view(d_in, a[head:], View(Z, Z - head, head, pc, Y, X, Y * X, X, Y * X, X), ks[0], flow,
                            exact=self.exact)
        finally:
            up.close()
        _mark(torch, "Z tail")
        eng.filter_view(a, b, View(Y, Y, 0, pc, Z, X, X, Y * X, X, Y * X), ks[1], flow, exact=self.exact)   # b = Z+Y
        _mark(torch, "Y")
        dl_zy = _Download(b, self.vol, torch)                                   # ... goes home while X runs
        vt = eng.transpose_yx(b, a.view(Z, X, Y))
        out = d_in                                                              # dead since the Z pass
        Xb = X - tail
        eng.filter_view(vt, ot, View(X, Xb, 0, pc, Z, Y, Y, X * Y, Y, X * Y), ks[2], flow, exact=self.exact)
        eng.transpose_strided(ot, 0, X * Y, Y, out, 0, Y * X, X, Z, Xb, Y)
        _mark(torch, "X body")
        if pre is not None:
            pre.join()
        dl_body = _DownloadCols(out, self.filtered_vol, 0, Xb, torch)
        eng.filter_view(vt, ot.view(-1)[Xb * Y:], View(X, tail, Xb, pc, Z, Y, Y, X * Y, Y, X * Y), ks[2], flow,
                        exact=self.exact)
        eng.transpose_strided(ot, Xb * Y, X * Y, Y, out, Xb, Y * X, X, Z, tail, Y)
        _mark(torch, "X tail")
        dl_tail = _DownloadCols(out, self.filtered_vol, Xb, X, torch)
        dl_body.wait()
        _mark(torch, "body home")
        dl_tail.wait()
        _mark(torch, "tail home")
        dl_zy.wait()
        self._end_device_call(Z + Y + X)
        return self.filtered_vol

    def feedback(self):
        while True:
            logging.info(f"{100*self.progress/np.sum(self.vol.shape):3.2f} % filtering completed")
            time.sleep(1)


class FlowDenoising(GaussianDenoising):
    '''src/flowdenoising.py:297-373. ``get_flow`` selects the chaining mode exactly like the reference's
    injected callable: get_flow_with_prev_flow (default) or get_flow_without_prev_flow (--recompute_flow);
    ``warp_slice`` is accepted for signature compatibility (the remap is fused into the accumulation kernel).'''

    def __init__(self, number_of_processes, vol, l=OF_LEVELS, w=OF_WINDOW_SIZE, get_flow=None, warp_slice=None,
                 iterations=OF_ITERS, poly_n=OF_POLY_N, poly_sigma=OF_POLY_SIGMA, gaussian_window=False,
                 keep_dtype=False):
        super().__init__(number_of_processes, vol, keep_dtype=keep_dtype)
        self.l = l
        self.w = w
        self.get_flow = get_flow if get_flow is not None else get_flow_with_prev_flow
        self.warp_slice = warp_slice
        use_prev = self.get_flow is not get_flow_without_prev_flow
        self._flow_params = FlowParams(int(l), int(w), int(iterations), int(poly_n), float(poly_sigma), use_prev,
                                       bool(gaussian_window))


class _Stack:
    """A sequence of same-shape 3-D host arrays seen as one [n, Z, Y, X] array by the staging upload (slices along the
    first axis are stacked when the staging copy asks for them: no host copy of the whole batch)."""

    def __init__(self, items):
        self.items = items
        self.shape = (len(items),) + tuple(int(s) for s in items[0].shape)

    def __getitem__(self, sl):
        return np.stack([np.asarray(v, dtype=np.float32) for v in self.items[sl]])

    def __array__(self, dtype=None, copy=None):
        return self[0:len(self.items)] if dtype is None else self[0:len(self.items)].astype(dtype)


def filter_volumes(vols, kernels, l=OF_LEVELS, w=OF_WINDOW_SIZE, get_flow=get_flow_with_prev_flow, no_OF=False,
                   iterations=OF_ITERS, poly_n=OF_POLY_N, poly_sigma=OF_POLY_SIGMA, gaussian_window=False, exact=True,
                   border="wrap"):
    '''Z+Y+X results of many volumes (subtomograms, montage tiles): a 4-D host array [n, Z, Y, X] or a sequence of 3-D
    host arrays, any dtype NumPy casts (filtered as float32, like FlowDenoising(...).filter). Volumes of one shape are
    filtered together, many per device call (DeviceEngine.filter_batch); each result equals
    FlowDenoising(1, vol, ...).filter(kernels) (GaussianDenoising with no_OF) on that volume alone, bit for bit, with
    the same `border` ("wrap", "reflect", "mirror" or "nearest"; "mean" raises ValueError).
    Returns a list of float32 arrays in input order. Not part of the reference's surface.'''
    if border == "mean":
        raise ValueError("filter_volumes: border 'mean' is not supported (it streams volume by volume; use "
                         "wrap, reflect, mirror or nearest)")
    _engine.border_code(border)
    items = list(vols)
    for v in items:
        if np.ndim(v) != 3:
            raise ValueError("every volume must be a 3-D array (Z, Y, X)")
    ks = [np.asarray(k, np.float64) for k in kernels]
    for k in ks:
        assert k.size % 2 != 0  # kernel.size must be odd (src/flowdenoising.py:309)
    flow = None if no_OF else FlowParams(int(l), int(w), int(iterations), int(poly_n), float(poly_sigma),
                                         get_flow is not get_flow_without_prev_flow, bool(gaussian_window))
    groups = {}
    for i, v in enumerate(items):
        groups.setdefault(tuple(int(s) for s in np.shape(v)), []).append(i)
    results = [None] * len(items)
    if not items:
        return results
    eng = _get_engine()
    torch = eng.torch
    for shape, idx in groups.items():
        # host sub-batches: the batch, its Z result / Z+Y / transposed buffers take 16 bytes per voxel of the device;
        # up to a quarter of the free memory goes to them, the rest to the workspace (filter_batch splits further)
        free, _total = torch.cuda.mem_get_info(eng.device)
        per_vol = 16 * int(np.prod(shape))
        n = max(1, min(len(idx), int(0.25 * free) // per_vol))
        for j0 in range(0, len(idx), n):
            part = idx[j0:j0 + n]
            d = _upload_volume(_Stack([items[i] for i in part]), torch, eng.device)
            # (wrap goes without the keyword: an engine that predates the borders still serves it)
            bkw = {} if border == "wrap" else {"border": border}
            _zy, zyx = eng.filter_batch(d, ks, flow, exact=exact, **bkw)
            res = np.empty((len(part),) + shape, np.float32)
            dl = _Download(zyx, res, torch)
            dl.wait()
            del d, _zy, zyx
            for j, i in enumerate(part):
                results[i] = res[j]
    return results


def int_or_str(text):
    '''Helper function for argument parsing.'''
    try:
        return int(text)
    except ValueError:
        return text


number_of_PUs = multiprocessing.cpu_count()


def build_parser():
    '''Same flags and defaults as src/flowdenoising.py:382-415, plus --iterations/--poly_n/--poly_sigma
    (fixed constants in the reference, :50-52), --gaussian_window (OpenCV's OPTFLOW_FARNEBACK_GAUSSIAN) and
    --compat_zy_output (reproduces quirk Q1).'''
    parser = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    parser.add_argument("-i", "--input", type=int_or_str, help="Input a MRC-file or a multi-image TIFF-file",
                        default="./volume.mrc")
    parser.add_argument("-o", "--output", type=int_or_str, help="Output a MRC-file or a multi-image TIFF-file",
                        default="./denoised_volume.mrc")
    parser.add_argument("-s", "--sigma", nargs="+", help="Gaussian sigma for each dimension in the order (Z, Y, X)",
                        default=(SIGMA, SIGMA, SIGMA))
    parser.add_argument("-l", "--levels", type=int_or_str,
                        help="Number of levels of the Gaussian pyramid used by the optical flow estimator",
                        default=OF_LEVELS)
    parser.add_argument("-w", "--winsize", type=int_or_str,
                        help="Size of the window used by the optical flow estimator", default=OF_WINDOW_SIZE)
    parser.add_argument("-v", "--verbosity", type=int_or_str, help="Verbosity level", default=0)
    parser.add_argument("-n", "--no_OF", action="store_true", help="Disable optical flow compensation")
    parser.add_argument("-m", "--memory_map", action="store_true",
                        help="Enable memory-mapping (only for MRC files)")
    parser.add_argument("-p", "--number_of_processes", type=int_or_str,
                        help="Maximum number of processes (accepted for compatibility; slices are batched on the GPU, "
                             "see --gpus)",
                        default=number_of_PUs)
    parser.add_argument("--gpus", type=int, default=1,
                        help="Number of GPUs of this node to spread each pass over (slabs of slices with an r-slice halo)")
    parser.add_argument("--border", choices=["wrap", "reflect", "mirror", "nearest", "mean"], default="wrap",
                        help="Border along the filtered axis. wrap: periodic, the far end of the volume continues it, "
                             "like flowdenoising.py (the reference); reflect: the volume mirrored about its end face, "
                             "edge slice repeated (d c b a | a b c d, SciPy's reflect); mirror: mirrored about the edge "
                             "slice (d c b | a b c d, SciPy's mirror, OpenCV's BORDER_REFLECT_101); nearest: the edge "
                             "slice repeated (a a a | a b c d); mean: padded with the volume's mean like "
                             "flowdenoising_sequential.py (float32, always streamed slab by slab)")
    parser.add_argument("--slab_slices", type=int, default=None,
                        help="Output slices per streamed slab when the volume does not stay on the device "
                             "(default: sized from the free device memory)")
    parser.add_argument("--recompute_flow", action="store_true", help="Disable the use of adjacent optical flow fields")
    parser.add_argument("--show_fingerprint", action="store_true", help="Show a hash of this file")
    parser.add_argument("--iterations", type=int, default=OF_ITERS, help="Farneback iterations per pyramid level")
    parser.add_argument("--poly_n", type=int, default=OF_POLY_N, help="Farneback polynomial-expansion neighbourhood")
    parser.add_argument("--poly_sigma", type=float, default=OF_POLY_SIGMA, help="Farneback polynomial-expansion sigma")
    parser.add_argument("--gaussian_window", action="store_true",
                        help="Farneback with a Gaussian window instead of the box window (cv2.OPTFLOW_FARNEBACK_GAUSSIAN): "
                             "changes the flow estimate, usually more accurate; it is not a speed switch. Wants a larger "
                             "--winsize for the same robustness; winsize 2m and 2m+1 give the same window")
    parser.add_argument("--keep_dtype", action="store_true",
                        help="Filter an integer MRC volume (modes 0, 1, 6) in its own dtype with the reference's integer "
                             "arithmetic (integer remap, truncation after every pass), for bit-for-bit parity with "
                             "flowdenoising.py on integer input. Without it integer volumes are filtered as float32. "
                             "Works in core, with -m (the map stays in its dtype and streams through the device) and "
                             "with --gpus N. TIFF input is float32 either way; the output file is float32 (MRC mode 2), "
                             "which holds the integer result exactly. Not with --border mean; int8 (mode 0) only with "
                             "--no_OF")
    parser.add_argument("--compat_zy_output", action="store_true",
                        help="Write the Z+Y intermediate like the reference CLI does (flowdenoising.py:520) "
                             "instead of the full Z+Y+X result")
    parser.add_argument("--inputs", nargs="+", default=None, metavar="FILE",
                        help="Filter many MRC / TIFF volumes (subtomograms, montage tiles); volumes of one shape run "
                             "together, many per device call. Each result is written as --output_dir/<basename> "
                             "(float32). Instead of -i / -o")
    parser.add_argument("--output_dir", default=None, metavar="DIR",
                        help="Directory of the --inputs results (created if missing)")
    return parser


parser = build_parser()


def main(argv=None):
    from . import volume_io
    print("Python version =", sys.version)
    args = parser.parse_args(argv)
    if args.show_fingerprint:
        hash_algorithm = hashlib.new(name="sha256")
        with open(os.path.abspath(__file__), "rb") as file:
            while chunk := file.read(512):
                hash_algorithm.update(chunk)
        print("fingerprint =", hash_algorithm.hexdigest())

    if args.verbosity == 2:
        logging.basicConfig(format=LOGGING_FORMAT, level=logging.DEBUG)
        logging.info("Verbosity level = 2")
    elif args.verbosity == 1:
        logging.basicConfig(format=LOGGING_FORMAT, level=logging.INFO)
        logging.info("Verbosity level = 1")
    else:
        logging.basicConfig(format=LOGGING_FORMAT, level=logging.CRITICAL)

    for name in ("levels", "winsize"):
        if not isinstance(getattr(args, name), int):
            parser.error(f"--{name} must be an integer")   # the reference crashes inside cv2 instead (Q6)
    if not isinstance(args.input, str) or not isinstance(args.output, str):
        parser.error("--input/--output must be file names")

    if args.recompute_flow:
        get_flow = get_flow_without_prev_flow
        logging.info("No reusing adjacent OF fields as predictions")
    else:
        get_flow = get_flow_with_prev_flow
        logging.info("Using adjacent OF fields as predictions")

    sigma = [float(i) for i in args.sigma]
    if len(sigma) == 1:
        sigma = sigma * 3
    if len(sigma) != 3:
        parser.error("--sigma takes one or three values (Z, Y, X)")
    logging.info(f"sigma={tuple(sigma)}")
    if args.inputs is not None or args.output_dir is not None:
        return _main_batch(args, argv, sigma, get_flow)

    logging.info(f"reading \"{args.input}\"")
    time_0 = time.perf_counter()
    vol = volume_io.read_volume(args.input, memory_map=args.memory_map)
    logging.info(f"read \"{args.input}\" in {time.perf_counter() - time_0} seconds")
    mapped = isinstance(vol, np.memmap)
    if args.keep_dtype and vol.dtype.kind in "iu" and not mapped:
        vol = np.ascontiguousarray(vol, dtype=vol.dtype.newbyteorder("="))      # (-m: the map keeps its dtype)
    elif args.keep_dtype and vol.dtype == np.float16:
        pass                                                                    # ValueError in filter
    elif not mapped:      # (-m: the volume stays in the file and streams through the device slab by slab)
        vol = np.ascontiguousarray(vol, dtype=np.float32)

    kernels = [get_gaussian_kernel(s) for s in sigma]
    logging.info(f"length of each filter (Z, Y, X) = {[len(i) for i in kernels]}")
    logging.info(f"{args.input} type = {vol.dtype}")
    logging.info(f"{args.input} max = {vol.max()}")
    logging.info(f"{args.input} min = {vol.min()}")
    logging.info(f"{args.input} average = {vol.mean()}")

    if args.no_OF:
        fd = GaussianDenoising(args.number_of_processes, vol, keep_dtype=args.keep_dtype)
    else:
        fd = FlowDenoising(args.number_of_processes, vol, args.levels, args.winsize, get_flow, warp_slice,
                           iterations=args.iterations, poly_n=args.poly_n, poly_sigma=args.poly_sigma,
                           gaussian_window=args.gaussian_window, keep_dtype=args.keep_dtype)
    fd.border = args.border
    fd.slab_slices = args.slab_slices
    if args.gpus > 1:
        import torch
        if args.gpus > torch.cuda.device_count():
            parser.error(f"--gpus {args.gpus}: this node has {torch.cuda.device_count()} CUDA devices")
        fd.devices = list(range(args.gpus))
    out_map = None
    if mapped and volume_io.is_mrc_output(args.output) and not args.compat_zy_output:
        # the result is written in place into the output file as well
        out_map = volume_io.create_mrc_memmap(args.output, vol.shape)
        fd.filtered_vol = out_map

    thread = threading.Thread(target=fd.feedback)
    thread.daemon = True  # To obey CTRL+C interruption.
    if args.verbosity:
        thread.start()

    logging.info("Filtering ...")
    time_0 = time.perf_counter()
    filtered_vol = fd.filter(kernels)
    if args.compat_zy_output:
        filtered_vol = np.array(fd.vol, dtype=np.float32)
    logging.info(f"Volume filtered in {time.perf_counter() - time_0} seconds")

    logging.info(f"{args.output} type = {filtered_vol.dtype}")
    logging.info(f"{args.output} max = {filtered_vol.max()}")
    logging.info(f"{args.output} min = {filtered_vol.min()}")
    logging.info(f"{args.output} average = {filtered_vol.mean()}")

    logging.info(f"writing \"{args.output}\"")
    time_0 = time.perf_counter()
    if out_map is not None:
        volume_io.finish_mrc_memmap(args.output, out_map)
    else:
        volume_io.write_volume(args.output, np.asarray(filtered_vol, dtype=np.float32))
    logging.info(f"written \"{args.output}\" in {time.perf_counter() - time_0} seconds")
    return 0


def _main_batch(args, argv, sigma, get_flow):
    """--inputs / --output_dir: every input filtered with filter_volumes, written as output_dir/<basename>."""
    from . import volume_io
    if args.inputs is None:
        parser.error("--output_dir needs --inputs")
    if args.output_dir is None:
        parser.error("--inputs needs --output_dir")
    probe = build_parser()
    probe.set_defaults(input=argparse.SUPPRESS, output=argparse.SUPPRESS)
    explicit = probe.parse_args(argv)
    if explicit.input != argparse.SUPPRESS or explicit.output != argparse.SUPPRESS:
        parser.error("--inputs replaces -i / -o (results go to --output_dir)")
    for flag, bad in (("-m", args.memory_map), ("--gpus > 1", args.gpus > 1), ("--border mean", args.border == "mean"),
                      ("--slab_slices", args.slab_slices is not None), ("--keep_dtype", args.keep_dtype),
                      ("--compat_zy_output", args.compat_zy_output)):
        if bad:
            parser.error(f"--inputs does not support {flag} (in-core float32 volumes on one GPU)")
    names = [os.path.basename(p) for p in args.inputs]
    if len(set(names)) != len(names):
        dup = sorted({n for n in names if names.count(n) > 1})
        parser.error(f"--inputs: several inputs share a basename ({', '.join(dup)}); their results would collide")
    vols = []
    for p in args.inputs:
        logging.info(f"reading \"{p}\"")
        vols.append(np.ascontiguousarray(volume_io.read_volume(p), dtype=np.float32))
    kernels = [get_gaussian_kernel(s) for s in sigma]
    logging.info(f"Filtering {len(vols)} volumes ...")
    time_0 = time.perf_counter()
    results = filter_volumes(vols, kernels, args.levels, args.winsize, get_flow, no_OF=args.no_OF,
                             iterations=args.iterations, poly_n=args.poly_n, poly_sigma=args.poly_sigma,
                             gaussian_window=args.gaussian_window, border=args.border)
    logging.info(f"{len(vols)} volumes filtered in {time.perf_counter() - time_0} seconds")
    os.makedirs(args.output_dir, exist_ok=True)
    for name, res in zip(names, results):
        out = os.path.join(args.output_dir, name)
        logging.info(f"writing \"{out}\"")
        volume_io.write_volume(out, np.asarray(res, dtype=np.float32))
    return 0


if __name__ == "__main__":
    sys.exit(main())
