#!/usr/bin/env python
"""bench.py -- Mvoxels/s of the OF-driven separable Gaussian denoise (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] ...    # the reference's CPU path on the host cores

A step = one full three-pass filter (Z, Y, X; src/flowdenoising.py:285-290) of the workload volume.
Default workload at every N: BASELINE.json configs[1] -- 512x1024x1024 float32 FIB-SEM-like synthetic volume, sigma=2
per axis, Farneback defaults (levels=3, winsize=5, iterations=3, poly 5/1.2). At N>1 the same volume is slab-sharded
(strong scaling; halo exchange + all-to-all re-slab, flowdenoising_b200/dist.py). `--config cfg1..cfg5` selects the
other BASELINE.json configurations (both arms); --shape/--sigma/--levels/--winsize/--dtype override single fields.

JSON keys follow the bench contract: `value` = device-resident whole-job throughput, `e2e` = the same through the
reference-facing Python classes with host buffers (H2D/D2H inside the timed region), `roofline` for the dominant
kernel (k_flow_iter) from CUDA events inside the timed region, `cpu_baseline` = the reference's CPU path (oracle
driver calling cv2 exactly like src/flowdenoising.py:306-327) timed on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "Mvoxels/s OF-Gaussian denoise"
UNIT = "Mvoxel/s"

# BASELINE.json configs[0..4] (SURVEY.md §8 size table): shape Z Y X, sigma per axis (Z, Y, X), Farneback levels /
# winsize, input dtype (uint8 TIFF stacks are cast to float32 at load, src/flowdenoising.py:475), OF on/off
CONFIGS = {
    "cfg1": dict(index=0, shape=(64, 256, 256), sigma=(2.0, 2.0, 2.0), levels=3, winsize=5, dtype="float32", no_of=False),
    "cfg2": dict(index=1, shape=(512, 1024, 1024), sigma=(2.0, 2.0, 2.0), levels=3, winsize=5, dtype="float32", no_of=False),
    "cfg3": dict(index=2, shape=(512, 1024, 1024), sigma=(2.0, 2.0, 2.0), levels=3, winsize=5, dtype="float32", no_of=True),
    "cfg4": dict(index=3, shape=(256, 2048, 2048), sigma=(4.0, 2.0, 2.0), levels=5, winsize=9, dtype="uint8", no_of=False),
    "cfg5": dict(index=4, shape=(1024, 2048, 2048), sigma=(2.0, 2.0, 2.0), levels=3, winsize=5, dtype="float32", no_of=False),
}
OF_ITERS = 3


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS), help="BASELINE.json configuration (default cfg2)")
    ap.add_argument("--shape", type=int, nargs=3, default=None, help="Z Y X (overrides the configuration)")
    ap.add_argument("--sigma", type=float, nargs="+", default=None, help="one value, or Z Y X")
    ap.add_argument("--levels", type=int, default=None)
    ap.add_argument("--winsize", type=int, default=None)
    ap.add_argument("--dtype", default=None, choices=["float32", "uint8"], help="input voxel type (values only: the filter runs in float32)")
    ap.add_argument("--no-of", action="store_true", help="OF disabled (plain separable Gaussian), as in cfg3")
    ap.add_argument("--fast-noof", action="store_true", help="no-OF path with float32 FMA arithmetic")
    ap.add_argument("--recompute-flow", action="store_true",
                    help="the reference's --recompute_flow: every flow starts from zero instead of the previous chain step")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-parity", action="store_true")
    ap.add_argument("--cpu-slices", type=int, default=0, help="slices per axis in the CPU sample (0: one per core)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the arrays the last step returned as DIR/<name>.npy (float32): "
                         "whole volumes up to 4 Mi voxels, else a fixed seeded sample of 4 Mi voxels (dump_sample_index)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.warmup < 0:
        ap.error("--warmup must not be negative")
    if a.dump_outputs is not None and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    cfg = dict(CONFIGS[a.config])
    a.customised = any(v is not None for v in (a.shape, a.sigma, a.levels, a.winsize, a.dtype)) or \
        (a.no_of and not cfg["no_of"]) or a.recompute_flow
    if a.shape is not None:
        cfg["shape"] = tuple(a.shape)
    if a.sigma is not None:
        if len(a.sigma) not in (1, 3):
            ap.error("--sigma takes one value or three (Z Y X)")
        cfg["sigma"] = tuple(a.sigma * 3) if len(a.sigma) == 1 else tuple(a.sigma)
    if a.levels is not None:
        cfg["levels"] = a.levels
    if a.winsize is not None:
        cfg["winsize"] = a.winsize
    if a.dtype is not None:
        cfg["dtype"] = a.dtype
    if a.no_of:
        cfg["no_of"] = True
    a.shape, a.sigma, a.levels, a.winsize, a.dtype, a.no_of = (list(cfg["shape"]), cfg["sigma"], cfg["levels"],
                                                                cfg["winsize"], cfg["dtype"], cfg["no_of"])
    a.config_index = cfg["index"]
    return a


def level_sizes(H, W, levels):
    """Pyramid level sizes OpenCV runs for an H x W slice (level cropping, SURVEY.md App. A.0)."""
    k, scale = 0, 1.0
    while k < levels:
        scale *= 0.5
        if W * scale < 32 or H * scale < 32:
            break
        k += 1
    return [(int(np.rint(H * 0.5 ** j)), int(np.rint(W * 0.5 ** j))) for j in range(k + 1)]


def model_bytes_per_voxel(shape, sigma, levels, no_of):
    """SURVEY.md §8d algorithmic-bytes model: per pass B_a = 12 + 28 L_a + 2 r_a (56 I L_a + 12) with L_a = sum of
    the level pixel counts over the slice pixel count, r_a = int(4 sigma_a + 0.5), I = 3; no-OF: 8 per pass."""
    if no_of:
        return 24.0
    Z, Y, X = shape
    total = 0.0
    for (H, W), sg in zip(((Y, X), (Z, X), (Z, Y)), sigma):
        L = sum(h * w for h, w in level_sizes(H, W, levels)) / float(H * W)
        r = int(4 * sg + 0.5)
        total += 12 + 28 * L + 2 * r * (56 * OF_ITERS * L + 12)
    return total


# ----------------------------------------------------------------------------------------------------------------
def synthetic_volume_torch(shape, device, seed=1, noise_sigma=10.0, integer=False):
    """FIB-SEM-like 8-bit-amplitude volume generated on the device (SURVEY.md §8d: structure drifting ~1 px/slice
    + membranes + Gaussian noise, clipped to [0, 255])."""
    import torch
    Z, Y, X = shape
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    out = torch.empty(shape, dtype=torch.float32, device=device)
    y = torch.arange(Y, device=device, dtype=torch.float32)[None, :, None]
    x = torch.arange(X, device=device, dtype=torch.float32)[None, None, :]
    step = 16
    for z0 in range(0, Z, step):
        z1 = min(Z, z0 + step)
        z = torch.arange(z0, z1, device=device, dtype=torch.float32)[:, None, None]
        v = 128.0 + 60.0 * torch.sin(x / 9.0 + z / 13.0) * torch.cos(y / 7.0 - z / 17.0) \
            + 30.0 * torch.sin((x + y) / 23.0)
        rr = torch.sqrt((x - X / 2 - 0.7 * z) ** 2 + (y - Y / 2 + 0.4 * z) ** 2)
        v = v + 35.0 * torch.tanh(4.0 * torch.sin(rr / 37.0))           # membrane-like rings drifting with z
        v = v + noise_sigma * torch.randn(v.shape, device=device, generator=g)
        v = torch.clamp(v, 0.0, 255.0)
        out[z0:z1] = torch.round(v) if integer else v     # uint8 stacks: integer values held in float32
    return out


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons with NVML during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()
        self.err = None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
                getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
            }
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
                getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
            while not self._stop_evt.is_set():
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = get_reasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.2)
        except Exception as e:  # NVML missing: report, do not fail the bench
            self.err = repr(e)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        d = {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
             "reasons": sorted(self.reasons), "samples": len(self.samples)}
        if self.err:
            d["error"] = self.err
        return d


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ----------------------------------------------------------------------------------------------------------------
def cpu_reference_sample(vol_host, kernels, args, slices_per_axis, cores):
    """The reference's CPU path (oracle driver -> cv2.calcOpticalFlowFarneback / cv2.remap with a thread pool of
    `cores` workers, src/flowdenoising.py:187-206, :306-327) on `slices_per_axis` slices of each pass of the full-size
    volume (every pass reads the ORIGINAL volume here). Returns (extrapolated Mvoxel/s, seconds spent, description,
    {axis: (slice indices, oracle output slices)}): the slices are the bench's parity reference."""
    from oracle import fd_oracle as O
    Z, Y, X = vol_host.shape
    o = O.OracleDenoiser(cores, vol_host, use_OF=not args.no_of, l=args.levels, w=args.winsize, backend="cv2",
                         recompute_flow=args.recompute_flow)
    total = 0.0
    spent = 0.0
    slices = {}
    for axis, n in enumerate((Z, Y, X)):
        ns = min(n, slices_per_axis)
        idx = sorted(set(int(i) for i in np.linspace(0, n - 1, ns).round()))
        t0 = time.perf_counter()
        o.filter_along_axis(axis, kernels[axis], indices=idx)
        dt = time.perf_counter() - t0
        spent += dt
        total += dt * n / len(idx)
        slices[axis] = (idx, np.stack([np.take(o.filtered_vol, i, axis=axis) for i in idx]))
    mvox = Z * Y * X / total / 1e6
    try:
        import cv2
        ver = cv2.__version__
    except Exception:
        ver = "?"
    desc = (f"{slices_per_axis} slices of each of the Z/Y/X passes on the full {Z}x{Y}x{X} volume, {cores} threads, "
            f"cv2 {ver}; extrapolated linearly in slices (per-slice cost is uniform)")
    return mvox, spent, desc, slices


def host_volume(args):
    """Host copy of the workload for the CPU arm (same generator family as the GPU arm's device volume)."""
    from oracle import fd_oracle as O
    shape = tuple(args.shape)
    integer = args.dtype == "uint8"
    if np.prod(shape) <= (1 << 24):
        return O.synthetic_volume(shape, seed=1, noise_sigma=10.0)
    rng = np.random.default_rng(1)
    Z, Y, X = shape
    vol = np.empty(shape, np.float32)
    y = np.arange(Y, dtype=np.float32)[:, None]
    x = np.arange(X, dtype=np.float32)[None, :]
    for z in range(Z):
        v = 128.0 + 60.0 * np.sin(x / 9.0 + z / 13.0) * np.cos(y / 7.0 - z / 17.0) + 30.0 * np.sin((x + y) / 23.0)
        rr = np.sqrt((x - X / 2 - 0.7 * z) ** 2 + (y - Y / 2 + 0.4 * z) ** 2)
        v = v + 35.0 * np.tanh(4.0 * np.sin(rr / 37.0)) + rng.standard_normal((Y, X), dtype=np.float32) * 10.0
        v = np.clip(v, 0, 255)
        vol[z] = np.rint(v) if integer else v
    return vol


def run_reference_arm(args, rank, world):
    """--impl reference: the reference's own CPU implementation on the host cores (rank 0 only)."""
    if rank != 0:
        return
    from oracle import fd_oracle as O
    shape = tuple(args.shape)
    cores = os.cpu_count() or 1
    spa = args.cpu_slices or cores
    vol = host_volume(args)
    kernels = [O.get_gaussian_kernel(sg) for sg in args.sigma]
    vals = []
    desc = ""
    for i in range(args.warmup + args.steps):
        mv, spent, desc, _ = cpu_reference_sample(vol, kernels, args, spa, cores)
        if i >= args.warmup:
            vals.append(mv)
    v = float(np.mean(vals))
    nvox = float(np.prod(shape))
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": nvox / v / 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config(args):
    Z, Y, X = args.shape
    sg = args.sigma
    sig = f"sigma={sg[0]:g} per axis" if sg[0] == sg[1] == sg[2] else f"sigma (Z, Y, X) = ({sg[0]:g}, {sg[1]:g}, {sg[2]:g})"
    kind = "uint8-valued (cast to float32 at load, like the reference's TIFF path)" if args.dtype == "uint8" else "float32"
    return {"workload": f"{Z}x{Y}x{X} {kind} FIB-SEM-like synthetic volume, {sig}, "
                        + ("OF disabled (plain separable Gaussian)" if args.no_of else
                           f"Farneback levels={args.levels} winsize={args.winsize} iterations=3 poly_n=5 poly_sigma=1.2"
                           + (", --recompute_flow (no chained initial flow)" if args.recompute_flow else "")),
            "baseline_config": (f"BASELINE.json configs[{args.config_index}]" if not args.customised else
                                f"custom (started from BASELINE.json configs[{args.config_index}])"),
            "shape": [Z, Y, X], "sigma": list(sg), "levels": args.levels, "winsize": args.winsize,
            "input_dtype": args.dtype, "of": not args.no_of, "recompute_flow": bool(args.recompute_flow),
            "l2_policy": "inputs_exceed_l2 (volume and cached expansions are >> 126 MB)"
                         if Z * Y * X * 4 > (200 << 20) else "l2_flushed_between_steps (256 MiB device buffer rewritten)",
            "model_bytes_per_voxel": round(model_bytes_per_voxel((Z, Y, X), sg, args.levels, args.no_of), 1)}


def slab_digests(t):
    """SHA-256 of every Z-slice of a device tensor [z][Y][X] (host side, outside any timed region)."""
    import hashlib
    out = []
    step = 16
    for z0 in range(0, t.shape[0], step):
        h = t[z0:z0 + step].cpu().numpy()
        out.extend(hashlib.sha256(h[i].tobytes()).hexdigest() for i in range(h.shape[0]))
    return out


DUMP_VOXELS = 1 << 22      # per array: 16 MiB of float32, so the two results of a step stay well under 64 MB


def dump_sample_index(nvox):
    """Flat (C-order) indices of the voxels --dump-outputs writes: all of them up to DUMP_VOXELS, else one voxel
    drawn with a fixed seed from each of DUMP_VOXELS equal runs of the volume, so the sample covers all of it."""
    if nvox <= DUMP_VOXELS:
        return np.arange(nvox, dtype=np.int64)
    run = nvox // DUMP_VOXELS
    return np.arange(DUMP_VOXELS, dtype=np.int64) * run + np.random.default_rng(0).integers(0, run, DUMP_VOXELS)


def dump_outputs(path, arrays, shape, z_range, rank, world):
    """arrays: name -> this rank's Z-slab [z1 - z0][Y][X] of a result (device tensor). Every rank takes its part of
    the voxels at dump_sample_index(); rank 0 writes path/<name>.npy in index order, shaped [Z][Y][X] when the
    whole volume fits the budget."""
    import torch
    import torch.distributed as dist
    Z, Y, X = shape
    idx = dump_sample_index(Z * Y * X)
    lo, hi = z_range[0] * Y * X, z_range[1] * Y * X
    mine = np.nonzero((idx >= lo) & (idx < hi))[0]
    if rank == 0:
        os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        local = torch.from_numpy(idx[mine] - lo).to(t.device)
        part = (mine, torch.take(t, local).cpu().numpy())
        parts = [None] * world
        if world > 1:
            dist.gather_object(part, parts if rank == 0 else None, dst=0)
        else:
            parts[0] = part
        if rank == 0:
            out = np.empty(idx.size, np.float32)
            for pos, vals in parts:
                out[pos] = vals
            np.save(os.path.join(path, f"{name}.npy"), out.reshape(shape) if idx.size == Z * Y * X else out)


# ----------------------------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return 0

    import hashlib
    import torch
    import torch.distributed as dist
    from flowdenoising_b200 import _lib
    from flowdenoising_b200 import flowdenoising as fd
    from flowdenoising_b200.engine import DeviceEngine, FlowParams, gaussian_kernel

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    lib = _lib.load()
    shape = tuple(args.shape)
    Z, Y, X = shape
    nvox = float(Z * Y * X)
    kernels = [gaussian_kernel(sg) for sg in args.sigma]
    flow = None if args.no_of else FlowParams(levels=args.levels, winsize=args.winsize,
                                              use_prev_flow=not args.recompute_flow)
    exact = not args.fast_noof
    integer = args.dtype == "uint8"
    eng = DeviceEngine(device)
    small = Z * Y * X * 4 <= (200 << 20)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=device) if small else None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- workload (device resident before the timed region) ----
    # Volumes of more than 2^31 voxels (cfg5) are never synthesised in one piece: they are DEFINED as eight Z-slabs,
    # slab i generated with seed 1 + i, so that 1, 2, 4 and 8 ranks see the same volume and their result hashes compare
    big = Z * Y * X > (1 << 31)

    def big_slab(z0, z1):
        if Z % 8 or z0 % (Z // 8) or z1 % (Z // 8):      # other splits: a private slab per rank (hashes not comparable)
            return synthetic_volume_torch((z1 - z0, Y, X), device, seed=1 + rank, integer=integer)
        zs = Z // 8
        out = torch.empty((z1 - z0, Y, X), dtype=torch.float32, device=device)
        for i in range(z0 // zs, z1 // zs):
            out[i * zs - z0:(i + 1) * zs - z0] = synthetic_volume_torch((zs, Y, X), device, seed=1 + i, integer=integer)
        return out

    if world == 1:
        d_vol = big_slab(0, Z) if big else synthetic_volume_torch(shape, device, seed=1, integer=integer)
        run_once = lambda: eng.filter(d_vol, kernels, flow, exact=exact)
    else:
        from flowdenoising_b200.dist import DistributedDenoiser
        dd = DistributedDenoiser(eng, shape, flow, exact=exact)
        z0, z1 = dd.z_range
        if big:
            d_slab = big_slab(z0, z1)
        else:
            full_seeded = synthetic_volume_torch(shape, device, seed=1, integer=integer)
            d_slab = full_seeded[z0:z1].contiguous()
            del full_seeded
        run_once = lambda: dd.filter(d_slab, kernels)

    def runner():
        if flush_buf is not None:
            flush_buf.fill_(1)      # small volumes fit the 126 MB L2: rewrite a larger buffer between steps
        return run_once()

    # ---- device-resident throughput (`value`) ----
    res = None
    for _ in range(args.warmup):
        res = None          # drop the previous step's volumes before the next step allocates its own
        res = runner()
    barrier()
    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()
    lib.fdn_reset_launch_count()
    lib.fdn_profile_reset()
    lib.fdn_profile_enable(1)
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        res = None
        res = runner()
    ev1.record()
    barrier()
    lib.fdn_profile_enable(0)
    clocks = sampler.stop()
    ms_total = ev0.elapsed_time(ev1)
    launches = int(lib.fdn_launch_count())
    t = torch.tensor([ms_total], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    value = nvox / (ms_step * 1e-3) / 1e6
    phases = None
    if world > 1 and hasattr(dd, "phase_ms"):
        phases = {k: round(v / (args.warmup + args.steps), 3) for k, v in dd.phase_ms().items()}

    # ---- per-kernel event times -> roofline of the dominant kernel ----
    kern = {}
    for i in range(lib.fdn_profile_kernel_count()):
        ms = C.c_double(); n = C.c_int64(); by = C.c_double()
        _lib.check(lib.fdn_profile_read(i, C.byref(ms), C.byref(n), C.byref(by)))
        if n.value:
            kern[lib.fdn_profile_kernel_name(i).decode()] = {"ms": ms.value, "launches": int(n.value), "bytes": by.value}
    # the dominant kernel per pyramid-level image size (launch records carry n, h, w)
    by_level = {}
    flow_id = [i for i in range(lib.fdn_profile_kernel_count()) if lib.fdn_profile_kernel_name(i) == b"k_flow_iter"][0]
    for i in range(lib.fdn_profile_record_count()):
        kid = C.c_int(); rn = C.c_int(); rh = C.c_int(); rw = C.c_int(); ms = C.c_double(); by = C.c_double()
        _lib.check(lib.fdn_profile_record(i, C.byref(kid), C.byref(rn), C.byref(rh), C.byref(rw), C.byref(ms), C.byref(by)))
        if kid.value == flow_id:
            d = by_level.setdefault(f"{rh.value}x{rw.value}", {"ms": 0.0, "bytes": 0.0, "launches": 0})
            d["ms"] += ms.value; d["bytes"] += by.value; d["launches"] += 1
    lib.fdn_profile_reset()
    peak, peak_src = measured_peak()
    dom = max(kern, key=lambda k: kern[k]["ms"]) if kern else None
    roofline = None
    if dom:
        kd = kern[dom]
        achieved = kd["bytes"] / (kd["ms"] * 1e-3) / 1e9
        # DRAM traffic per launch: bytes-per-algorithmic-byte ratio of the kernel's committed `ncu --set full` capture
        # (profiles/traffic.json) x the algorithmic bytes of this run's average launch; null without a capture
        traffic, traffic_src = None, None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                tr = json.load(f).get(dom)
            if tr:
                traffic = tr["dram_bytes_per_algorithmic_byte"] * kd["bytes"] / kd["launches"]
                traffic_src = tr["source"]
        except Exception:
            pass
        roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": peak_src,
                    "avg_launch_ms": kd["ms"] / kd["launches"], "launches": kd["launches"],
                    "algorithmic_bytes_per_launch": kd["bytes"] / kd["launches"],
                    "share_of_step": kd["ms"] / (ms_total if ms_total > 0 else 1.0),
                    "kernel_ms_per_step": {k: round(v["ms"] / args.steps, 3) for k, v in sorted(kern.items())},
                    # every kernel of the path against the same peak (algorithmic bytes / CUDA-event time)
                    "kernel_frac_of_peak": {k: round(v["bytes"] / (v["ms"] * 1e-3) / 1e9 / peak, 3)
                                            for k, v in sorted(kern.items()) if v["ms"] > 0},
                    "flow_iter_by_level": {k: {"ms_per_step": round(v["ms"] / args.steps, 2), "launches": v["launches"],
                                               "frac_of_peak": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9 / peak, 3)}
                                           for k, v in by_level.items() if v["ms"] > 0}}
    model_b = model_bytes_per_voxel(shape, args.sigma, args.levels, args.no_of)
    whole_job_frac = (model_b * nvox / (ms_step * 1e-3) / 1e9) / (world * peak)

    # ---- identity of the result: SHA-256 over the per-Z-slice SHA-256 digests, in Z order (independent of N) ----
    zyx = res[1]
    digests = slab_digests(zyx)
    own_digests = list(digests)
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, digests)
        digests = [d for part in gathered for d in part]
    result_sha = hashlib.sha256("".join(digests).encode()).hexdigest()
    expected = None
    try:
        with open(os.path.join(ROOT, "profiles", "expected_hashes.json")) as f:
            expected = json.load(f).get(hash_key(args, exact))
    except Exception:
        pass
    identity = {"result_sha256": result_sha, "what": "sha256 over the sha256 of every Z slice of the Z+Y+X result",
                "expected_n1_sha256": expected,
                "equals_n1": (result_sha == expected) if expected else None}
    if args.dump_outputs:
        # what a caller of the timed path receives: (zy, zyx) at N = 1; at N > 1 the result slabs (no zy is asked for)
        dump_outputs(args.dump_outputs, {name: t for name, t in zip(("zy", "zyx"), res) if t is not None}, shape,
                     (0, Z) if world == 1 else dd.z_range, rank, world)

    del res, zyx
    eng.release_workspace()
    torch.cuda.empty_cache()

    # ---- end to end through the reference-facing classes with host buffers ----
    e2e = None
    if not args.skip_e2e and world == 1:
        host = torch.empty(shape, dtype=torch.float32, pin_memory=True)
        host.copy_(d_vol)
        pristine = host.clone()
        h_vol = host.numpy()
        n_e2e = max(1, min(args.steps, 3))
        times = []
        for i in range(1 + n_e2e):          # first one is warm-up
            h_vol[...] = pristine.numpy()   # filter() overwrites vol with the Z+Y intermediate (reference :289)
            obj = fd.GaussianDenoising(os.cpu_count(), h_vol) if args.no_of else \
                fd.FlowDenoising(os.cpu_count(), h_vol, args.levels, args.winsize,
                                 fd.get_flow_without_prev_flow if args.recompute_flow else fd.get_flow_with_prev_flow, fd.warp_slice)
            obj.exact = exact
            obj.filtered_vol = torch.empty(shape, dtype=torch.float32, pin_memory=True).numpy()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            obj.filter(kernels)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if i > 0:
                times.append(dt)
        # median of the samples (all of them are in the line): a call that starts on an idle device while its upload
        # is still running now and then takes 50-100 ms longer than the others (profiles/r2_overlap_lab2.json)
        e2e_s = float(np.median(times))
        e2e = {"value": nvox / e2e_s / 1e6, "unit": UNIT, "h2d_bytes_per_step": int(nvox * 4),
               "d2h_bytes_per_step": int(nvox * 8), "ms_per_step": e2e_s * 1e3, "steps": n_e2e,
               "statistic": "median", "samples_ms": [round(t * 1e3, 1) for t in times],
               "mean_ms_per_step": float(np.mean(times)) * 1e3,
               "api": "flowdenoising_b200.flowdenoising.FlowDenoising(P, vol_numpy, ...).filter(kernels)",
               "host_memory": "pinned (torch pin_memory arrays handed to the classes)"}
        # the same call from ordinary (pageable) NumPy arrays, as a CLI user has them: one sample
        try:
            pv = np.array(pristine.numpy())
            obj = fd.GaussianDenoising(os.cpu_count(), pv) if args.no_of else \
                fd.FlowDenoising(os.cpu_count(), pv, args.levels, args.winsize,
                                 fd.get_flow_without_prev_flow if args.recompute_flow else fd.get_flow_with_prev_flow, fd.warp_slice)
            obj.exact = exact
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            obj.filter(kernels)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            e2e["pageable"] = {"value": nvox / dt / 1e6, "ms_per_step": dt * 1e3, "steps": 1}
            del pv
        except MemoryError:
            pass
        del host, pristine, obj
        fd.release_device_memory()
    elif world > 1 and not args.skip_e2e:
        # host slab -> distributed filter -> host slab, per rank (pinned); max over ranks. filter_host() hides the
        # copies behind the passes (edge slices first, Z pass / X pass split into windows); should it fail on every
        # rank, the plain sequence upload, filter(), download is measured instead and the line says so.
        host = torch.empty(d_slab.shape, dtype=torch.float32, pin_memory=True)
        host.copy_(d_slab)
        out_host = torch.empty(d_slab.shape, dtype=torch.float32, pin_memory=True)
        api = "flowdenoising_b200.dist.DistributedDenoiser.filter_host (pinned host slabs in / out, transfers hidden)"

        def e2e_once(hidden):
            if hidden:
                return dd.filter_host(host, out_host, kernels)
            d_tmp = host.to(device, non_blocking=True)
            _zy, zyx_ = dd.filter(d_tmp, kernels)
            out_host.copy_(zyx_, non_blocking=True)
            return zyx_
        hidden = True
        try:
            r_ = e2e_once(True); del r_     # warm-up: workspace and pinned staging reach their final sizes
        except Exception as ex:             # noqa: BLE001 -- reported in the line
            hidden = False
            api = f"DistributedDenoiser.filter on pinned host slabs (filter_host failed: {type(ex).__name__}: {ex})"
        flag = torch.tensor([1 if hidden else 0], dtype=torch.int32, device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        hidden = bool(flag.item())
        times = []
        for i in range(2):
            barrier()
            t0 = time.perf_counter()
            r_ = e2e_once(hidden)
            barrier()
            times.append(time.perf_counter() - t0)
            del r_
        tt = torch.tensor([times[-1]], dtype=torch.float64, device=device)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_s = float(tt.item())
        same = torch.tensor([1 if slab_digests(out_host) == own_digests else 0], dtype=torch.int32, device=device)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        e2e = {"value": nvox / e2e_s / 1e6, "unit": UNIT, "h2d_bytes_per_step": int(nvox * 4),
               "d2h_bytes_per_step": int(nvox * 4), "ms_per_step": e2e_s * 1e3, "steps": 1, "api": api,
               "result_equals_device_run": bool(same.item())}

    # ---- CPU baseline (rank 0, N = 1 only): bounded sample; its output slices are the parity reference ----
    cpu = None
    parity = None
    if rank == 0 and world == 1 and not args.skip_cpu_baseline:
        from oracle import fd_oracle as O
        cores = os.cpu_count() or 1
        vol_host = d_vol.cpu().numpy()
        okernels = [O.get_gaussian_kernel(sg) for sg in args.sigma]     # SciPy taps, as the reference computes them
        mv, spent, desc, oslices = cpu_reference_sample(vol_host, okernels, args, args.cpu_slices or cores, cores)
        cpu = {"value": mv, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc, "seconds_spent": spent}
        if not args.skip_parity:
            # the same single-axis passes of the ORIGINAL volume on the device, compared slice by slice
            out = torch.empty_like(d_vol)
            tot = same = 0
            max_abs = 0.0
            for axis in range(3):
                eng.filter_along_axis(d_vol, out, axis, okernels[axis], flow, exact=exact)
                idx, ref = oslices[axis]
                got = torch.index_select(out, axis, torch.tensor(idx, device=device)).movedim(axis, 0).cpu().numpy()
                tot += ref.size
                same += int(np.count_nonzero(got.view(np.uint32) == ref.view(np.uint32)))
                max_abs = max(max_abs, float(np.max(np.abs(got.astype(np.float64) - ref.astype(np.float64)))))
            parity = {"checked_voxels": tot, "bit_equal": same == tot, "bit_equal_fraction": same / tot,
                      "max_abs": max_abs, "tolerance_max_abs": 1e-3 * 255.0,
                      "what": "the oracle's output slices of the CPU sample (each pass applied to the original volume) "
                              "vs the same passes on the device"}
            del out

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args), "clocks": clocks, "gpu_launches": launches,
            "e2e": e2e, "roofline": roofline, "cpu_baseline": cpu, "parity": parity, "identity": identity,
            "whole_job_model_frac_of_hbm_peak": whole_job_frac,
        }
        if phases:
            line["phases_ms_per_step"] = phases
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def hash_key(args, exact=True):
    Z, Y, X = args.shape
    sg = args.sigma
    return (f"{Z}x{Y}x{X}_{args.dtype}_s{sg[0]:g}-{sg[1]:g}-{sg[2]:g}_" +
            ("noof_" + ("exact" if exact else "fast") if args.no_of else
             f"l{args.levels}w{args.winsize}" + ("_recompute" if args.recompute_flow else "")))


if __name__ == "__main__":
    sys.exit(main())
