"""Typed (integer) slabs vs the float32 route on several GPUs (DistributedDenoiser) and out of core (streaming a memory
map), keep_dtype.

    python tools/integer_sharded_bench.py [--gpus 1 2 4 8] [--steps 2] [--volumes ...] [--out FILE]

Sharded: bench.py's synthetic volume (seed 1, integers 0..255) as a uint8 volume of BASELINE.json configs[3]'s shape
(256 x 2048 x 2048, sigma 4/2/2, 5 levels, winsize 9) and as an int16 volume (v * 12 - 1536) of configs[1]'s shape
(512 x 1024 x 1024, sigma 2, 3 levels, winsize 5). For every N of --gpus that the node has, one process per GPU runs
DistributedDenoiser.filter() on device-resident Z-slabs, typed and float32 ALTERNATED after one warm-up step of each.
Recorded per route: step times and Mvoxel/s; the bytes and CUDA-event time of the exchanges (re-slab all-to-alls and
the Z halo send/recv, rank 0; events on the compute stream around each exchange, so a time includes waiting for the
slowest peer); the library profiler's time and model bytes of k_copy3d and k_transpose (one profiled step, rank 0);
and the result digest (SHA-256 of the per-Z-slice SHA-256 digests, independent of N).

Streaming (one GPU): the uint8 volume of configs[3]'s shape in a read-only np.memmap, filter() of the module surface
(the -m route) with OF and without, typed and float32 alternated, one step each after no warm-up (a warm-up is a whole
run). Recorded: wall time and the host <-> device bytes of the slabs (counted from the slab geometry).

Parity: the first --parity-slices Z-pass output slices of the typed in-core pass (DeviceEngine, the same kernels the
slabs run) against the C oracle without OF, and, for the sharded N = 1 typed route, equality of its digest with the
in-core typed DeviceEngine.filter(). The card's name and power limit are read in the same run. Writes one JSON
document (stdout, and --out).
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import socket
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

VOLUMES = {   # name -> (dtype, shape, sigmas, levels, winsize)
    "uint8_cfg4": ("uint8", (256, 2048, 2048), (4.0, 2.0, 2.0), 5, 9),
    "int16_cfg2": ("int16", (512, 1024, 1024), (2.0, 2.0, 2.0), 3, 5),
}


def card_info(index):
    try:
        return subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm",
                               "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:   # the torch device name is still recorded
        return f"nvidia-smi unavailable: {e}"


def _typed_volume(torch, name, dev):
    from bench import synthetic_volume_torch
    dt, shape, _s, _l, _w = VOLUMES[name]
    v = synthetic_volume_torch(shape, dev, seed=1, integer=True)
    return (v.to(torch.uint8) if dt == "uint8" else (v * 12 - 1536).to(torch.int16)).contiguous()


def _digest(torch, dist, t):
    """SHA-256 over the per-slice digests of the Z-slabs of all ranks, in Z order (the same for any N)."""
    h = t.cpu().numpy()
    mine = [hashlib.sha256(h[i].tobytes()).hexdigest() for i in range(h.shape[0])]
    allv = [None] * dist.get_world_size()
    dist.all_gather_object(allv, mine)
    return hashlib.sha256("".join(d for part in allv for d in part).encode()).hexdigest()


def _sharded_worker(rank, world, port, names, steps, out_path):
    import numpy as np
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from flowdenoising_b200 import _lib
        from flowdenoising_b200.dist import DistributedDenoiser, split_range
        from flowdenoising_b200.engine import DeviceEngine, FlowParams, gaussian_kernel
        lib = _lib.load()
        kn = [lib.fdn_profile_kernel_name(i).decode() for i in range(lib.fdn_profile_kernel_count())]
        eng = DeviceEngine(dev)
        doc = {}
        for name in names:
            dt, shape, sigmas, levels, win = VOLUMES[name]
            zs, ze = split_range(shape[0], world, rank)
            full = _typed_volume(torch, name, dev)
            typed = full[zs:ze].clone()
            del full
            routes = {"typed": typed, "float32": typed.to(torch.float32)}
            torch.cuda.empty_cache()
            ks = [gaussian_kernel(s) for s in sigmas]
            dd = DistributedDenoiser(eng, shape, FlowParams(levels, win))
            exch = []

            def timed(fn, kind):
                def wrapped(*a, **kw):
                    if kind == "all_to_all":
                        nbytes = sum(int(n) for n in a[1]) * a[0].element_size()
                    else:
                        nbytes = 2 * a[1] * (shape[1] * shape[2]) * a[0].element_size()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    res = fn(*a, **kw)
                    e1.record()
                    exch.append((kind, nbytes, e0, e1))
                    return res
                return wrapped
            dd._all_to_all = timed(dd._all_to_all, "all_to_all")
            dd._z_halo_fill = timed(dd._z_halo_fill, "z_halo")

            def step(t):
                exch.clear()
                torch.cuda.synchronize()
                dist.barrier()
                t0 = time.perf_counter()
                _zy, out = dd.filter(t, ks)
                torch.cuda.synchronize()
                dist.barrier()
                return time.perf_counter() - t0, out

            for r, t in routes.items():                 # warm-up
                step(t)
            times = {r: [] for r in routes}
            for _ in range(steps):
                for r, t in routes.items():
                    times[r].append(step(t)[0])
            rec = {}
            nvox = float(np.prod(shape))
            for r, t in routes.items():
                lib.fdn_profile_reset()
                lib.fdn_profile_enable(1)
                _s, out = step(t)
                lib.fdn_profile_enable(0)
                torch.cuda.synchronize()
                ex = {}
                for kind, nbytes, e0, e1 in exch:
                    x = ex.setdefault(kind, {"calls": 0, "bytes": 0, "ms": 0.0})
                    x["calls"] += 1
                    x["bytes"] += nbytes
                    x["ms"] = round(x["ms"] + e0.elapsed_time(e1), 3)
                kern = {}
                for i, nm in enumerate(kn):
                    if nm not in ("k_copy3d", "k_transpose"):
                        continue
                    ms, n, by = C.c_double(), C.c_int64(), C.c_double()
                    _lib.check(lib.fdn_profile_read(i, C.byref(ms), C.byref(n), C.byref(by)))
                    kern[nm] = {"ms": round(ms.value, 3), "launches": int(n.value), "model_bytes": by.value}
                lib.fdn_profile_reset()
                med = statistics.median(times[r])
                rec[r] = {"step_s": [round(x, 4) for x in times[r]], "median_s": round(med, 4),
                          "mvoxel_s": round(nvox / med / 1e6, 1), "exchanges_rank0": ex, "kernels_rank0": kern,
                          "digest": _digest(torch, dist, out if r == "typed" else out.to(typed.dtype))}
                del out
            doc[name] = rec
            del routes, typed
            torch.cuda.empty_cache()
        if rank == 0:
            with open(out_path, "w") as f:
                json.dump(doc, f)
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def streaming_runs(torch, modes):
    """The -m route on one GPU: a read-only uint8 map of configs[3]'s shape."""
    import numpy as np
    from flowdenoising_b200 import flowdenoising as F
    from flowdenoising_b200 import streaming as S
    from flowdenoising_b200.engine import gaussian_kernel
    dt, shape, sigmas, levels, win = VOLUMES["uint8_cfg4"]
    ks = [gaussian_kernel(s) for s in sigmas]
    moved = {"h2d": 0, "d2h": 0}
    orig = S.StreamingDenoiser._start

    def start(self, lane, src, axis, a, b, r, kernel, mean, pd=np.float32):
        plane = int(np.prod(src.shape)) // src.shape[axis]
        moved["h2d"] += (b - a + 2 * r) * plane * np.dtype(pd).itemsize
        moved["d2h"] += (b - a) * plane * np.dtype(pd).itemsize
        return orig(self, lane, src, axis, a, b, r, kernel, mean, pd)
    S.StreamingDenoiser._start = start
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "vol.raw")
        _typed_volume(torch, "uint8_cfg4", torch.device("cuda", 0)).cpu().numpy().tofile(path)
        torch.cuda.empty_cache()
        mm = np.memmap(path, dtype=np.uint8, mode="r", shape=shape)
        digests = {}
        for mode in modes:
            out[mode] = {}
            for route in ("typed", "float32"):
                moved["h2d"] = moved["d2h"] = 0
                if mode == "of":
                    d = F.FlowDenoising(1, mm, levels, win, keep_dtype=route == "typed")
                else:
                    d = F.GaussianDenoising(1, mm, keep_dtype=route == "typed")
                d.filtered_vol = np.empty(shape, np.float32)      # like the CLI's float32 output map
                t0 = time.perf_counter()
                res = d.filter(ks)
                wall = time.perf_counter() - t0
                digests[(mode, route)] = hashlib.sha256(res.astype(np.uint8).tobytes()).hexdigest()
                out[mode][route] = {"wall_s": round(wall, 3), "pcie_h2d_bytes": moved["h2d"],
                                    "pcie_d2h_bytes": moved["d2h"],
                                    "result_sha256_as_uint8": digests[(mode, route)]}
                print(json.dumps({"streaming": {mode: {route: out[mode][route]["wall_s"]}}}), flush=True)
                del d, res
                F.release_device_memory()
    S.StreamingDenoiser._start = orig
    return out


def parity(torch, names, slices):
    """Sampled Z-pass output slices of the typed pass vs the C oracle (no OF), and the in-core typed digest."""
    import numpy as np
    from flowdenoising_b200.engine import DeviceEngine, FlowParams, gaussian_kernel
    from oracle import fd_oracle_int as I
    dev = torch.device("cuda", 0)
    eng = DeviceEngine(dev)
    res = {}
    for name in names:
        dt, shape, sigmas, levels, win = VOLUMES[name]
        typed = _typed_volume(torch, name, dev)
        ks = [gaussian_kernel(s) for s in sigmas]
        z = torch.empty_like(typed)
        eng.filter_along_axis(typed, z, 0, ks[0], None)
        got = z[:slices].cpu().numpy()
        host = typed.cpu().numpy()
        d = I.IntegerDenoiser(os.cpu_count() or 1, host, use_OF=False, backend="c")
        d.filtered_vol = np.zeros((slices,) + host.shape[1:], host.dtype)
        d.filter_along_axis(0, ks[0], indices=range(slices))
        del z
        _zy, zyx = eng.filter(typed, ks, FlowParams(levels, win))
        h = zyx.cpu().numpy()
        digest = hashlib.sha256("".join(hashlib.sha256(h[i].tobytes()).hexdigest()
                                        for i in range(h.shape[0])).encode()).hexdigest()
        res[name] = {"z_slices_no_of_equal_oracle": {str(s): bool(np.array_equal(got[s], d.filtered_vol[s]))
                                                     for s in range(slices)},
                     "in_core_typed_digest": digest}
        del typed, zyx, _zy
        eng.release_workspace()
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, nargs="+", default=[1, 2, 4, 8])
    ap.add_argument("--volumes", nargs="+", default=list(VOLUMES), choices=list(VOLUMES))
    ap.add_argument("--steps", type=int, default=2, help="timed steps per route (alternated)")
    ap.add_argument("--streaming", nargs="*", default=["of", "no_of"], choices=["of", "no_of"])
    ap.add_argument("--parity-slices", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import torch
    import torch.multiprocessing as mp
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    ndev = torch.cuda.device_count()
    doc = {"device": torch.cuda.get_device_name(0), "devices_on_node": ndev, "nvidia_smi": card_info(0),
           "sharded": {}, "gpus_not_measured": [n for n in a.gpus if n > ndev]}

    def save():        # after every section: a run cut short still leaves what it measured
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                f.write(json.dumps(doc, indent=1) + "\n")
    for n in [n for n in a.gpus if n <= ndev]:
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "rank0.json")
            mp.spawn(_sharded_worker, args=(n, _free_port(), a.volumes, a.steps, path), nprocs=n, join=True)
            with open(path) as f:
                doc["sharded"][str(n)] = json.load(f)
        print(json.dumps({"N": n, **{v: {r: doc["sharded"][str(n)][v][r]["mvoxel_s"] for r in ("typed", "float32")}
                                     for v in a.volumes}}), flush=True)
        save()
    for v in a.volumes:
        ds = {r: {doc["sharded"][n][v][r]["digest"] for n in doc["sharded"]} for r in ("typed", "float32")}
        doc.setdefault("digests_equal_for_every_N", {})[v] = {r: len(s) == 1 for r, s in ds.items()}
    if a.streaming:
        doc["streaming_uint8_cfg4_memmap"] = streaming_runs(torch, a.streaming)
        save()
    if a.parity_slices > 0:
        doc["parity"] = parity(torch, a.volumes, a.parity_slices)
        if "1" in doc["sharded"]:
            for v in a.volumes:
                doc["parity"][v]["sharded_n1_typed_equals_in_core"] = \
                    doc["sharded"]["1"][v]["typed"]["digest"] == doc["parity"][v]["in_core_typed_digest"]
    doc["nvidia_smi_after"] = card_info(0)
    save()
    print(json.dumps(doc, indent=1))


if __name__ == "__main__":
    main()
