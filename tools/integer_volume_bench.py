"""Typed (integer) passes vs the float32 route on integer volumes, one GPU.

    python tools/integer_volume_bench.py [--steps 1] [--parity-slices 1] [--out FILE]

Two volumes, bench.py's synthetic volume (seed 1, integers 0..255): a uint8 volume of BASELINE.json configs[3]'s shape
(256 x 2048 x 2048, sigma 4/2/2, 5 levels, winsize 9) and an int16 volume (v * 12 - 1536) of configs[1]'s shape
(512 x 1024 x 1024, sigma 2, 3 levels, winsize 5). For each, with OF and without, device-resident DeviceEngine.filter()
(Z, Y, X passes) runs on the integer tensor (typed passes, keep_dtype) and on its float32 copy (today's route),
ALTERNATED after one warm-up run of each; then one profiled step per route with the library's CUDA-event profiler:
per-kernel time and model bytes (ProfScope, sizeof(T) per volume element) over that time, as a fraction of the
6545.9 GB/s HBM roofline. The first --parity-slices Z-pass output slices of the typed route are compared bit for bit
with the C oracle (fd_oracle_int.IntegerDenoiser, backend "c"): without OF for both volumes, with OF for the volumes of
--parity-of (default int16_cfg2: the oracle's Farneback on 2048 x 2048 slices takes minutes per slice). The card's
name and power limit are read in the same run. Writes one JSON document (stdout, and --out).
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PEAK_GBS = 6545.9   # MEASURED_PEAKS.json hbm_gbs of the B200 the project's records use (DESIGN.md §5)

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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--volumes", nargs="+", default=list(VOLUMES), choices=list(VOLUMES))
    ap.add_argument("--steps", type=int, default=1, help="timed steps per route (alternated)")
    ap.add_argument("--parity-slices", type=int, default=1, help="Z-pass output slices compared with the oracle")
    ap.add_argument("--parity-of", nargs="*", default=["int16_cfg2"], choices=list(VOLUMES))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import numpy as np
    import torch
    from bench import synthetic_volume_torch
    from flowdenoising_b200 import _lib
    from flowdenoising_b200.engine import DeviceEngine, FlowParams, gaussian_kernel
    from oracle import fd_oracle_int as I

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    lib = _lib.load()
    eng = DeviceEngine(dev)
    names = [lib.fdn_profile_kernel_name(i).decode() for i in range(lib.fdn_profile_kernel_count())]
    doc = {"device": torch.cuda.get_device_name(dev), "nvidia_smi": card_info(0), "peak_gbs": PEAK_GBS, "volumes": {}}

    def step(vol, ks, p):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = eng.filter(vol, ks, p)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, res

    def profiled(vol, ks, p):
        lib.fdn_profile_reset()
        lib.fdn_profile_enable(1)
        step(vol, ks, p)
        lib.fdn_profile_enable(0)
        kern = {}
        for i, nm in enumerate(names):
            ms, n, by = C.c_double(), C.c_int64(), C.c_double()
            _lib.check(lib.fdn_profile_read(i, C.byref(ms), C.byref(n), C.byref(by)))
            if n.value:
                kern[nm] = {"ms": round(ms.value, 3), "launches": int(n.value), "bytes": by.value,
                            "frac_of_roofline": round(by.value / (ms.value * 1e-3) / 1e9 / PEAK_GBS, 4)}
        lib.fdn_profile_reset()
        return kern

    for name in a.volumes:
        dt, shape, sigmas, levels, win = VOLUMES[name]
        v = synthetic_volume_torch(shape, dev, seed=1, integer=True)
        typed = (v.to(torch.uint8) if dt == "uint8" else (v * 12 - 1536).to(torch.int16)).contiguous()
        del v
        flt = typed.to(torch.float32)
        ks = [gaussian_kernel(s) for s in sigmas]
        nvox = float(np.prod(shape))
        rec = {"dtype": dt, "shape": list(shape), "sigma": list(sigmas), "levels": levels, "winsize": win, "modes": {}}
        for mode, p in (("of", FlowParams(levels, win)), ("no_of", None)):
            routes = {"typed": typed, "float32": flt}
            times = {r: [] for r in routes}
            for r, t in routes.items():     # warm-up
                step(t, ks, p)
            for _ in range(a.steps):
                for r, t in routes.items():
                    times[r].append(step(t, ks, p)[0])
            m = {}
            for r, t in routes.items():
                med = statistics.median(times[r])
                m[r] = {"step_s": [round(x, 4) for x in times[r]], "median_s": round(med, 4),
                        "mvoxel_s": round(nvox / med / 1e6, 1), "kernels": profiled(t, ks, p)}
            rec["modes"][mode] = m
            print(json.dumps({name: {mode: {r: m[r]["median_s"] for r in m}}}), flush=True)
        if a.parity_slices > 0:   # sampled Z-pass slices of the typed route against the oracle
            s1 = a.parity_slices
            host = typed.cpu().numpy()
            par = {}
            for mode, p in (("of", FlowParams(levels, win)), ("no_of", None)):
                if p is not None and name not in a.parity_of:
                    continue
                z = torch.empty_like(typed)
                eng.filter_along_axis(typed, z, 0, ks[0], p)
                got = z[:s1].cpu().numpy()
                del z
                d = I.IntegerDenoiser(os.cpu_count() or 1, host, use_OF=p is not None, l=levels, w=win, backend="c")
                d.filtered_vol = np.zeros((s1,) + host.shape[1:], host.dtype)
                d.filter_along_axis(0, ks[0], indices=range(s1))
                par[mode] = {str(s): bool(np.array_equal(got[s], d.filtered_vol[s])) for s in range(s1)}
            rec["parity_z_slices_vs_oracle"] = par
        doc["volumes"][name] = rec
        del typed, flt
        torch.cuda.empty_cache()
    doc["nvidia_smi_after"] = card_info(0)
    s = json.dumps(doc, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
