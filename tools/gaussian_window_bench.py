"""Box window vs Gaussian window (OPTFLOW_FARNEBACK_GAUSSIAN) on the bench volume, one GPU.

    python tools/gaussian_window_bench.py [--shape 512 1024 1024] [--winsizes 5 9 15] [--steps 2] [--out FILE]

For every winsize: device-resident DeviceEngine.filter() (Z, Y, X passes, sigma 2, 3 levels, 3 iterations) on
BASELINE.json configs[1] (bench.py's synthetic volume, seed 1), box and Gaussian runs ALTERNATED after one warm-up run
of each, median step time and Mvoxel/s; then one profiled step per mode with the library's CUDA-event profiler:
per-kernel time and the flow-iteration kernel's algorithmic bytes (56 B per pixel and iteration) over its time, as a
fraction of the 6545.9 GB/s HBM roofline. The Gaussian-window output slices of a sample are compared bit for bit with
the C oracle run with the flag (Z pass from the original volume). The card's name and power limit are read in the same
run. Writes one JSON document (stdout, and --out if given).
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


def card_info(index):
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        return out
    except Exception as e:   # the torch device name is still recorded
        return f"nvidia-smi unavailable: {e}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", type=int, nargs=3, default=[512, 1024, 1024])
    ap.add_argument("--winsizes", type=int, nargs="+", default=[5, 9, 15])
    ap.add_argument("--steps", type=int, default=2, help="timed steps per mode and winsize (alternated)")
    ap.add_argument("--parity-slices", type=int, nargs=2, default=[0, 4], metavar=("S0", "S1"),
                    help="Z-pass output slices [S0, S1) compared with the oracle")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import numpy as np
    import torch
    from bench import synthetic_volume_torch
    from flowdenoising_b200 import _lib
    from flowdenoising_b200.engine import DeviceEngine, FlowParams, gaussian_kernel
    from oracle import fd_oracle_gw as GW

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    lib = _lib.load()
    eng = DeviceEngine(dev)
    shape = tuple(a.shape)
    nvox = float(np.prod(shape))
    vol = synthetic_volume_torch(shape, dev, seed=1)
    kernels = [gaussian_kernel(2.0)] * 3
    names = [lib.fdn_profile_kernel_name(i).decode() for i in range(lib.fdn_profile_kernel_count())]
    doc = {"shape": list(shape), "sigma": 2.0, "levels": 3, "iterations": 3,
           "device": torch.cuda.get_device_name(dev), "nvidia_smi": card_info(0), "peak_gbs": PEAK_GBS,
           "winsizes": {}}

    def step(p):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = eng.filter(vol, kernels, p)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, res

    def profiled(p):
        lib.fdn_profile_reset()
        lib.fdn_profile_enable(1)
        step(p)
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

    host = None
    for win in a.winsizes:
        modes = {"box": FlowParams(3, win), "gaussian": FlowParams(3, win, gaussian_window=True)}
        times = {m: [] for m in modes}
        for m, p in modes.items():      # warm-up
            step(p)
        for _ in range(a.steps):
            for m, p in modes.items():
                times[m].append(step(p)[0])
        rec = {}
        for m, p in modes.items():
            med = statistics.median(times[m])
            kern = profiled(p)
            flow_k = "k_flow_gauss_iter" if m == "gaussian" else "k_flow_iter"   # (k_flow_iter_ws records as k_flow_iter)
            rec[m] = {"step_s": [round(t, 4) for t in times[m]], "median_s": round(med, 4),
                      "mvoxel_s": round(nvox / med / 1e6, 1), "kernels": kern, "flow_kernel": flow_k}
        # parity of a sample of Gaussian-window output slices (Z pass) against the C oracle
        z = torch.empty_like(vol)
        eng.filter_along_axis(vol, z, 0, kernels[0], modes["gaussian"])
        if host is None:
            host = vol.cpu().numpy()
        out = np.zeros_like(host)
        got = z.cpu().numpy()
        s0, s1 = a.parity_slices
        GW.flow_axis_c(host, 0, kernels[0], winsize=win, s0=s0, s1=s1, out=out)
        rec["gaussian"]["parity_z_slices_vs_oracle"] = {str(s): bool(np.array_equal(got[s], out[s])) for s in range(s0, s1)}
        del z, got
        doc["winsizes"][str(win)] = rec
        print(json.dumps({str(win): {m: {k: rec[m][k] for k in ("median_s", "mvoxel_s", "flow_kernel")}
                                     for m in modes}}), flush=True)
    doc["nvidia_smi_after"] = card_info(0)
    s = json.dumps(doc, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
