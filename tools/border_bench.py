"""Cost of the reflect / mirror / nearest borders against the periodic pass (wrap), float32, sigma = 2, Farneback defaults.

    python tools/border_bench.py [--out FILE (default profiles/border_bench.json)] [--rounds 3] [--workloads ...]

Workloads (device-resident volumes, the three passes of DeviceEngine.filter / filter_batch):
  cfg2        512 x 1024 x 1024 with optical flow (bench.py cfg2's shape)
  cfg3_fast   512 x 1024 x 1024 without optical flow, float32 FMA arithmetic (bench.py cfg3)
  cfg3_exact  the same in the exact arithmetic
  batch       256 volumes of 64^3 with optical flow (subtomograms, where the faces are most of the voxels)
Each round runs wrap and every border once, alternately, after a warm-up of each; the record holds the median ms per
step, the library launches per step (fdn_launch_count) and the SHA-256 of each border's result, with the GPU's name and
power limit. The volumes (2 GB, 256 MB) are larger than the 126 MB L2 of a B200.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BORDERS = ["wrap", "reflect", "mirror", "nearest"]
WORKLOADS = ["cfg2", "cfg3_fast", "cfg3_exact", "batch"]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power = [s.strip() for s in out[0].split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:     # the record says why instead of guessing
        return {"error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "border_bench.json"))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--workloads", nargs="+", default=WORKLOADS, choices=WORKLOADS)
    args = ap.parse_args()

    import torch
    from flowdenoising_b200.engine import DeviceEngine, FlowParams, gaussian_kernel

    if not torch.cuda.is_available():
        raise SystemExit("border_bench: no CUDA device (timings are only meaningful on the GPU)")
    eng = DeviceEngine()
    lib = eng.lib
    ks = [gaussian_kernel(2.0)] * 3
    g = torch.Generator(device="cuda")
    g.manual_seed(1)
    record = {"gpu": gpu_info(), "sigma": 2.0, "rounds": args.rounds, "workloads": {}}
    for wl in args.workloads:
        if wl == "batch":
            vol = torch.rand((256, 64, 64, 64), generator=g, device="cuda") * 255.0
            run = lambda b: eng.filter_batch(vol, ks, FlowParams(), border=b)[1]
        else:
            vol = torch.rand((512, 1024, 1024), generator=g, device="cuda") * 255.0
            flow = FlowParams() if wl == "cfg2" else None
            exact = wl != "cfg3_fast"
            run = lambda b, flow=flow, exact=exact: eng.filter(vol, ks, flow, exact=exact, border=b)[1]
        times = {b: [] for b in BORDERS}
        launches, hashes = {}, {}
        for b in BORDERS:                                   # warm-up (modules, workspace)
            run(b)
        torch.cuda.synchronize()
        for _ in range(args.rounds):
            for b in BORDERS:
                lib.fdn_reset_launch_count()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out = run(b)
                torch.cuda.synchronize()
                times[b].append(1e3 * (time.perf_counter() - t0))
                launches[b] = int(lib.fdn_launch_count())
                hashes[b] = hashlib.sha256(out.cpu().numpy().tobytes()).hexdigest()
                del out
        rec = {"shape": list(vol.shape), "ms_per_step": {b: float(np.median(t)) for b, t in times.items()},
               "ms_all": times, "launches_per_step": launches, "sha256": hashes}
        rec["ratio_to_wrap"] = {b: rec["ms_per_step"][b] / rec["ms_per_step"]["wrap"] for b in BORDERS}
        record["workloads"][wl] = rec
        print(wl, json.dumps({k: rec[k] for k in ("ms_per_step", "launches_per_step", "ratio_to_wrap")}), flush=True)
        del vol, run
        eng.release_workspace()
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(record, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
