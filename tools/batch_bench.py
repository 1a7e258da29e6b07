"""Batched filtering of many same-shape volumes vs the per-volume loop (float32, sigma = 2, Farneback defaults).

    python tools/batch_bench.py [--out FILE (default profiles/batch_bench.json)] [--rounds 3] [--sizes 256x64x64x64 ...]

For every size (B volumes of Z x Y x X) the two routes run alternately in one process, after a warm-up of every shape:
  device   the volumes already on the GPU: DeviceEngine.filter per volume vs DeviceEngine.filter_batch
  e2e      host arrays in, host results out: FlowDenoising(1, vol).filter per volume vs filter_volumes
It records ms per volume and Mvoxel/s (median over the rounds), library launches per volume (fdn_launch_count), the
sub-batch size filter_batch used, whether the results of the two routes are equal (SHA-256 of the Z+Y+X volumes), and
the GPU's name and power limit. Every default batch (bytes_per_batch in the record) is larger than the 126 MB L2 of a
B200, so the rounds do not run from L2.
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

SIZES = ["256x64x64x64", "64x96x96x96", "32x128x128x128", "8x64x256x256"]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power = [s.strip() for s in out[0].split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:     # the record says why instead of guessing
        return {"error": repr(e)}


def sha(arrs):
    h = hashlib.sha256()
    for a in arrs:
        h.update(np.ascontiguousarray(a, np.float32).tobytes())
    return h.hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "batch_bench.json"))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--sizes", nargs="+", default=SIZES)
    args = ap.parse_args()

    import torch
    from flowdenoising_b200 import flowdenoising as fd
    from flowdenoising_b200.engine import FlowParams, gaussian_kernel

    if not torch.cuda.is_available():
        raise SystemExit("batch_bench: no CUDA device (timings are only meaningful on the GPU)")
    eng = fd._get_engine()
    lib = eng.lib
    ks = [gaussian_kernel(2.0)] * 3
    flow = FlowParams()
    rec = {"gpu": gpu_info(), "torch": torch.__version__, "sigma": 2.0, "flow": vars(flow), "rounds": args.rounds,
           "sizes": []}
    print(json.dumps(rec["gpu"]), flush=True)

    def timed(fn):
        torch.cuda.synchronize()
        n0 = lib.fdn_launch_count()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0, lib.fdn_launch_count() - n0, out

    for size in args.sizes:
        B, Z, Y, X = (int(s) for s in size.split("x"))
        rng = np.random.default_rng(B * Z)
        host = (rng.random((B, Z, Y, X), dtype=np.float32) * 255).astype(np.float32)
        vols_list = [host[g] for g in range(B)]
        d = torch.from_numpy(host).cuda()
        vox = B * Z * Y * X

        def dev_loop():
            outs = []
            for g in range(B):
                outs.append(eng.filter(d[g], ks, flow)[1])
            return outs

        def dev_batch():
            return eng.filter_batch(d, ks, flow)[1]

        def e2e_loop():
            return [fd.FlowDenoising(1, vols_list[g].copy()).filter(ks) for g in range(B)]

        def e2e_batch():
            return fd.filter_volumes(vols_list, ks)

        # warm-up of every route and shape (module loads, workspaces, first-use attributes)
        eng.filter(d[0], ks, flow)
        eng.filter_batch(d, ks, flow)
        fd.FlowDenoising(1, vols_list[0].copy()).filter(ks)
        fd.filter_volumes(vols_list[:2], ks)
        torch.cuda.synchronize()

        t = {"device_loop": [], "device_batch": [], "e2e_loop": [], "e2e_batch": []}
        launches = {}
        hashes = {}
        for r in range(args.rounds):
            s, n, out = timed(dev_loop)
            t["device_loop"].append(s); launches["device_loop"] = n / B
            if r == 0:
                hashes["device_loop"] = sha([o.cpu().numpy() for o in out])
            del out
            s, n, out = timed(dev_batch)
            t["device_batch"].append(s); launches["device_batch"] = n / B
            sub = eng.sub_batch
            if r == 0:
                hashes["device_batch"] = sha([out[g].cpu().numpy() for g in range(B)])
            del out
            s, _n, out = timed(e2e_loop)
            t["e2e_loop"].append(s)
            if r == 0:
                hashes["e2e_loop"] = sha(out)
            del out
            s, _n, out = timed(e2e_batch)
            t["e2e_batch"].append(s)
            if r == 0:
                hashes["e2e_batch"] = sha(out)
            del out
        row = {"size": size, "batch": B, "shape": [Z, Y, X], "bytes_per_batch": 4 * vox, "sub_batch": sub,
               "launches_per_volume": launches,
               "results_equal": len(set(hashes.values())) == 1, "sha256": hashes, "seconds": t}
        for k, v in t.items():
            med = float(np.median(v))
            row[k] = {"ms_per_volume": 1e3 * med / B, "mvoxel_per_s": vox / med / 1e6,
                      "spread_ms_per_volume": [1e3 * min(v) / B, 1e3 * max(v) / B]}
        row["speedup_device"] = row["device_loop"]["ms_per_volume"] / row["device_batch"]["ms_per_volume"]
        row["speedup_e2e"] = row["e2e_loop"]["ms_per_volume"] / row["e2e_batch"]["ms_per_volume"]
        rec["sizes"].append(row)
        print(json.dumps({k: row[k] for k in ("size", "sub_batch", "launches_per_volume", "results_equal",
                                              "speedup_device", "speedup_e2e")}), flush=True)
        for k in t:
            print(f"  {k:13s} {row[k]['ms_per_volume']:9.3f} ms/vol {row[k]['mvoxel_per_s']:8.1f} Mvox/s", flush=True)
        del d
        eng.release_workspace()
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps({"written": args.out}))


if __name__ == "__main__":
    main()
