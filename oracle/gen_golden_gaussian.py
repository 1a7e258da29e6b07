#!/usr/bin/env python
"""Generate tests/golden/gaussian_window.npz: OpenCV's Farneback with the Gaussian window (OPTFLOW_FARNEBACK_GAUSSIAN)
and the FlowDenoising passes driven by it.

    python oracle/gen_golden_gaussian.py

The reference never sets the flag, so these fixtures come from live cv2 through the oracle's cv2-backed restatement of
the reference's slice loops (fd_oracle_gw.GaussianWindowDenoiser(backend="cv2"): fd_oracle.OracleDenoiser, the same
arm as bench.py --impl reference, with the flag). The cv2 / numpy versions that produced the file are stored in it.
Every input is regenerated from a seed, so the file holds SHA-256 digests only (the C oracle reproduces the arrays).

Contents:
  flows    for every case of CASES and both init modes (flags 256 and 256|4): "sha_<case>_f<flags>". Images:
           synthetic_volume((2, H, W), seed=H+W), slice 0 = prev, slice 1 = next; the initial flow of the 256|4 mode is
           init_flow(H, W).
  toy      the toy_of.npz volume (12x64x72, seed 21, sigmas 1.0/1.5/0.75, l=3 w=5) after Z, ZY, ZYX, chained
           ("toy_sha_Z", ...) and with --recompute_flow ("toyr_sha_Z", ...).
  cfg1     the cfg 1 volume (64x256x256, seed 0, noise 20, sigma 2, l=3 w=5) after each pass ("cfg1_sha_Z", ...).
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import fd_oracle as O  # noqa: E402
from oracle import fd_oracle_gw as GW  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "gaussian_window.npz")

# (H, W, levels, winsize, iterations, poly_n, poly_sigma)
CASES = [(256, 256, 3, 5, 3, 5, 1.2), (200, 333, 3, 5, 3, 5, 1.2), (256, 512, 5, 9, 3, 5, 1.2),
         (260, 300, 3, 5, 2, 7, 1.5), (64, 256, 3, 5, 3, 5, 1.2), (1024, 1024, 3, 5, 3, 5, 1.2),
         (130, 97, 3, 5, 4, 5, 1.2)]
CASES += [(H, W, 3, w, 3, 5, 1.2) for (H, W) in [(77, 150), (33, 40), (12, 300)] for w in (1, 2, 3, 4, 6, 8, 13, 21, 31)]
TOY_SIGMAS = (1.0, 1.5, 0.75)


def case_key(c):
    H, W, l, w, it, pn, ps = c
    return f"{H}x{W}_l{l}_w{w}_i{it}_n{pn}_s{ps}"


def case_images(H, W):
    v = O.synthetic_volume((2, H, W), seed=H + W, noise_sigma=10.0)
    return v[0], v[1]


def init_flow(H, W):
    """A smooth initial flow on a 1/64-pixel grid (exactly representable, the same on every host)."""
    y, x = np.mgrid[0:H, 0:W].astype(np.float64)
    f = np.stack([1.5 * np.sin(x / 17.0 + y / 23.0), 1.2 * np.cos(x / 19.0 - y / 29.0)], axis=-1)
    return (np.round(f * 64.0) / 64.0).astype(np.float32)


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def toy_volume():
    return O.synthetic_volume((12, 64, 72), seed=21, noise_sigma=8.0)


def cfg1_volume():
    return O.synthetic_volume((64, 256, 256), seed=0, noise_sigma=20.0)


def run_passes(vol, sigmas, recompute, P):
    """OracleDenoiser.filter step by step: [after Z, after ZY, after ZYX]."""
    o = GW.GaussianWindowDenoiser(P, vol.copy(), True, 3, 5, recompute_flow=recompute, backend="cv2")
    outs = []
    for axis, s in enumerate(sigmas):
        o.filter_along_axis(axis, O.get_gaussian_kernel(s))
        outs.append(o.filtered_vol.copy())
        o.vol[...] = o.filtered_vol[...]
    return outs


def main():
    import cv2
    d = {"versions": str(dict(cv2=cv2.__version__, numpy=np.__version__))}
    keys = []
    for c in CASES:
        H, W, l, w, it, pn, ps = c
        prev, nxt = case_images(H, W)
        for flags in (256, 256 | 4):
            flow = init_flow(H, W) if flags & 4 else None
            f = cv2.calcOpticalFlowFarneback(prev, nxt, flow, 0.5, l, w, it, pn, ps, flags)
            k = f"{case_key(c)}_f{flags}"
            keys.append(k)
            d[f"sha_{k}"] = sha(f)
    d["cases"] = np.array(CASES, dtype=np.float64)
    d["keys"] = np.array(keys)
    print("flows done")
    toy = toy_volume()
    for prefix, rec in (("toy", False), ("toyr", True)):
        outs = run_passes(toy, TOY_SIGMAS, rec, os.cpu_count())
        for name, o in zip(("Z", "ZY", "ZYX"), outs):
            d[f"{prefix}_sha_{name}"] = sha(o)
    print("toy done")
    vol = cfg1_volume()
    d["cfg1_input_sha256"] = sha(vol)
    outs = run_passes(vol, (2.0, 2.0, 2.0), False, os.cpu_count())
    for name, o in zip(("Z", "ZY", "ZYX"), outs):
        d[f"cfg1_sha_{name}"] = sha(o)
    print("cfg1 done")
    np.savez_compressed(OUT, **d)
    print(OUT, os.path.getsize(OUT))


if __name__ == "__main__":
    main()
