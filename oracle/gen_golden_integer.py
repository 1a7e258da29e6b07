#!/usr/bin/env python
"""Generate tests/golden/integer_volumes.npz: the reference's passes on integer volumes, from live cv2.

    python oracle/gen_golden_integer.py

The reference keeps an integer volume's dtype through every pass (SURVEY App. B Q3). fd_oracle.OracleDenoiser with the
cv2 backend restates its slice loops with the same buffers (``filtered_vol = zeros_like(vol)``, integer cv2.remap,
float32 accumulation, truncating store, integer copy-back between passes), so it produces what the reference produces.
Every input is regenerated from a seed (fd_oracle_int.integer_volume), so the file holds SHA-256 digests only. The
cv2 / numpy versions that produced it are stored in it.

Cases ("<case>_sha_Z", "<case>_sha_ZY", "<case>_sha_ZYX": the result after each pass of filter()):
  toy volume (8, 64, 72), seed 21, sigmas (1.0, 1.5, 0.75), -l 3 -w 5, for uint8, uint16 and int16:
    "<dtype>_of"       chained flows (the default)
    "<dtype>_ofr"      --recompute_flow
    "<dtype>_noof"     --no_OF
  "int8_noof"          int8 without optical flow (cv2.remap rejects int8, so the OF path cannot run on it)
  "uint8_gw"           uint8, chained flows with the Gaussian window (OPTFLOW_FARNEBACK_GAUSSIAN), -w 9
  "cfg1_uint8"         the cfg 1 shape (64, 256, 256) as uint8, seed 0, noise 20, sigma 2, chained flows
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import fd_oracle as O  # noqa: E402
from oracle import fd_oracle_int as I  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "integer_volumes.npz")

TOY_SHAPE = (8, 64, 72)
TOY_SEED = 21
TOY_SIGMAS = (1.0, 1.5, 0.75)
CFG1_SHAPE = (64, 256, 256)
CFG1_SEED = 0
CFG1_NOISE = 20.0
CFG1_SIGMA = 2.0

# name -> (dtype, shape, seed, noise, sigmas, mode, winsize); mode: "of", "ofr" (recompute), "noof", "gw"
CASES = {}
for _dt in ("uint8", "uint16", "int16"):
    for _mode in ("of", "ofr", "noof"):
        CASES[f"{_dt}_{_mode}"] = (_dt, TOY_SHAPE, TOY_SEED, 10.0, TOY_SIGMAS, _mode, 5)
CASES["int8_noof"] = ("int8", TOY_SHAPE, TOY_SEED, 10.0, TOY_SIGMAS, "noof", 5)
CASES["uint8_gw"] = ("uint8", TOY_SHAPE, TOY_SEED, 10.0, TOY_SIGMAS, "gw", 9)
CASES["cfg1_uint8"] = ("uint8", CFG1_SHAPE, CFG1_SEED, CFG1_NOISE, (CFG1_SIGMA,) * 3, "of", 5)


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def case_volume(name):
    dt, shape, seed, noise, _s, _m, _w = CASES[name]
    return I.integer_volume(shape, dt, seed, noise)


def denoiser(name, vol, backend, threads=os.cpu_count() or 1):
    """The oracle driver of a case (vol is used in place, like the reference's)."""
    _dt, _shape, _seed, _noise, _s, mode, w = CASES[name]
    if mode == "gw":
        return I.IntegerGaussianWindowDenoiser(threads, vol, use_OF=True, w=w, backend=backend)
    return I.IntegerDenoiser(threads, vol, use_OF=mode != "noof", w=w, recompute_flow=mode == "ofr", backend=backend)


def run_case(name, backend="cv2"):
    """(Z, ZY, ZYX) results of the case's filter(), each in the volume's dtype."""
    sigmas = CASES[name][4]
    ks = [O.get_gaussian_kernel(s) for s in sigmas]
    d = denoiser(name, case_volume(name), backend)
    d.filter_along_Z(ks[0])
    z = d.filtered_vol.copy()
    d.vol[...] = d.filtered_vol
    d.filter_along_Y(ks[1])
    zy = d.filtered_vol.copy()
    d.vol[...] = d.filtered_vol
    d.filter_along_X(ks[2])
    return z, zy, d.filtered_vol.copy()


def main():
    import cv2
    out = {"cv2_version": np.array(cv2.__version__), "numpy_version": np.array(np.__version__)}
    for name, (dt, shape, seed, noise, sigmas, mode, w) in CASES.items():
        out[f"{name}_input_sha"] = np.array(sha(case_volume(name)))
        z, zy, zyx = run_case(name, "cv2")
        for tag, a in (("Z", z), ("ZY", zy), ("ZYX", zyx)):
            assert a.dtype == np.dtype(dt)
            out[f"{name}_sha_{tag}"] = np.array(sha(a))
        print(name, "done", flush=True)
    np.savez_compressed(OUT, **out)
    print("wrote", OUT)


if __name__ == "__main__":
    main()
