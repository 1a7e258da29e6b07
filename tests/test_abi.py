"""CPU-side checks: the C-ABI library builds/loads and exports every symbol include/fdn_b200.h declares; host-only
entry points (kernel taps, pyramid geometry) match the oracle / the reference's golden vectors. No GPU needed."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from flowdenoising_b200 import _lib, engine
from oracle import fd_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_symbols_exported():
    lib = _lib.load()
    hdr = open(os.path.join(ROOT, "include", "fdn_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b(fdn_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), f"{n} declared in fdn_b200.h but not exported"
        assert n in _lib.SIGNATURES, f"{n} has no ctypes signature"
    assert lib.fdn_version() >= 100


def test_gaussian_kernel_matches_reference(golden):
    g = golden("kernels.npz")
    for s in g["sigmas"]:
        np.testing.assert_allclose(engine.gaussian_kernel(float(s)), g[f"k_{s}"], rtol=4e-16, atol=0)
    with pytest.raises(ValueError):
        engine.gaussian_kernel(0.0)


def test_level_geometry_matches_oracle():
    for (H, W, l) in [(256, 256, 3), (64, 256, 3), (255, 255, 3), (1024, 1024, 5), (2048, 2048, 5), (260, 300, 3),
                      (12, 72, 3), (31, 500, 3), (100, 100, 0)]:
        assert engine.level_geometry(H, W, l) == O.level_geometry(H, W, l)


def test_bad_arguments_are_reported_not_crashed():
    lib = _lib.load()
    v = _lib.View(4, 4, 0, 1, 8, 8, 64, 8, 64, 8)
    k = (C.c_double * 2)(0.5, 0.5)
    rc = lib.fdn_gauss_axis(1, 1, C.byref(v), k, 2, 1, None)   # even kernel length; pointers never dereferenced
    assert rc == 1 and b"odd" in lib.fdn_last_error()
    p = _lib.OfParams(3, 99, 3, 5, 1.2, 1)
    assert lib.fdn_workspace_bytes(C.byref(v), 3, C.byref(p), 0) == 0 and b"winsize" in lib.fdn_last_error()
    with pytest.raises(ValueError):
        _lib.check(rc)


def test_workspace_layout_grows_with_chunk():
    """The exact pass workspace, its flow-iteration flags sized by the real strip count (not a fixed 64 per pair)."""
    lib = _lib.load()
    v = _lib.View(64, 64, 0, 1, 256, 256, 65536, 256, 65536, 256)
    p = _lib.OfParams(3, 5, 3, 5, 1.2, 1)
    a = lib.fdn_workspace_bytes(C.byref(v), 17, C.byref(p), 8)
    b = lib.fdn_workspace_bytes(C.byref(v), 17, C.byref(p), 0)
    assert 0 < a < b
    # all 64 slices cached once: R = 64 slots * 5 * (256^2 + 128^2 + 64^2 + 32^2) floats; both chain directions advance
    # together: 3 flow buffers of 2 * 64 pairs; the remapped forward neighbours wait in a stash of r = 8 chunk volumes;
    # + the scratch of the flow iteration for 128 pairs: ticket / finish counters, 3 * 128 dependency counters, the
    # flags + carries of the strip kernel (2 strips of 128 columns per image) and the carry packets of the
    # warp-specialised kernel (3 strips of <= 120 columns, 16 bytes per carry), all sized by level 0, the largest here
    R = 64 * 5 * (256 * 256 + 128 * 128 + 64 * 64 + 32 * 32) * 4
    flows = 3 * (128 * 256 * 256 * 2 * 4)
    stash = 8 * 64 * 256 * 256 * 4
    al = lambda v: (v + 255) // 256 * 256
    scratch = 256 + al(3 * 128 * 4) + 128 * 2 * 8 + 128 * 3 * 256 * 5 * 16 + 128 * 2 * 256 * 5 * 8
    assert b == R + flows + stash + scratch
