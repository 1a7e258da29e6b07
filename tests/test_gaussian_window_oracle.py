"""CPU checks of the Gaussian window (OPTFLOW_FARNEBACK_GAUSSIAN, flag 256): the C oracle against live cv2 and the
committed fixtures (tests/golden/gaussian_window.npz, oracle/gen_golden_gaussian.py; the oracle is
oracle/fd_oracle_gw.*), the oracle's two backends against
each other, and the flag's plumbing through the C ABI structure and the Python / CLI surface. No GPU needed."""
import ctypes as C
import hashlib

import numpy as np
import pytest

from oracle import fd_oracle as O
from oracle import fd_oracle_gw as GW
from oracle import gen_golden_gaussian as G


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def oracle_flow(case, flags):
    H, W, l, w, it, pn, ps = case
    prev, nxt = G.case_images(H, W)
    flow = G.init_flow(H, W) if flags & 4 else None
    return GW.farneback_c(prev, nxt, flow, l, w, it, pn, ps, flags=flags)


@pytest.mark.parametrize("case", G.CASES, ids=G.case_key)
def test_oracle_equals_golden(golden, case):
    g = golden("gaussian_window.npz")
    for flags in (256, 256 | 4):
        k = f"{G.case_key(case)}_f{flags}"
        got = oracle_flow(case, flags)
        assert sha(got) == str(g[f"sha_{k}"]), k


@pytest.mark.parametrize("case", G.CASES, ids=G.case_key)
def test_oracle_equals_live_cv2(case):
    cv2 = pytest.importorskip("cv2")
    H, W, l, w, it, pn, ps = case
    prev, nxt = G.case_images(H, W)
    for flags in (cv2.OPTFLOW_FARNEBACK_GAUSSIAN, cv2.OPTFLOW_FARNEBACK_GAUSSIAN | cv2.OPTFLOW_USE_INITIAL_FLOW):
        init = G.init_flow(H, W) if flags & 4 else None
        ref = cv2.calcOpticalFlowFarneback(prev, nxt, None if init is None else init.copy(), 0.5, l, w, it, pn, ps, flags)
        assert np.array_equal(oracle_flow(case, flags), ref), flags


def test_even_winsize_is_the_next_odd_window():
    """m = winsize // 2 fixes the Gaussian window: 2m and 2m + 1 give the same flow (not so for the box window)."""
    case = (77, 150, 3, 8, 3, 5, 1.2)
    odd = (77, 150, 3, 9, 3, 5, 1.2)
    assert np.array_equal(oracle_flow(case, 256), oracle_flow(odd, 256))
    prev, nxt = G.case_images(77, 150)
    assert not np.array_equal(O.farneback_c(prev, nxt, None, 3, 8), O.farneback_c(prev, nxt, None, 3, 9))


def test_gaussian_and_box_flows_differ():
    prev, nxt = G.case_images(77, 150)
    box = O.farneback_c(prev, nxt, None, 3, 5, flags=0)
    assert np.array_equal(GW.farneback_c(prev, nxt, None, 3, 5, flags=0), box)      # flag unset: the box window
    gauss = GW.farneback_c(prev, nxt, None, 3, 5, flags=256)
    assert np.mean(box != gauss) > 0.5
    R0, R1 = O.polyexp(prev), O.polyexp(nxt)
    M = O.update_matrices(R0, R1, np.zeros((77, 150, 2), np.float32))
    assert not np.array_equal(GW.gauss_blur_solve(M, 5), O.blur_solve(M, 5))


@pytest.mark.parametrize("recompute", [False, True])
def test_oracle_backends_agree_on_toy(golden, recompute):
    """OracleDenoiser, Gaussian window: the C backend equals the cv2 backend, and both equal the fixture."""
    pytest.importorskip("cv2")
    g = golden("gaussian_window.npz")
    toy = G.toy_volume()
    outs = {}
    for backend in ("cv2", "c"):
        o = GW.GaussianWindowDenoiser(4, toy.copy(), True, 3, 5, recompute_flow=recompute, backend=backend)
        res = []
        for axis, s in enumerate(G.TOY_SIGMAS):
            o.filter_along_axis(axis, O.get_gaussian_kernel(s))
            res.append(o.filtered_vol.copy())
            o.vol[...] = o.filtered_vol[...]
        outs[backend] = res
    prefix = "toyr" if recompute else "toy"
    for name, a, b in zip(("Z", "ZY", "ZYX"), outs["cv2"], outs["c"]):
        assert np.array_equal(a, b), name
        assert sha(b) == str(g[f"{prefix}_sha_{name}"]), name


def test_flow_axis_c_takes_the_flag(golden):
    g = golden("gaussian_window.npz")
    toy = G.toy_volume()
    k = O.get_gaussian_kernel(G.TOY_SIGMAS[0])
    assert sha(GW.flow_axis_c(toy, 0, k)) == str(g["toy_sha_Z"])
    assert np.array_equal(GW.flow_axis_c(toy, 0, k, flags=0), O.flow_axis_c(toy, 0, k))
    assert sha(O.flow_axis_c(toy, 0, k)) != str(g["toy_sha_Z"])


def test_of_params_flags_field():
    from flowdenoising_b200 import _lib
    from flowdenoising_b200.engine import FlowParams
    assert C.sizeof(_lib.OfParams) == 32
    assert _lib.OfParams.flags.offset == 28
    assert _lib.OfParams(3, 5, 3, 5, 1.2, 1).flags == 0
    assert FlowParams().c_struct().flags == 0
    assert FlowParams(gaussian_window=True).c_struct().flags == 256 == _lib.FARNEBACK_GAUSSIAN


def test_unknown_flags_are_rejected():
    from flowdenoising_b200 import _lib
    lib = _lib.load()
    assert lib.fdn_version() == 101
    v = _lib.View(64, 64, 0, 1, 256, 256, 65536, 256, 65536, 256)
    for flags in (4, 1, 512, 256 | 4):
        p = _lib.OfParams(3, 5, 3, 5, 1.2, 1, flags)
        assert lib.fdn_workspace_bytes(C.byref(v), 17, C.byref(p), 0) == 0 and b"flags" in lib.fdn_last_error()
        assert lib.fdn_farneback(1, 1, 1, 1, 64, 64, C.byref(p), 1, 1 << 40, None) == 1
    p = _lib.OfParams(3, 5, 3, 5, 1.2, 1, 256)
    assert lib.fdn_workspace_bytes(C.byref(v), 17, C.byref(p), 0) > 0
    assert lib.fdn_farneback_workspace_bytes(4, 256, 256, C.byref(p)) > 0


def test_cli_and_api_defaults():
    import inspect
    from flowdenoising_b200 import flowdenoising as fd
    assert fd.build_parser().parse_args([]).gaussian_window is False
    assert fd.build_parser().parse_args(["--gaussian_window"]).gaussian_window is True
    help_text = fd.build_parser().format_help()
    assert "--gaussian_window" in help_text and "not a speed switch" in " ".join(help_text.split())
    for f in (fd.get_flow_with_prev_flow, fd.get_flow_without_prev_flow, fd.FlowDenoising.__init__):
        assert inspect.signature(f).parameters["gaussian_window"].default is False
    obj = fd.FlowDenoising(1, np.zeros((4, 8, 8), np.float32), gaussian_window=True)
    assert obj._flow_params.gaussian_window and obj._flow_params.c_struct().flags == 256
    assert fd.FlowDenoising(1, np.zeros((4, 8, 8), np.float32))._flow_params.c_struct().flags == 0
