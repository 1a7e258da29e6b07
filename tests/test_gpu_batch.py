"""GPU tests of batched filtering (fdn_filter_axis_batch / fdn_gauss_axis_batch, DeviceEngine.filter_batch,
filter_volumes, --inputs): volume g of a batch equals the single-volume path on that volume alone, bit for bit, in every
float32 mode; the reference's golden outputs and the C oracle hold inside a batch; a batch takes the launches of one
volume; sub-batches, the chunked fallback, launches of more than 65535 image pairs and the CLI."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import fd_oracle as O

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from flowdenoising_b200 import _lib  # noqa: E402
from flowdenoising_b200.engine import DeviceEngine, FlowParams  # noqa: E402

FDN_ERR_INVALID = 1   # include/fdn_b200.h


@pytest.fixture(scope="module")
def eng():
    return DeviceEngine()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def batch_of(shape, n, seed):
    return np.stack([O.synthetic_volume(shape, seed=seed + i, noise_sigma=8.0) for i in range(n)]).astype(np.float32)


def single(eng, vol, kernels, flow, exact=True):
    zy, zyx = eng.filter(dev(vol), kernels, flow, exact=exact)
    return zy.cpu().numpy(), zyx.cpu().numpy()


def assert_batch_equals_single(eng, vols, kernels, flow, exact=True, sample=None):
    zy, zyx = eng.filter_batch(dev(vols), kernels, flow, exact=exact)
    zy, zyx = zy.cpu().numpy(), zyx.cpu().numpy()
    for g in (range(len(vols)) if sample is None else sample):
        s_zy, s_zyx = single(eng, vols[g], kernels, flow, exact)
        assert np.array_equal(zy[g], s_zy), g
        assert np.array_equal(zyx[g], s_zyx), g


MODES = {
    "of_chained": FlowParams(),
    "recompute_flow": FlowParams(use_prev_flow=False),
    "gaussian_window_9": FlowParams(winsize=9, gaussian_window=True),
}


# a width that is no multiple of 4 (scalar kernels) and an axis shorter than the kernel (the wrap applies twice)
@pytest.mark.parametrize("shape", [(17, 33, 45), (6, 40, 64)])
@pytest.mark.parametrize("mode", sorted(MODES))
def test_batch_equals_single_volume_path_with_flow(eng, shape, mode):
    kernels = [O.get_gaussian_kernel(2.0), O.get_gaussian_kernel(1.0), O.get_gaussian_kernel(1.5)]
    assert_batch_equals_single(eng, batch_of(shape, 5, seed=100), kernels, MODES[mode])


@pytest.mark.parametrize("shape", [(17, 33, 45), (6, 40, 64)])
@pytest.mark.parametrize("exact", [True, False])
def test_batch_equals_single_volume_path_without_flow(eng, shape, exact):
    kernels = [O.get_gaussian_kernel(2.0), O.get_gaussian_kernel(0.75), O.get_gaussian_kernel(1.5)]  # ring, generic
    assert_batch_equals_single(eng, batch_of(shape, 5, seed=200), kernels, None, exact=exact)


def _z_pass_batch(eng, vols, k, flow):
    """The Z pass alone through fdn_filter_axis_batch."""
    B, Z, Y, X = vols.shape
    d = dev(vols)
    out = torch.empty_like(d)
    v = eng._batch_views(Z, Y, X)[0]
    kk = np.ascontiguousarray(k, np.float64)
    ofp = flow.c_struct()
    nbytes = eng.lib.fdn_workspace_bytes_batch(C.byref(v), B, kk.size, C.byref(ofp))
    ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    _lib.check(eng.lib.fdn_filter_axis_batch(d.data_ptr(), out.data_ptr(), C.byref(v), B, Z * Y * X, Z * Y * X,
                                             kk.ctypes.data_as(C.POINTER(C.c_double)), kk.size, C.byref(ofp),
                                             ws.data_ptr(), nbytes, None))
    return out.cpu().numpy()


def test_reference_golden_inside_a_batch(eng, golden):
    g = golden("toy_of.npz")
    vol = g["vol"].astype(np.float32)
    vols = np.stack([O.synthetic_volume(vol.shape, seed=7, noise_sigma=8.0), vol,
                     O.synthetic_volume(vol.shape, seed=8, noise_sigma=8.0)]).astype(np.float32)
    kernels = [O.get_gaussian_kernel(float(s)) for s in g["sigmas"]]
    p = FlowParams(int(g["l"]), int(g["w"]))
    assert np.array_equal(_z_pass_batch(eng, vols, kernels[0], p)[1], g["Z"])
    zy, zyx = eng.filter_batch(dev(vols), kernels, p)
    assert np.array_equal(zy[1].cpu().numpy(), g["ZY"])
    assert np.array_equal(zyx[1].cpu().numpy(), g["ZYX"])
    g = golden("toy_of_recompute.npz")
    vols[1] = g["vol"].astype(np.float32)
    p = FlowParams(int(g["l"]), int(g["w"]), use_prev_flow=False)
    assert np.array_equal(_z_pass_batch(eng, vols, O.get_gaussian_kernel(float(g["sigmas"][0])), p)[1], g["Z"])


def test_batch_equals_the_c_oracle(eng):
    vols = batch_of((7, 36, 44), 3, seed=300)
    kernels = [O.get_gaussian_kernel(1.0), O.get_gaussian_kernel(0.75), O.get_gaussian_kernel(1.0)]
    zy, zyx = eng.filter_batch(dev(vols), kernels, FlowParams(levels=2, winsize=5))
    for g in range(3):
        o = O.OracleDenoiser(1, vols[g].copy(), use_OF=True, l=2, w=5, backend="c")
        assert np.array_equal(zyx[g].cpu().numpy(), o.filter(kernels)), g
        assert np.array_equal(zy[g].cpu().numpy(), o.vol), g


def _launches(eng, vols, kernels, flow):
    lib = eng.lib
    d = dev(vols)
    eng.filter_batch(d, kernels, flow)            # warm: workspace allocated, first-use attributes set
    torch.cuda.synchronize()
    n0 = lib.fdn_launch_count()
    lib.fdn_launch_log_enable(1)
    eng.filter_batch(d, kernels, flow)
    torch.cuda.synchronize()
    names = [lib.fdn_launch_log_name(i) for i in range(lib.fdn_launch_log_count())]
    lib.fdn_launch_log_enable(0)
    return lib.fdn_launch_count() - n0, names, eng.sub_batch


@pytest.mark.parametrize("flow", [FlowParams(), None], ids=["of", "no_of"])
def test_a_batch_takes_the_launches_of_one_volume(eng, flow):
    kernels = [O.get_gaussian_kernel(2.0)] * 3
    vols = batch_of((32, 64, 64), 8, seed=400)
    n8, names8, sb = _launches(eng, vols, kernels, flow)
    assert sb == 8
    n1, names1, _ = _launches(eng, vols[:1], kernels, flow)
    assert n8 == n1 and names8 == names1 and n1 > 0


def test_sub_batches_and_the_chunked_fallback(eng):
    kernels = [O.get_gaussian_kernel(1.0)] * 3
    flow = FlowParams()
    ofp = flow.c_struct()
    vols = batch_of((12, 40, 48), 7, seed=500)
    views = DeviceEngine._batch_views(12, 40, 48)
    need = lambda b: max(eng.lib.fdn_workspace_bytes_batch(C.byref(v), b, 9, C.byref(ofp)) for v in views)
    small = DeviceEngine(workspace_limit_bytes=need(3))
    zy, zyx = small.filter_batch(dev(vols), kernels, flow)
    assert small.sub_batch == 3
    for g in range(7):
        s_zy, s_zyx = single(eng, vols[g], kernels, flow)
        assert np.array_equal(zy[g].cpu().numpy(), s_zy) and np.array_equal(zyx[g].cpu().numpy(), s_zyx), g
    # not even one whole volume fits: each volume goes through the chunked single-volume path
    chunked = max(eng.lib.fdn_workspace_bytes(C.byref(v), 9, C.byref(ofp), 2) for v in views)
    assert chunked < need(1)
    tiny = DeviceEngine(workspace_limit_bytes=chunked)
    zy, zyx = tiny.filter_batch(dev(vols[:2]), kernels, flow)
    assert tiny.sub_batch == 0
    for g in range(2):
        s_zy, s_zyx = single(eng, vols[g], kernels, flow)
        assert np.array_equal(zy[g].cpu().numpy(), s_zy) and np.array_equal(zyx[g].cpu().numpy(), s_zyx), g


def test_more_than_65535_image_pairs_per_launch(eng):
    """2100 volumes of 16 x 32 x 32: 67 200 image pairs per launch of the Z and Y passes (split over blockIdx.z)."""
    kernels = [O.get_gaussian_kernel(1.0)] * 3
    vols = batch_of((16, 32, 32), 2100, seed=600)
    assert_batch_equals_single(eng, vols, kernels, FlowParams(), sample=[0, 1, 1037, 2098, 2099])


@pytest.mark.parametrize("sigma", [2.0, 0.75], ids=["ring", "generic"])
def test_no_of_batch_larger_than_one_launch(eng, sigma):
    """70 000 volumes of 3 x 4 x 8: more volumes x slices (or segments) than blockIdx.z holds, and a Y pass of more
    than 65535 rows."""
    rng = np.random.default_rng(7)
    vols = (rng.random((70000, 3, 4, 8)) * 255).astype(np.float32)
    kernels = [O.get_gaussian_kernel(sigma)] * 3
    assert_batch_equals_single(eng, vols, kernels, None, sample=[0, 21844, 21845, 43690, 65535, 69999])


def test_argument_checks_launch_nothing(eng):
    lib = eng.lib
    d = torch.zeros(4 * 16 * 8 * 8, device="cuda")
    ws = torch.empty(1 << 24, dtype=torch.uint8, device="cuda")
    whole = _lib.View(16, 16, 0, 1, 8, 8, 64, 8, 64, 8)
    of = _lib.OfParams(3, 5, 3, 5, 1.2, 1, 0)
    k = (C.c_double * 257)(*([1.0 / 257] * 257))
    cases = [(whole, 0, 17, of), (whole, 2, 259, of), (whole, 2, 17, _lib.OfParams(3, 5, 0, 5, 1.2, 1, 0)),
             (_lib.View(16, 16, 0, 0, 8, 8, 64, 8, 64, 8), 2, 17, of), (_lib.View(16, 8, 4, 1, 8, 8, 64, 8, 64, 8), 2, 17, of)]
    torch.cuda.synchronize()
    n0 = lib.fdn_launch_count()
    for v, b, klen, p in cases:
        assert lib.fdn_filter_axis_batch(d.data_ptr(), d.data_ptr() + 4096, C.byref(v), b, 1024, 1024, k, klen,
                                         C.byref(p), ws.data_ptr(), ws.numel(), None) == FDN_ERR_INVALID
        if p is of:
            assert lib.fdn_gauss_axis_batch(d.data_ptr(), d.data_ptr() + 4096, C.byref(v), b, 1024, 1024, k, klen, 1,
                                            None) == FDN_ERR_INVALID
    assert lib.fdn_launch_count() == n0


def test_cli_inputs_equal_single_runs(tmp_path):
    from flowdenoising_b200 import flowdenoising as fd
    from flowdenoising_b200 import volume_io
    src = tmp_path / "in"
    os.makedirs(src)
    vols = {"a.mrc": O.synthetic_volume((10, 32, 40), seed=1), "b.mrc": O.synthetic_volume((10, 32, 40), seed=2),
            "c.mrc": O.synthetic_volume((8, 36, 28), seed=3), "d.tif": O.synthetic_volume((10, 32, 40), seed=4)}
    for name, v in vols.items():
        volume_io.write_volume(str(src / name), v.astype(np.float32))
    flags = ["-s", "1.5", "-l", "2"]
    assert fd.main(["--inputs"] + [str(src / n) for n in vols] + ["--output_dir", str(tmp_path / "out")] + flags) == 0
    for name in vols:
        one = str(tmp_path / ("single_" + name))
        assert fd.main(["-i", str(src / name), "-o", one] + flags) == 0
        a, b = volume_io.read_volume(str(tmp_path / "out" / name)), volume_io.read_volume(one)
        assert a.dtype == np.float32 and np.array_equal(a, b), name


@pytest.mark.parametrize("pad", [1, 2])
@pytest.mark.parametrize("axis", [0, 1])
def test_batch_strides_off_the_vector_alignment(eng, axis, pad):
    """Volumes packed `pad` elements apart (batch strides Z*Y*X + pad, X a multiple of 4, so every volume but the first
    is off the 16-byte grid): each volume equals the single-volume entry point on that volume alone, and nothing is
    written between the volumes."""
    from flowdenoising_b200.engine import gaussian_kernel
    B, Z, Y, X = 3, 9, 24, 32
    vs = Z * Y * X
    stride = vs + pad
    vols = batch_of((Z, Y, X), B, seed=700)
    flat_in = torch.zeros(B * stride, device="cuda")
    for g in range(B):
        flat_in[g * stride:g * stride + vs] = dev(vols[g]).view(-1)
    v = DeviceEngine._batch_views(Z, Y, X)[axis]
    k = np.ascontiguousarray(gaussian_kernel(1.0))
    kp = k.ctypes.data_as(C.POINTER(C.c_double))
    for flow, exact in ((FlowParams(), True), (None, True), (None, False)):
        flat_out = torch.full((B * stride,), float("nan"), device="cuda")
        if flow is not None:
            ofp = flow.c_struct()
            nbytes = eng.lib.fdn_workspace_bytes_batch(C.byref(v), B, k.size, C.byref(ofp))
            ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
            _lib.check(eng.lib.fdn_filter_axis_batch(flat_in.data_ptr(), flat_out.data_ptr(), C.byref(v), B, stride,
                                                     stride, kp, k.size, C.byref(ofp), ws.data_ptr(), nbytes, None))
        else:
            _lib.check(eng.lib.fdn_gauss_axis_batch(flat_in.data_ptr(), flat_out.data_ptr(), C.byref(v), B, stride,
                                                    stride, kp, k.size, int(exact), None))
        got = flat_out.cpu().numpy()
        for g in range(B):
            ref = torch.empty((Z, Y, X), device="cuda")
            eng.filter_along_axis(dev(vols[g]), ref, axis, k, flow, exact=exact)
            assert np.array_equal(got[g * stride:g * stride + vs].reshape(Z, Y, X), ref.cpu().numpy()), (flow, exact, g)
            assert np.isnan(got[g * stride + vs:(g + 1) * stride]).all(), (flow, exact, g)
