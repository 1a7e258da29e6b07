"""The reflect / mirror / nearest borders on the device. Contract (include/fdn_b200.h): a pass with border B equals,
bit for bit, the periodic pass on the volume padded by r slices along its axis with np.pad's mode for B, cropped back
to n. Checked for every axis x border x flow mode x dtype on toy shapes with an axis shorter than r and an axis of
length 1, against the C oracle, through chunked passes, the overlapped filter(), streaming, batches and the launch
log (a bordered pass runs exactly the launches of the wrapped one: no extra R images)."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import fd_oracle as O  # noqa: E402

pytestmark = pytest.mark.gpu

NP_MODE = {"reflect": "symmetric", "mirror": "reflect", "nearest": "edge"}   # SciPy name -> np.pad mode
BORDERS = list(NP_MODE)


@pytest.fixture(scope="module")
def eng():
    from flowdenoising_b200.engine import DeviceEngine
    torch.cuda.set_device(0)
    return DeviceEngine()


def _flows():
    from flowdenoising_b200.engine import FlowParams
    return {"chained": FlowParams(levels=2), "recompute": FlowParams(levels=2, use_prev_flow=False),
            "gaussian": FlowParams(levels=2, gaussian_window=True), "exact": None, "fast": None}


def _vol(shape, dtype, seed):
    v = O.synthetic_volume(shape, seed=seed, noise_sigma=8.0)
    if dtype == np.float32:
        return v
    info = np.iinfo(dtype)
    scale = 200.0 if info.bits == 16 else 1.0
    off = -100.0 if dtype == np.int8 else 0.0
    return np.clip(v * scale + off, info.min, info.max).astype(dtype)


def _pass(eng, vol, axis, k, flow, exact=True, border="wrap", chunk=None):
    d = torch.from_numpy(np.ascontiguousarray(vol)).cuda()
    o = torch.empty_like(d)
    eng.filter_along_axis(d, o, axis, k, flow, chunk, exact, border=border)
    return o.cpu().numpy()


def _padded_pass(eng, vol, axis, k, flow, border, exact=True):
    r = k.size // 2
    pad = [(0, 0)] * 3
    pad[axis] = (r, r)
    out = _pass(eng, np.pad(vol, pad, mode=NP_MODE[border]), axis, k, flow, exact)
    sl = [slice(None)] * 3
    sl[axis] = slice(r, r + vol.shape[axis])
    return out[tuple(sl)]


# (Z, Y, X): every axis longer and shorter than r = 4 (sigma 1), an axis of length 1, X % 4 == 0 and != 0 (the row
# kernels with and without 16-byte groups)
SHAPES = [(9, 20, 24), (3, 18, 22), (1, 12, 20), (10, 1, 3)]


@pytest.mark.parametrize("border", BORDERS)
@pytest.mark.parametrize("mode", ["chained", "recompute", "gaussian", "exact", "fast"])
def test_padding_identity_float32(eng, border, mode):
    flow = _flows()[mode]
    exact = mode != "fast"
    for i, shape in enumerate(SHAPES):
        vol = _vol(shape, np.float32, 10 + i)
        for sigma in ((1.0,) if flow is not None else (1.0, 0.75, 2.0)):    # no-OF: ring / generic kernels
            k = O.get_gaussian_kernel(sigma)
            for axis in range(3):
                got = _pass(eng, vol, axis, k, flow, exact, border)
                assert np.array_equal(got, _padded_pass(eng, vol, axis, k, flow, border, exact)), (shape, axis, sigma)


@pytest.mark.parametrize("border", BORDERS)
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.int16, np.int8])
def test_padding_identity_typed(eng, border, dtype):
    flows = [None] if dtype == np.int8 else [None, _flows()["chained"], _flows()["recompute"]]
    k = O.get_gaussian_kernel(1.0)
    for i, shape in enumerate(SHAPES[:3]):
        vol = _vol(shape, dtype, 30 + i)
        for flow in flows:
            for axis in range(3):
                got = _pass(eng, vol, axis, k, flow, True, border)
                assert got.dtype == dtype
                assert np.array_equal(got, _padded_pass(eng, vol, axis, k, flow, border)), (shape, axis, flow)


@pytest.mark.parametrize("border", BORDERS)
def test_against_the_c_oracle_on_the_padded_volume(eng, border):
    """The bordered pass is the reference's filter_along_{Z,Y,X} (C restatement) run on the np.pad-ed volume."""
    from flowdenoising_b200.engine import FlowParams
    vol = _vol((6, 20, 24), np.float32, 5)
    k = O.get_gaussian_kernel(1.0)
    r = k.size // 2
    for axis in range(3):
        pad = [(0, 0)] * 3
        pad[axis] = (r, r)
        padded = np.pad(vol, pad, mode=NP_MODE[border])
        sl = [slice(None)] * 3
        sl[axis] = slice(r, r + vol.shape[axis])
        for use_of in (True, False):
            o = O.OracleDenoiser(1, padded.copy(), use_OF=use_of, l=2, w=5, backend="c")
            o.filter_along_axis(axis, k, indices=range(r, r + vol.shape[axis]))
            got = _pass(eng, vol, axis, k, FlowParams(levels=2) if use_of else None, True, border)
            assert np.array_equal(got, o.filtered_vol[tuple(sl)]), (axis, use_of)


@pytest.mark.parametrize("border", BORDERS)
def test_chunked_and_windowed_passes_equal_the_whole_pass(eng, border):
    from flowdenoising_b200 import _lib
    from flowdenoising_b200.engine import DeviceEngine, FlowParams, border_code
    vol = _vol((23, 16, 20), np.float32, 7)
    k = O.get_gaussian_kernel(1.0)
    flow = FlowParams(levels=2)
    whole = _pass(eng, vol, 0, k, flow, border=border)
    for chunk in (1, 5, 9):   # 9 + 2r < 23: chunks without the whole-axis R cache
        assert np.array_equal(_pass(eng, vol, 0, k, flow, border=border, chunk=chunk), whole), chunk
    small = DeviceEngine(workspace_limit_bytes=eng.lib.fdn_workspace_bytes(
        _lib.View(23, 23, 0, 1, 16, 20, 320, 20, 320, 20), k.size, flow.c_struct(), 3))
    assert np.array_equal(_pass(small, vol, 0, k, flow, border=border), whole)
    # windows of the bordered axis (the overlapped filter's head and tail calls)
    d = torch.from_numpy(vol).cuda()
    o = torch.empty_like(d)
    for h0, h1 in ((0, 3), (3, 20), (20, 23)):
        v = _lib.View(23, h1 - h0, h0, border_code(border), 16, 20, 320, 20, 320, 20)
        eng.filter_view(d, o[h0:], v, k, flow)
    assert np.array_equal(o.cpu().numpy(), whole)


@pytest.mark.parametrize("border", BORDERS)
def test_overlapped_filter_equals_the_plain_sequence(border, monkeypatch):
    from flowdenoising_b200 import flowdenoising as fd
    vol = _vol((40, 64, 72), np.float32, 8)
    kernels = [O.get_gaussian_kernel(1.0)] * 3
    monkeypatch.setattr(fd, "_OVERLAP_MIN_BYTES", 1)
    a = fd.FlowDenoising(1, vol.copy(), l=2)
    a.border = border
    assert a._overlap_plan(torch, [np.asarray(k) for k in kernels]) is not None
    res_a, zy_a = a.filter(kernels).copy(), a.vol.copy()
    monkeypatch.setattr(fd, "_OVERLAP_MIN_BYTES", 1 << 60)
    b = fd.FlowDenoising(1, vol.copy(), l=2)
    b.border = border
    res_b = b.filter(kernels)
    assert np.array_equal(res_a, res_b) and np.array_equal(zy_a, b.vol)
    # and each pass of it is the padded pass
    from flowdenoising_b200.engine import DeviceEngine
    e = DeviceEngine()
    z = _padded_pass(e, vol, 0, kernels[0], a._flow(), border)
    zy = _padded_pass(e, z, 1, kernels[1], a._flow(), border)
    assert np.array_equal(zy, zy_a)
    assert np.array_equal(_padded_pass(e, zy, 2, kernels[2], a._flow(), border), res_a)


@pytest.mark.parametrize("border", BORDERS)
@pytest.mark.parametrize("typed", [False, True])
def test_streaming_equals_in_core(eng, border, typed):
    from flowdenoising_b200.engine import FlowParams
    from flowdenoising_b200.streaming import StreamingDenoiser
    vol = _vol((11, 18, 20), np.uint16 if typed else np.float32, 9)
    kernels = [O.get_gaussian_kernel(1.0)] * 3
    for flow in (FlowParams(levels=2), None):
        d = torch.from_numpy(vol).cuda()
        zy_ref, zyx_ref = (t.cpu().numpy() for t in eng.filter(d, kernels, flow, border=border))
        for lanes in ([0], [0, 0]):
            sd = StreamingDenoiser(flow, border=border, slab_slices=3, devices=lanes, keep_dtype=typed)
            zy, zyx = sd.filter(vol.copy(), kernels)
            assert np.array_equal(zy, zy_ref) and np.array_equal(zyx, zyx_ref), (flow is not None, lanes)


@pytest.mark.parametrize("border", BORDERS)
def test_module_surface_in_core_streamed_and_sliced(border):
    """GaussianDenoising / FlowDenoising with border: in core, streamed (forced) and the per-slice entry points agree."""
    from flowdenoising_b200 import flowdenoising as fd
    vol = _vol((7, 16, 20), np.float32, 11)
    kernels = [O.get_gaussian_kernel(1.0)] * 3
    for typed in (False, True):
        v = vol.astype(np.uint8) if typed else vol
        ref = fd.FlowDenoising(1, v.copy(), l=2, keep_dtype=typed)
        ref.border = border
        res = ref.filter(kernels).copy()
        st = fd.FlowDenoising(1, v.copy(), l=2, keep_dtype=typed)
        st.border, st.streaming, st.slab_slices = border, True, 2
        assert np.array_equal(st.filter(kernels), res), typed
    one = fd.FlowDenoising(1, vol.copy(), l=2)
    one.border = border
    one.filter_along_Y(kernels[1])
    sl = fd.FlowDenoising(1, vol.copy(), l=2)
    sl.border = border
    for y in (0, 1, 15):
        sl.filter_along_Y_slice(y, kernels[1])
    sl.filter_along_Y_chunk(1, 5, 2, kernels[1])        # slices 7 .. 11
    for y in (0, 1, 15, 7, 11):
        assert np.array_equal(sl.filtered_vol[:, y], one.filtered_vol[:, y]), y


@pytest.mark.parametrize("border", BORDERS)
def test_filter_volumes_equals_the_single_volume_path(border):
    from flowdenoising_b200 import flowdenoising as fd
    vols = [_vol((6, 16, 20), np.float32, 40 + i) for i in range(3)] + [_vol((1, 8, 12), np.float32, 50)]
    kernels = [O.get_gaussian_kernel(1.0)] * 3
    for no_of in (False, True):
        res = fd.filter_volumes(vols, kernels, l=2, no_OF=no_of, border=border)
        for v, r in zip(vols, res):
            one = fd.GaussianDenoising(1, v.copy()) if no_of else fd.FlowDenoising(1, v.copy(), l=2)
            one.border = border
            assert np.array_equal(r, one.filter(kernels)), no_of


def _launch_log(lib, fn):
    lib.fdn_launch_log_enable(1)
    fn()
    torch.cuda.synchronize()
    names = [lib.fdn_launch_log_name(i).decode() for i in range(lib.fdn_launch_log_count())]
    lib.fdn_launch_log_enable(0)
    return names


@pytest.mark.parametrize("border", BORDERS)
def test_bordered_launches_equal_the_wrapped_ones(eng, border):
    """Same kernels in the same order and numbers: the bordered pass builds no extra pyramid / polynomial images."""
    from flowdenoising_b200.engine import FlowParams
    vol = _vol((12, 24, 28), np.float32, 12)
    d = torch.from_numpy(vol).cuda()
    o = torch.empty_like(d)
    k = O.get_gaussian_kernel(1.0)
    for flow in (FlowParams(levels=2), FlowParams(levels=2, gaussian_window=True), None):
        for axis in range(3):
            for exact in (True, False) if flow is None else (True,):
                run = lambda b: _launch_log(eng.lib, lambda: eng.filter_along_axis(d, o, axis, k, flow, None, exact,
                                                                                  border=b))
                assert run(border) == run("wrap"), (axis, flow is not None, exact)
        bat = torch.from_numpy(np.stack([vol] * 3)).cuda()
        run = lambda b: _launch_log(eng.lib, lambda: eng.filter_batch(bat, [k] * 3, flow, border=b))
        assert run(border) == run("wrap")


def test_wrap_launch_log_of_a_cfg1_sized_pass_is_unchanged(eng):
    """The periodic pass keeps its launch sequence: the names of the parent's Z pass at a cfg-1-like shape."""
    from flowdenoising_b200.engine import FlowParams
    vol = _vol((24, 256, 256), np.float32, 13)
    d = torch.from_numpy(vol).cuda()
    o = torch.empty_like(d)
    k = O.get_gaussian_kernel(2.0)
    names = _launch_log(eng.lib, lambda: eng.filter_along_axis(d, o, 0, k, FlowParams()))
    r = k.size // 2
    # 4 pyramid levels of every slice (rows, cols, resize above level 0, polyexp), then per chain step one Farneback
    # over both chains (flow down-scale for chained flows, per level: iterations, upsample) and one warp
    assert names.count("k_warp_pair") == r and names.count("k_acc_finish") == 1
    assert names[-1] == "k_acc_finish"
    wrap = names
    for b in BORDERS:
        assert _launch_log(eng.lib, lambda: eng.filter_along_axis(d, o, 0, k, FlowParams(), border=b)) == wrap
