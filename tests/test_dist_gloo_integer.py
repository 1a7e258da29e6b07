"""Multi-rank host logic of flowdenoising_b200/dist.py on TYPED (integer) slabs, exercised on CPU with the gloo backend
at world sizes 2 and 3 (uneven slabs included).

The compute object is a typed CPU stand-in built on the integer ORACLE (test infrastructure): its filter_view is
fd_oracle_int.IntegerDenoiser with the C backend on the non-periodic halo slab, its copy3d / transpose_strided have the
NumPy semantics of the C-ABI contracts (include/fdn_b200.h) on buffers of any dtype. The gathered Z+Y and Z+Y+X results
of filter() and filter_host() must hash to the cv2 digests of tests/golden/integer_volumes.npz, and every tensor that an
exchange carries must be a byte view (NCCL has no 16-bit integer type). The GPU twin is tests/test_gpu_integer_sharded.py.
"""
import hashlib
import os
import socket

import numpy as np
import pytest

torch = pytest.importorskip("torch")
import torch.distributed as dist  # noqa: E402
import torch.multiprocessing as mp  # noqa: E402

from oracle import fd_oracle as O  # noqa: E402
from oracle import fd_oracle_int as I  # noqa: E402
from oracle import gen_golden_integer as G  # noqa: E402

TOY_CASES = [f"{dt}_{m}" for dt in ("uint8", "uint16", "int16") for m in ("of", "ofr", "noof")] + ["int8_noof"]
SENTINEL = 77


class TypedCpuOps:
    """Oracle-backed stand-in for DeviceEngine on typed slabs (same method contracts, CPU tensors)."""
    torch = torch

    def __init__(self):
        self.empty_dtypes = []

    def empty(self, shape, dtype=torch.float32):
        self.empty_dtypes.append(dtype)
        return torch.full(tuple(int(s) for s in shape), SENTINEL, dtype=dtype)

    @staticmethod
    def _flat(t):
        assert t.is_contiguous()
        return t.view(-1).numpy()

    def copy3d(self, src, src_off, in_sa, in_sb, b0, bw, c0, cw, dst, dst_off, out_sa, out_sb, A, B, C):
        assert src.dtype == dst.dtype
        s, d = self._flat(src), self._flat(dst)
        a = np.arange(A)[:, None, None]
        b = np.arange(B)[None, :, None]
        c = np.arange(C)[None, None, :]
        d[dst_off + a * out_sa + b * out_sb + c] = s[src_off + a * in_sa + ((b0 + b) % bw) * in_sb + (c0 + c) % cw]

    def transpose_strided(self, src, src_off, in_sn, in_sa, dst, dst_off, out_sn, out_sb, n, A, B):
        assert src.dtype == dst.dtype
        s, d = self._flat(src), self._flat(dst)
        i = np.arange(n)[:, None, None]
        a = np.arange(A)[None, :, None]
        b = np.arange(B)[None, None, :]
        d[dst_off + i * out_sn + b * out_sb + a] = s[src_off + i * in_sn + a * in_sa + b]

    def filter_view(self, d_in, d_out, v, kernel, flow, chunk=None, exact=True):
        assert d_in.dtype == d_out.dtype and d_in.dtype != torch.float32
        es = d_in.element_size()
        src = np.lib.stride_tricks.as_strided(self._flat(d_in), (v.n_in, v.H, v.W),
                                              (es * v.in_slice_stride, es * v.in_row_stride, es))
        dst = np.lib.stride_tricks.as_strided(self._flat(d_out), (v.n_out, v.H, v.W),
                                              (es * v.out_slice_stride, es * v.out_row_stride, es))
        assert not v.periodic and v.halo >= kernel.size // 2
        slab = np.ascontiguousarray(src)
        kw = {} if flow is None else dict(l=flow.levels, w=flow.winsize, recompute_flow=not flow.use_prev_flow)
        o = I.IntegerDenoiser(1, slab, use_OF=flow is not None, backend="c", **kw)
        for s in range(v.n_out):
            o.filter_slice(0, s + v.halo, kernel)       # never wraps: halo >= r on both sides
            dst[s] = o.filtered_vol[s + v.halo]


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def case_flow(name):
    from flowdenoising_b200.engine import FlowParams
    _dt, _shape, _seed, _noise, sigmas, mode, w = G.CASES[name]
    ks = [O.get_gaussian_kernel(s) for s in sigmas]
    return (None if mode == "noof" else FlowParams(3, w, 3, 5, 1.2, mode != "ofr")), ks


def _worker(rank, world, port, name, result_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    carried = []
    orig_p2p = dist.P2POp

    def p2p(op, tensor, *a, **kw):          # every exchange of dist.py goes through P2POp under gloo
        carried.append(tensor.dtype)
        return orig_p2p(op, tensor, *a, **kw)
    dist.P2POp = p2p
    try:
        from flowdenoising_b200.dist import DistributedDenoiser
        vol = G.case_volume(name)
        flow, kernels = case_flow(name)
        ops = TypedCpuOps()
        dd = DistributedDenoiser(ops, vol.shape, flow)
        zs, ze = dd.z_range
        zy, zyx = dd.filter(torch.from_numpy(vol[zs:ze].copy()), kernels, want_zy=True)
        assert zy.dtype == zyx.dtype == torch.from_numpy(vol).dtype
        np.save(os.path.join(result_dir, f"zy_{rank}.npy"), zy.numpy())
        np.save(os.path.join(result_dir, f"zyx_{rank}.npy"), zyx.numpy())
        out_host = torch.full((ze - zs,) + tuple(vol.shape[1:]), SENTINEL, dtype=zy.dtype)
        res = dd.filter_host(torch.from_numpy(vol[zs:ze].copy()), out_host, kernels)
        assert torch.equal(res, out_host)
        np.save(os.path.join(result_dir, f"zyxh_{rank}.npy"), out_host.numpy())
        # every buffer in the slab's dtype, every exchanged tensor a byte view
        assert set(ops.empty_dtypes) == {zy.dtype}, ops.empty_dtypes
        assert carried and set(carried) == {torch.uint8}, carried
    finally:
        dist.P2POp = orig_p2p
        dist.destroy_process_group()


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.mark.parametrize("world,name", [(2, c) for c in TOY_CASES] +
                         [(3, c) for c in ("uint8_of", "uint16_ofr", "int16_of", "int16_noof", "int8_noof")])
def test_distributed_typed_equals_golden(tmp_path, golden, world, name):
    """world 3 on the (8, 64, 72) toy volume: Z-slabs of 3, 3, 2 (r = 4: halos from several ranks), Y-slabs of 22, 21,
    21."""
    g = golden("integer_volumes.npz")
    mp.spawn(_worker, args=(world, _free_port(), name, str(tmp_path)), nprocs=world, join=True)
    dt = np.dtype(G.CASES[name][0])
    for tag, key in (("zy", "ZY"), ("zyx", "ZYX"), ("zyxh", "ZYX")):
        got = np.concatenate([np.load(tmp_path / f"{tag}_{r}.npy") for r in range(world)])
        assert got.dtype == dt and got.shape == G.CASES[name][1]
        assert sha(got) == str(g[f"{name}_sha_{key}"]), (name, tag)
