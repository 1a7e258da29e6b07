"""Multi-GPU slab sharding of the three passes (one process per GPU, torch.distributed / NCCL over NVLink).

Within a pass every output slice depends only on its 2r neighbour slices (src/flowdenoising.py:306-327), so each
pass shards its slice index into contiguous slabs with an r-slice PERIODIC halo (`% shape`, :312). Between passes
the slice orientation changes, so the volume is re-slabbed with an all-to-all (SURVEY.md §8e):

    input       rank g holds the Z-slab            vol[zs_g:ze_g, :, :]
    Z pass      halo exchange (peer-to-peer send/recv of r slices each way), slab pass        -> A  [Zl][Y][X]
    re-slab     all-to-all; block g->h = A[:, (ys_h-r .. ye_h+r) mod Y, :]  (the sender owns every y of its z range,
                so the receiver's periodic halo travels with the block: no extra halo exchange) -> Ae [Z][Yl+2r][X]
    Y pass      slices are Ae[:, y, :]: slice stride X, row stride (Yl+2r)*X                    -> B  [Z][Yl][X]
    re-slab     all-to-all; block g->h = B[:, :, (xs_h-r .. xe_h+r) mod X], transposed while unpacking
                                                                                                -> Ce [Z][Xl+2r][Y]
    X pass      slices are Ce[:, x, :] (Z x Y images, y contiguous)                             -> D  [Z][Xl][Y]
    re-slab     all-to-all back to Z-slabs, transposed while unpacking                          -> out[Zl][Y][X]

Packing / transposing are the library's own kernels (fdn_copy3d, fdn_transpose_strided); the exchanges are NCCL
all-to-all / grouped send-recv (torch.distributed is plumbing only). Results are bit-identical for any number of
ranks because every slice is computed from identical inputs by the same kernels.

A typed slab (keep_dtype: uint8, int8, uint16 or int16) runs the same sequence in its own dtype: every buffer has the
slab's dtype, the kernels are the typed ones (fdn_copy3d_typed, fdn_transpose_strided_typed, typed passes), and the
exchanges carry byte views of the buffers, because NCCL has no 16-bit integer type (an exchange only moves bits).

The compute object (`ops`) is a DeviceEngine; tests inject a CPU stand-in to exercise this host logic with the gloo
backend (tests/test_dist_gloo.py).
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np

from ._lib import View


def split_range(n: int, parts: int, idx: int):
    """Balanced contiguous split of range(n) into `parts`; returns [start, end) of part idx."""
    base, rem = divmod(n, parts)
    start = idx * base + min(idx, rem)
    return start, start + base + (1 if idx < rem else 0)


class DistributedDenoiser:
    def __init__(self, ops, shape: Sequence[int], flow, exact: bool = True, group=None, chunk: Optional[int] = None):
        import torch.distributed as dist
        self.dist = dist
        self.ops = ops
        self.torch = ops.torch
        self.shape = tuple(int(s) for s in shape)
        self.flow = flow
        self.exact = exact
        self.chunk = chunk
        self.group = group
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        Z, Y, X = self.shape
        if min(Z, Y, X) < self.world:
            raise ValueError("every axis must have at least one slice per rank")
        self.z_range = split_range(Z, self.world, self.rank)
        self.y_range = split_range(Y, self.world, self.rank)
        self.x_range = split_range(X, self.world, self.rank)
        self.backend = dist.get_backend(group)
        self.dtype = self.torch.float32       # of the slab being filtered (set by filter / filter_host)

    def _empty(self, shape):
        """A buffer in the slab's dtype (float32 slabs: the one-argument call of the float route)."""
        if self.dtype == self.torch.float32:
            return self.ops.empty(shape)
        return self.ops.empty(shape, self.dtype)

    def _wire(self, t):
        """What an exchange carries for the contiguous tensor t: t itself for float32, its bytes otherwise (NCCL has no
        16-bit integer type; the exchanges only move bits, so a byte view is right for every dtype)."""
        if t.dtype == self.torch.float32:
            return t
        return t.reshape(-1).view(self.torch.uint8)

    def _use_dtype(self, t):
        if t.dtype != self.torch.float32:
            from .engine import dtype_code
            dtype_code(t)                     # ValueError for an unsupported dtype
        self.dtype = t.dtype

    # ------------------------------------------------------------------ communication primitives
    def _all_to_all(self, send_flat, send_sizes, recv_flat, recv_sizes):
        """One flat buffer per direction, split per peer (own block included); typed buffers travel as bytes."""
        dist = self.dist
        if send_flat.dtype != self.torch.float32:
            k = send_flat.element_size()
            send_flat, recv_flat = self._wire(send_flat), self._wire(recv_flat)
            send_sizes, recv_sizes = [k * int(n) for n in send_sizes], [k * int(n) for n in recv_sizes]
        if self.backend == "nccl":
            dist.all_to_all_single(recv_flat, send_flat, list(recv_sizes), list(send_sizes), group=self.group)
            return
        # gloo (CPU tests) has no all-to-all: the same exchange as grouped send/recv
        so = np.concatenate([[0], np.cumsum(send_sizes)]).astype(np.int64)
        ro = np.concatenate([[0], np.cumsum(recv_sizes)]).astype(np.int64)
        ops = []
        for p in range(self.world):
            sv = send_flat[int(so[p]):int(so[p + 1])]
            rv = recv_flat[int(ro[p]):int(ro[p + 1])]
            if p == self.rank:
                rv.copy_(sv)
                continue
            ops.append(dist.P2POp(dist.isend, sv, self._global_rank(p), self.group))
            ops.append(dist.P2POp(dist.irecv, rv, self._global_rank(p), self.group))
        if ops:
            for w in dist.batch_isend_irecv(ops):
                w.wait()

    def _global_rank(self, p):
        return p if self.group is None else self.dist.get_global_rank(self.group, p)

    def _alltoall_blocks(self, send_shapes, recv_shapes, pack):
        """Generic re-slab: pack(p, buf) fills the (flat) block for peer p; returns the received flat blocks."""
        ops = self.ops
        ssz = [int(np.prod(sh)) for sh in send_shapes]
        rsz = [int(np.prod(sh)) for sh in recv_shapes]
        send_flat = self._empty((sum(ssz),))
        recv_flat = self._empty((sum(rsz),))
        off = 0
        for p in range(self.world):
            pack(p, send_flat[off:off + ssz[p]])
            off += ssz[p]
        self._all_to_all(send_flat, ssz, recv_flat, rsz)
        out, off = [], 0
        for p in range(self.world):
            out.append(recv_flat[off:off + rsz[p]])
            off += rsz[p]
        return out

    # ------------------------------------------------------------------ Z pass: explicit periodic halo exchange
    def _z_halo_fill(self, ext, r):
        """ext = [r + Zl + r][Y][X] with the local Z-slab in the middle (at least its first and last r slices): fills
        the r periodic halo slices on both sides from the owning ranks with grouped send/recv (P2P over NVLink under
        NCCL)."""
        dist, torch, ops = self.dist, self.torch, self.ops
        Z, Y, X = self.shape
        zs, ze = self.z_range
        Zl = ze - zs
        if r == 0:
            return ext
        slab = ext[r:r + Zl]
        owner_ranges = [split_range(Z, self.world, p) for p in range(self.world)]

        def owner_of(z):
            for p, (a, b) in enumerate(owner_ranges):
                if a <= z < b:
                    return p
            raise AssertionError

        # what I need: ext index e <-> global slice (zs - r + e) mod Z, for e in halo positions
        need = [(e, (zs - r + e) % Z) for e in list(range(r)) + list(range(r + Zl, Zl + 2 * r))]
        # what peer p needs from me, in p's own ext order (both sides enumerate identically -> matched messages)
        p2p = []
        recv_bufs = {}
        for p in range(self.world):
            if p == self.rank:
                continue
            mine = [(e, z) for (e, z) in need if owner_of(z) == p]
            if mine:
                buf = self._empty((len(mine), Y, X))
                recv_bufs[p] = (buf, mine)
                p2p.append(dist.P2POp(dist.irecv, self._wire(buf), self._global_rank(p), self.group))
            pzs, pze = owner_ranges[p]
            pl = pze - pzs
            theirs = [(pzs - r + e) % Z for e in list(range(r)) + list(range(r + pl, pl + 2 * r))]
            theirs = [z for z in theirs if zs <= z < ze]
            if theirs and self.dtype != torch.float32:
                sbuf = self._empty((len(theirs), Y, X))          # (plain copies: torch has few uint16 device kernels)
                for i, z in enumerate(theirs):
                    sbuf[i].copy_(slab[z - zs])
            elif theirs:
                sbuf = torch.stack([slab[z - zs] for z in theirs]) if len(theirs) > 1 else slab[theirs[0] - zs][None].contiguous()
            if theirs:
                p2p.append(dist.P2POp(dist.isend, self._wire(sbuf.contiguous()), self._global_rank(p), self.group))
        for (e, z) in need:                      # halo slices that wrap onto my own slab (few ranks / tiny Z)
            if zs <= z < ze:
                ext[e].copy_(slab[z - zs])
        if p2p:
            for w in dist.batch_isend_irecv(p2p):
                w.wait()
        for p, (buf, mine) in recv_bufs.items():
            for i, (e, _z) in enumerate(mine):
                ext[e].copy_(buf[i])
        return ext

    def _z_halo_extended(self, slab, r):
        """Returns [r + Zl + r][Y][X]: the local Z-slab with r periodic halo slices on both sides."""
        Z, Y, X = self.shape
        Zl = self.z_range[1] - self.z_range[0]
        ext = self._empty((Zl + 2 * r, Y, X))
        ext[r:r + Zl].copy_(slab)
        return self._z_halo_fill(ext, r)

    # ------------------------------------------------------------------ re-slabs between the passes
    def _ranges(self):
        G = self.world
        Z, Y, X = self.shape
        return ([split_range(Z, G, p) for p in range(G)], [split_range(Y, G, p) for p in range(G)],
                [split_range(X, G, p) for p in range(G)])

    def _reslab_zy(self, A, ry):
        """Z-slab A [Zl][Y][X] -> Ae [Z][Yl + 2 ry][X] (this rank's y range with its periodic halo)."""
        ops, G = self.ops, self.world
        Z, Y, X = self.shape
        zr, yr, _xr = self._ranges()
        Zl = self.z_range[1] - self.z_range[0]
        Yl = self.y_range[1] - self.y_range[0]

        def pack_zy(p, buf):
            a, b = yr[p]
            n = (b - a) + 2 * ry
            ops.copy3d(A, 0, Y * X, X, a - ry, Y, 0, X, buf, 0, n * X, X, Zl, n, X)
        blocks = self._alltoall_blocks([(Zl, (yr[p][1] - yr[p][0]) + 2 * ry, X) for p in range(G)],
                                       [(zr[p][1] - zr[p][0], Yl + 2 * ry, X) for p in range(G)], pack_zy)
        Ye = Yl + 2 * ry
        Ae = self._empty((Z, Ye, X))
        flatA = Ae.view(-1)
        for p in range(G):
            a, b = zr[p]
            flatA[a * Ye * X:b * Ye * X].copy_(blocks[p])
        return Ae

    def _reslab_yz(self, B):
        """Y-slab B [Z][Yl][X] (the Z+Y intermediate) -> Z-slab [Zl][Y][X]."""
        ops, G = self.ops, self.world
        Z, Y, X = self.shape
        zr, yr, _xr = self._ranges()
        Zl = self.z_range[1] - self.z_range[0]
        Yl = self.y_range[1] - self.y_range[0]

        def pack_b(p, buf):
            a, b = zr[p]
            ops.copy3d(B, a * Yl * X, Yl * X, X, 0, Yl, 0, X, buf, 0, Yl * X, X, b - a, Yl, X)
        blocks = self._alltoall_blocks([(zr[p][1] - zr[p][0], Yl, X) for p in range(G)],
                                       [(Zl, yr[p][1] - yr[p][0], X) for p in range(G)], pack_b)
        zy_slab = self._empty((Zl, Y, X))
        for p in range(G):
            a, b = yr[p]
            ops.copy3d(blocks[p], 0, (b - a) * X, X, 0, b - a, 0, X, zy_slab, a * X, Y * X, X, Zl, b - a, X)
        return zy_slab

    def _reslab_yx(self, B, rx):
        """Y-slab B [Z][Yl][X] -> Ce [Z][Xl + 2 rx][Y] (this rank's x range with its periodic halo, transposed while
        unpacking)."""
        ops, G = self.ops, self.world
        Z, Y, X = self.shape
        _zr, yr, xr = self._ranges()
        Yl = self.y_range[1] - self.y_range[0]
        Xl = self.x_range[1] - self.x_range[0]

        def pack_yx(p, buf):
            a, b = xr[p]
            n = (b - a) + 2 * rx
            ops.copy3d(B, 0, Yl * X, X, 0, Yl, a - rx, X, buf, 0, Yl * n, n, Z, Yl, n)
        Xe = Xl + 2 * rx
        blocks = self._alltoall_blocks([(Z, Yl, (xr[p][1] - xr[p][0]) + 2 * rx) for p in range(G)],
                                       [(Z, yr[p][1] - yr[p][0], Xe) for p in range(G)], pack_yx)
        Ce = self._empty((Z, Xe, Y))
        for p in range(G):
            a, b = yr[p]
            # block[z][y][x] -> Ce[z][x][a + y]
            ops.transpose_strided(blocks[p], 0, (b - a) * Xe, Xe, Ce, a, Xe * Y, Y, Z, b - a, Xe)
        return Ce

    def _reslab_xz(self, D, out, part="all", tail=0):
        """Columns of every rank's X-slab D [Z][Xl][Y] -> the same columns of the Z-slabs out [Zl][Y][X] (blocks are
        contiguous on the sending side; transposed while unpacking). part = "all", or "body" / "tail": all but the
        last `tail` columns / the last `tail` columns of EVERY rank's x range (ranges may differ by one column).
        Returns the [x0, x1) ranges of `out` that were written."""
        ops, G = self.ops, self.world
        Z, Y, X = self.shape
        zr, _yr, xr = self._ranges()
        Zl = self.z_range[1] - self.z_range[0]
        Xl = self.x_range[1] - self.x_range[0]

        def cols(p):        # (first, count) inside rank p's X-slab
            n = xr[p][1] - xr[p][0]
            return {"all": (0, n), "body": (0, n - tail), "tail": (n - tail, tail)}[part]
        first, mine = cols(self.rank)

        def pack_xz(p, buf):
            a, b = zr[p]
            ops.copy3d(D, a * Xl * Y, Xl * Y, Y, first, Xl, 0, Y, buf, 0, mine * Y, Y, b - a, mine, Y)
        blocks = self._alltoall_blocks([(zr[p][1] - zr[p][0], mine, Y) for p in range(G)],
                                       [(Zl, cols(p)[1], Y) for p in range(G)], pack_xz)
        written = []
        for p in range(G):
            f, n = cols(p)
            a = xr[p][0] + f
            # block[z][x][y] -> out[z][y][a + x]
            ops.transpose_strided(blocks[p], 0, n * Y, Y, out, a, Y * X, X, Zl, n, Y)
            written.append((a, a + n))
        return written

    # ------------------------------------------------------------------ the three passes
    def filter(self, slab, kernels, want_zy: bool = False):
        """slab: this rank's Z-slab [Zl][Y][X] (device; float32, or a typed volume's uint8 / int8 / uint16 / int16:
        every buffer and exchange is then in that dtype and each pass truncates like the reference's integer
        `filtered_vol`). Returns (zy_slab or None, zyx_slab), both Z-slabs in the slab's dtype."""
        ops = self.ops
        Z, Y, X = self.shape
        Zl = self.z_range[1] - self.z_range[0]
        Yl = self.y_range[1] - self.y_range[0]
        Xl = self.x_range[1] - self.x_range[0]
        kz, ky, kx = (np.asarray(k, np.float64) for k in kernels)
        rz, ry, rx = kz.size // 2, ky.size // 2, kx.size // 2
        if tuple(slab.shape) != (Zl, Y, X):
            raise ValueError(f"rank {self.rank} expects a Z-slab of shape {(Zl, Y, X)}, got {tuple(slab.shape)}")
        self._use_dtype(slab)

        # ---- Z pass
        ext = self._z_halo_extended(slab, rz)
        A = self._empty((Zl, Y, X))
        v = View(Zl + 2 * rz, Zl, rz, 0, Y, X, Y * X, X, Y * X, X)
        ops.filter_view(ext, A, v, kz, self.flow, self.chunk, self.exact)
        del ext
        return self._after_z(A, ky, kx, want_zy)

    def _after_z(self, A, ky, kx, want_zy, finish_x=None):
        """Re-slab, Y pass, re-slab, X pass, re-slab back. finish_x(Ce, D, Xe) replaces the plain X pass + re-slab
        (filter_host splits them to hide the download) and returns the result Z-slab."""
        ops = self.ops
        Z, Y, X = self.shape
        Zl = self.z_range[1] - self.z_range[0]
        Yl = self.y_range[1] - self.y_range[0]
        Xl = self.x_range[1] - self.x_range[0]
        ry, rx = ky.size // 2, kx.size // 2
        # ---- re-slab Z -> Y (halo included)
        Ae = self._reslab_zy(A, ry)
        del A
        Ye = Yl + 2 * ry

        # ---- Y pass
        B = self._empty((Z, Yl, X))
        v = View(Ye, Yl, ry, 0, Z, X, X, Ye * X, X, Yl * X)
        ops.filter_view(Ae, B, v, ky, self.flow, self.chunk, self.exact)
        del Ae

        # the reference leaves the Z+Y intermediate in `vol` (src/flowdenoising.py:289)
        zy_slab = self._reslab_yz(B) if want_zy else None

        # ---- re-slab Y -> X (halo included, transposed while unpacking)
        Ce = self._reslab_yx(B, rx)
        del B
        Xe = Xl + 2 * rx

        # ---- X pass, re-slab X -> Z
        D = self._empty((Z, Xl, Y))
        if finish_x is not None:
            return zy_slab, finish_x(Ce, D, Xe)
        v = View(Xe, Xl, rx, 0, Z, Y, Y, Xe * Y, Y, Xl * Y)
        ops.filter_view(Ce, D, v, kx, self.flow, self.chunk, self.exact)
        del Ce
        out = self._empty((Zl, Y, X))
        self._reslab_xz(D, out)
        return zy_slab, out

    # ------------------------------------------------------------------ host slabs in, host slabs out
    def filter_host(self, host_slab, out_host, kernels, head: Optional[int] = None, tail: Optional[int] = None):
        """The same three passes for a Z-slab that lives on the HOST (page-locked tensors [Zl][Y][X] of one dtype, float32
        or a typed volume's; the result is written to out_host), with the transfers hidden behind the passes like the single-device plugin
        (flowdenoising.py:_filter_overlapped): the slab's edge slices go up first and feed the halo exchange, the Z
        pass starts on its first `head` slices while the rest is still on its way, and the last `tail` columns of
        every rank's X-slab are computed while the other columns are already re-slabbed and travelling home.
        Every slice sees the same inputs as in filter(): same bits. Returns the result Z-slab on the device."""
        ops = self.ops
        Z, Y, X = self.shape
        Zl = self.z_range[1] - self.z_range[0]
        Xl = self.x_range[1] - self.x_range[0]
        kz, ky, kx = (np.asarray(k, np.float64) for k in kernels)
        rz, rx = kz.size // 2, kx.size // 2
        if tuple(host_slab.shape) != (Zl, Y, X) or tuple(out_host.shape) != (Zl, Y, X):
            raise ValueError(f"rank {self.rank} expects Z-slabs of shape {(Zl, Y, X)}")
        if out_host.dtype != host_slab.dtype:
            raise ValueError("filter_host writes the dtype it reads")
        self._use_dtype(host_slab)
        cp = _Copies(ops)
        _zr, _yr, xr = self._ranges()
        min_Zl = min(b - a for a, b in _zr)
        min_Xl = min(b - a for a, b in xr)
        # every rank takes the same decisions (the exchanges are collective)
        if head is None:
            head = max(1, min(32, min_Zl // 4))
        if tail is None:
            tail = max(1, min(64, min_Xl // 4))
        split_z = min_Zl >= 2 * rz + 2 and head + 2 * rz < min_Zl
        split_x = 1 <= tail < min_Xl

        # ---- upload (copy stream) and Z pass
        ext = self._empty((Zl + 2 * rz, Y, X))
        mid = ext[rz:rz + Zl]
        cp.fence()
        if split_z:
            cp.copy(mid[:rz], host_slab[:rz])                  # the edges: what the neighbours' halos need
            cp.copy(mid[Zl - rz:], host_slab[Zl - rz:])
            e_edges = cp.mark()
            cp.copy(mid[rz:head + rz], host_slab[rz:head + rz])
            e_head = cp.mark()
            cp.copy(mid[head + rz:Zl - rz], host_slab[head + rz:Zl - rz])
            e_all = cp.mark()
        else:
            cp.copy(mid, host_slab)
            e_edges = e_head = e_all = cp.mark()
        cp.compute_waits(e_edges)
        self._z_halo_fill(ext, rz)
        A = self._empty((Zl, Y, X))
        if split_z:
            cp.compute_waits(e_head)
            ops.filter_view(ext, A, View(head + 2 * rz, head, rz, 0, Y, X, Y * X, X, Y * X, X), kz, self.flow,
                            self.chunk, self.exact)
            cp.compute_waits(e_all)
            ops.filter_view(ext[head:], A[head:], View(Zl - head + 2 * rz, Zl - head, rz, 0, Y, X, Y * X, X, Y * X, X),
                            kz, self.flow, self.chunk, self.exact)
        else:
            cp.compute_waits(e_all)
            ops.filter_view(ext, A, View(Zl + 2 * rz, Zl, rz, 0, Y, X, Y * X, X, Y * X, X), kz, self.flow,
                            self.chunk, self.exact)
        del ext, mid

        # ---- X pass in two column ranges, each re-slabbed and sent home as soon as it is done
        def finish_x(Ce, D, Xe):
            out = self._empty((Zl, Y, X))
            flatC, flatD = Ce.view(-1), D.view(-1)
            parts = [("body", 0, Xl - tail), ("tail", Xl - tail, tail)] if split_x else [("all", 0, Xl)]
            for part, first, n in parts:
                # outputs first .. first + n - 1 of this rank's x range; their inputs start at Ce slice `first`
                ops.filter_view(flatC[first * Y:], flatD[first * Y:],
                                View(n + 2 * rx, n, rx, 0, Z, Y, Y, Xe * Y, Y, Xl * Y), kx, self.flow, self.chunk,
                                self.exact)
                written = self._reslab_xz(D, out, part, tail)
                cp.fence()
                for x0, x1 in written:
                    if x1 > x0:
                        cp.copy_cols(out_host, out, x0, x1)
            return out

        _zy, out = self._after_z(A, ky, kx, False, finish_x)
        cp.done()
        return out


class _Copies:
    """Host <-> device copies of filter_host: on a copy stream when the compute object lives on a CUDA device, inline
    for the CPU stand-in of the gloo tests."""

    def __init__(self, ops):
        self.ops = ops
        self.torch = ops.torch
        dev = getattr(ops, "device", None)
        self.cuda = dev is not None and dev.type == "cuda"
        self.stream = self.torch.cuda.Stream(device=dev) if self.cuda else None

    def fence(self):
        """Copies issued from now on start after everything already enqueued on the compute stream."""
        if self.cuda:
            self.stream.wait_stream(self.torch.cuda.current_stream())

    def copy(self, dst, src):
        if dst.numel() == 0:
            return
        if self.cuda:
            with self.torch.cuda.stream(self.stream):
                dst.copy_(src, non_blocking=True)
        else:
            dst.copy_(src)

    def copy_cols(self, dst_host, src_dev, x0, x1):
        """Columns [x0, x1) of a device volume [n][Y][X] -> the same columns of a host volume (pitched copy)."""
        if self.cuda:
            n, Y, X = (int(v) for v in src_dev.shape)
            es = src_dev.element_size()
            self.ops.copy2d_async(dst_host.data_ptr() + es * x0, es * X, src_dev.data_ptr() + es * x0, es * X,
                                  es * (x1 - x0), n * Y, 1, self.stream)
        else:
            dst_host[:, :, x0:x1].copy_(src_dev[:, :, x0:x1])

    def mark(self):
        if not self.cuda:
            return None
        e = self.torch.cuda.Event()
        e.record(self.stream)
        return e

    def compute_waits(self, e):
        if self.cuda and e is not None:
            self.torch.cuda.current_stream().wait_event(e)

    def done(self):
        if self.cuda:
            self.stream.synchronize()
