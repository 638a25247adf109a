"""Row-sharded forms of the hot path across the GPUs of one box (SURVEY.md 8e).

One process per GPU.  Rank g owns the contiguous row block [starts[g], starts[g+1]); its CSR block
keeps GLOBAL column indices.  What moves between ranks, and how:

  assembly   COO triplets start block-distributed by entry index.  Each rank partitions its
             triplets by owning rank on the device (spl_coo_route_dev: one stable radix pass, keys
             already packed for the receiver), one all-to-all (NCCL) moves them, the receiver
             concatenates the shares in source-rank order — which keeps the global insertion order
             among duplicates — and runs the single-GPU assembly (spl_mat_from_packed_dev).
             Bit-exact against the reference's From<&CooMatrix> on the whole matrix.
  SpMV       x stays where it lives.  Every rank keeps its slice of x in peer-visible memory
             (CUDA IPC over NVLink/NVSwitch), twice (products read the published buffer, the rank
             writes the other).  Banded / stencil shards: one small kernel is the device-side flag
             barrier and copies the few halo columns next to the own slice (spl_peer_barrier_halo),
             then the unsharded kernels run (spl_spmv_window); spl_spmv_peer, which gathers each
             x[c] from the slice that owns column c inside the kernel, stays available.  General
             (random / power-law) shards need the whole of x: ONE kernel pulls the peers' slices
             with TMA bulk copies while it multiplies block by block (spl_spmv_gather_fused), or
             x is pulled / all-gathered first (spl_peer_pull, NCCL in sharding.py).
  A^T x      each rank multiplies x's slice by its shard's transpose over the shard's column footprint only
             (spl_spmv_transpose_window) into one of two peer-visible partial buffers; one kernel then runs the
             flag barrier and sums, for every column of the rank's slice of y, the partials of the ranks whose
             footprint holds it, in ascending rank (spl_peer_reduce_windows): deterministic, and y lands in a
             column partition of the caller's choice (x's own for a square matrix).
  add/sub/neg  no exchange when the operands share the partition.
  mul        C = A * B with A, B row-sharded (B with any row partition): rank g's rows of C need exactly the rows
             of B that its shard's stored columns name.  Every rank copies its shard of B into three peer buffers
             (pointers, indices, values; sized by one all-gather of the shard sizes), one flag barrier, then
             spl_peer_gather_rows copies the named rows from their owners over NVLink into one local matrix of
             B's full height (other rows empty; runs of rows of one owner as TMA bulk copies), a second barrier,
             and the unsharded product A_local * gathered (spl_mat_mul): bit for bit the rows of the whole
             product.  Banded / stencil shards move a thin halo; random ones about all of B.  The CSC twin
             (column-sharded) gathers the columns of A that B's shard names.

torch.distributed is the plumbing (rendezvous, the all-to-all, object exchange of IPC handles);
the device work goes through the C ABI.  The CPU tests (gloo, world size 2) drive the same host
logic with a numpy stand-in for the two device calls.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import List, Optional, Sequence

import numpy as np

from . import _capi as capi
from .matrix import Context, CsrMatrix, Panic, _dtype_code, default_context
from .sharding import row_partition


def partition_starts(n: int, world: int) -> List[int]:
    """starts[g] = first row of rank g (equal-row blocks), starts[world] = n."""
    return [row_partition(n, world, g)[0] for g in range(world)] + [n]


def balanced_starts(bin_counts: Sequence[int], rows_per_bin: int, n: int, world: int) -> List[int]:
    """Row partition balanced on stored entries (SURVEY.md 8e: "boundaries chosen to balance nnz ...
    matters for C4"): bin_counts[b] = entries whose row lies in [b * rows_per_bin, (b+1) * rows_per_bin).
    starts[g] is the bin boundary closest to the g/world quantile of the entries (contiguous blocks,
    every rank non-empty when there are at least `world` bins)."""
    counts = np.asarray(bin_counts, dtype=np.float64)
    nb = len(counts)
    # balance rows + entries, as the single-GPU kernels do: empty stretches still cost pointer traffic
    w = counts + np.minimum(rows_per_bin, np.maximum(n - np.arange(nb) * rows_per_bin, 0))
    cum = np.concatenate([[0.0], np.cumsum(w)])
    starts = [0]
    for g in range(1, world):
        b = int(np.searchsorted(cum, cum[-1] * g / world, side="left"))
        b = min(max(b, starts[-1] // rows_per_bin + 1), nb - (world - g))     # strictly increasing, room for the rest
        starts.append(min(b * rows_per_bin, n))
    return starts + [n]


def balanced_starts_from_rows(dist, torch, rows, n: int, world: int, bins: int = 1 << 16, group=None) -> List[int]:
    """balanced_starts from this rank's int32 (uint32 bit pattern) row indices on the device: a coarse
    histogram per rank, one all-reduce, the boundaries computed identically on every rank."""
    rows_per_bin = max(1, -(-n // bins))
    nb = -(-n // rows_per_bin)
    r = rows.long() & 0xFFFFFFFF
    h = torch.bincount(torch.div(r, rows_per_bin, rounding_mode="floor"), minlength=nb).to(torch.int64)
    if world > 1:
        dist.all_reduce(h, group=group)
    return balanced_starts(h.cpu().numpy(), rows_per_bin, n, world)


def bits_for(count: int) -> int:
    """Bits needed for values in [0, count) — the packing rule of spl_coo_route_dev."""
    return 0 if count <= 1 else int(count - 1).bit_length()


# ------------------------------------------------------------------------- sharded assembly
def exchange_routed(dist, torch, keys, vals, counts: Sequence[int], group=None):
    """All-to-all of routed triplets.  `keys`/`vals` hold this rank's shares for rank 0, 1, ...
    back to back (`counts[g]` entries each).  Returns (recv_keys, recv_vals, recv_counts) with the
    received shares concatenated in SOURCE-RANK order (insertion order among duplicates)."""
    world = dist.get_world_size(group)
    send = torch.tensor(list(counts), dtype=torch.int64, device=keys.device)
    recv = torch.empty(world, dtype=torch.int64, device=keys.device)
    dist.all_to_all_single(recv, send, group=group)
    recv_counts = [int(v) for v in recv.tolist()]
    total = sum(recv_counts)
    rk = torch.empty(total, dtype=keys.dtype, device=keys.device)
    rv = torch.empty(total, dtype=vals.dtype, device=vals.device)
    dist.all_to_all_single(rk, keys, recv_counts, list(counts), group=group)
    dist.all_to_all_single(rv, vals, recv_counts, list(counts), group=group)
    return rk, rv, recv_counts


def _torch_to_ctx(torch):
    """Device tensors handed to the library were written on torch's current stream; the library works on
    the context's stream.  When the two are one stream (bench.py, the tests) this costs nothing."""
    if torch.cuda.is_available():
        torch.cuda.current_stream().synchronize()


def route_device(ctx: Context, torch, fmt: int, nrows: int, ncols: int, row, col, val, starts):
    """Device stable partition by owner (spl_coo_route_dev) of uint32 row/col (int32 tensors) and
    f32/f64 values.  Returns (keys int64 tensor, vals tensor, counts list)."""
    n = int(val.numel())
    world = len(starts) - 1
    keys = torch.empty(n, dtype=torch.int64, device=val.device)
    vals = torch.empty_like(val)
    st = (C.c_uint64 * (world + 1))(*starts)
    cnt = (C.c_uint64 * world)()
    ctx.check(ctx._lib.spl_coo_route_dev(
        ctx._h, fmt, _dtype_code(np.float32 if val.dtype == torch.float32 else np.float64), nrows, ncols, n,
        C.c_void_p(row.data_ptr()), C.c_void_p(col.data_ptr()), C.c_void_p(val.data_ptr()), world,
        C.cast(st, C.c_void_p), C.c_void_p(keys.data_ptr()), C.c_void_p(vals.data_ptr()),
        C.cast(cnt, C.c_void_p)))
    return keys, vals, [int(c) for c in cnt]


def _assemble_over_peers(dist, torch, fmt: int, nrows: int, ncols: int, row, col, val, exchange, dedup, dropzero,
                         starts=None):
    """Route this rank's triplets to the owners of their major index (rows for CSR, columns for CSC)
    through peer memory and assemble the own shard.  Returns (spl_mat handle, major partition)."""
    ctx, group = exchange.ctx, exchange.group
    world, rank = exchange.world, exchange.rank
    _torch_to_ctx(torch)                      # row/col/val were produced on torch's stream
    nmajor = nrows if fmt == capi.SPL_CSR else ncols
    starts = list(starts) if starts is not None else partition_starts(nmajor, world)
    n = int(val.numel())
    dtype = np.float32 if val.dtype == torch.float32 else np.float64
    st = (C.c_uint64 * (world + 1))(*starts)
    cnt = (C.c_uint64 * world)()
    ctx.check(ctx._lib.spl_coo_route_count_dev(ctx._h, fmt, nrows, ncols, n, C.c_void_p(row.data_ptr()),
                                               C.c_void_p(col.data_ptr()), world, C.cast(st, C.c_void_p),
                                               C.cast(cnt, C.c_void_p)))
    mine = torch.tensor([int(c) for c in cnt], dtype=torch.int64, device=val.device)
    allc = torch.empty(world * world, dtype=torch.int64, device=val.device)
    dist.all_gather_into_tensor(allc, mine, group=group)
    M = allc.view(world, world).tolist()                     # M[src][dst]
    recv_total = [sum(M[s][d] for s in range(world)) for d in range(world)]
    offs = [sum(M[s][d] for s in range(rank)) for d in range(world)]      # source-rank order
    exchange.ensure(max(recv_total), np.dtype(dtype).itemsize)
    kb = (C.c_void_p * world)(*exchange._keys.ptrs)
    vb = (C.c_void_p * world)(*exchange._vals.ptrs)
    off = (C.c_uint64 * world)(*offs)
    exchange.barrier()                                        # owners are done with the old contents
    ctx.check(ctx._lib.spl_coo_route_peers_dev(
        ctx._h, fmt, _dtype_code(dtype), nrows, ncols, n, C.c_void_p(row.data_ptr()),
        C.c_void_p(col.data_ptr()), C.c_void_p(val.data_ptr()), world, C.cast(st, C.c_void_p),
        C.cast(kb, C.c_void_p), C.cast(vb, C.c_void_p), C.cast(off, C.c_void_p)))
    exchange.barrier()                                        # every record has landed
    exchange.check()          # a barrier that gave up must not let a half-filled buffer be assembled (host sync:
    #                           the assembly below synchronises for its output size anyway)
    nloc = max(starts[rank + 1] - starts[rank], 1)
    h = C.c_void_p()
    ctx.check(ctx._lib.spl_mat_from_packed_dev(
        ctx._h, fmt, _dtype_code(dtype), nloc if fmt == capi.SPL_CSR else nrows,
        ncols if fmt == capi.SPL_CSR else nloc, recv_total[rank],
        C.c_void_p(exchange._keys.local), C.c_void_p(exchange._vals.local), int(dedup), int(dropzero),
        C.byref(h)))
    return h, starts


def gather_block_layout(torch, ptr, col, val, starts, rank: int, first):
    """The blocked form of a row shard that spl_spmv_gather_fused takes (plain tensor plumbing: runs on the
    device for prepare_gather and on the CPU in the tests).  ptr: int64[nloc+1] row pointers of the shard,
    col: int32 (uint32 bit pattern) GLOBAL columns, val: values; starts: column partition; first: ring offsets
    where blocks begin (block b = columns owned by ranks rank+first[b] .. rank+first[b+1]-1, mod world).
    Returns bptr int32[nblocks, stride] (absolute positions; every row padded to a multiple of 4 entries that
    repeat the end position, plus 4), bind / bval (entries stably regrouped by block, row order and column
    order kept inside a block, 4 entries of slack), stride, and caps = the most entries any 64 / 128 / 256 /
    512 / 1024 consecutive rows starting at a multiple of 32 hold in one block."""
    world = len(starts) - 1
    nloc = int(ptr.numel()) - 1
    nb = len(first) - 1
    dev = col.device
    rows = torch.repeat_interleave(torch.arange(nloc, device=dev), ptr[1:] - ptr[:-1])
    bounds = torch.tensor(list(starts[1:-1]), device=dev, dtype=torch.int64)
    owner = torch.searchsorted(bounds, col.long() & 0xFFFFFFFF, right=True)
    offset = (owner - rank) % world
    block = torch.searchsorted(torch.tensor(list(first[1:]), device=dev, dtype=torch.int64), offset, right=True).to(torch.int16)
    order = torch.sort(block, stable=True).indices
    bind = col[order].contiguous()
    bval = val[order].contiguous()
    key = block[order].long() * nloc + rows[order]
    counts = torch.bincount(key, minlength=nb * nloc).view(nb, nloc)
    base = torch.cumsum(counts.sum(1), 0) - counts.sum(1)                 # first position of every block
    # the kernel fetches whole tiles with 16-byte bulk copies: pointer arrays padded to a multiple of 4 entries (the
    # padding repeats the end position), four entries of slack behind the indices and values
    stride = (nloc + 1 + 3) // 4 * 4 + 4
    bptr = torch.zeros((nb, stride), dtype=torch.int64, device=dev)
    bptr[:, 1:nloc + 1] = torch.cumsum(counts, 1)
    bptr[:, nloc + 1:] = bptr[:, nloc:nloc + 1]
    bptr += base[:, None]
    pad = lambda t: torch.cat([t, torch.zeros(4, dtype=t.dtype, device=t.device)])
    at = torch.arange(0, max(nloc, 1), 32, device=dev)
    caps = [int((bptr[:, torch.clamp(at + w, max=nloc)] - bptr[:, at]).max().item()) for w in (64, 128, 256, 512, 1024)]
    return {"bptr": bptr.to(torch.int32).contiguous(), "bind": pad(bind), "bval": pad(bval), "stride": stride, "caps": caps}


class DistCsrMatrix:
    """Row block of a CSR matrix on this rank plus the partition it belongs to."""

    def __init__(self, local: CsrMatrix, starts: Sequence[int], rank: int, nrows: int, ncols: int):
        self.local, self.starts, self.rank = local, list(starts), int(rank)
        self.world = len(starts) - 1
        self._nrows, self._ncols = int(nrows), int(ncols)

    def nrows(self): return self._nrows
    def ncols(self): return self._ncols
    def local_rows(self): return self.starts[self.rank], self.starts[self.rank + 1]

    @classmethod
    def from_device_triplets_peer(cls, dist, torch, nrows: int, ncols: int, row, col, val, exchange: "PeerExchange",
                                  dedup=True, dropzero=True, starts=None, balance: Optional[str] = None):
        """Sharded From<&CooMatrix<T>> for CsrMatrix<T> with routing and exchange fused: the partition
        pass writes every triplet straight into its owner's receive buffer over NVLink (peer memory),
        bracketed by two device-side barriers; the only collective is the all-gather of world*world
        counts that lays the buffers out.  Same result, bit for bit, as from_device_triplets.
        `balance="nnz"` cuts the rows so that every rank gets about the same number of triplets."""
        if starts is None and balance == "nnz":
            starts = balanced_starts_from_rows(dist, torch, row, nrows, exchange.world, group=exchange.group)
        h, starts = _assemble_over_peers(dist, torch, capi.SPL_CSR, nrows, ncols, row, col, val, exchange,
                                         dedup, dropzero, starts)
        return cls(CsrMatrix._wrap(exchange.ctx, h), starts, exchange.rank, nrows, ncols)

    @classmethod
    def from_device_triplets(cls, dist, torch, nrows: int, ncols: int, row, col, val,
                             ctx: Optional[Context] = None, dedup=True, dropzero=True, group=None, starts=None,
                             balance: Optional[str] = None):
        """Sharded From<&CooMatrix<T>> for CsrMatrix<T> (src/csr/conv/coo.rs:3-116).  row/col are
        this rank's int32 (uint32 bit pattern) device tensors, val f32/f64; entries are
        block-distributed by entry index (rank 0 holds the first entries of the COO list)."""
        import os
        import time
        ctx = ctx or default_context()
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        if starts is None and balance == "nnz":
            starts = balanced_starts_from_rows(dist, torch, row, nrows, world, group=group)
        starts = list(starts) if starts is not None else partition_starts(nrows, world)
        timing = os.environ.get("SPL_DIST_TIMING") and rank == 0
        _torch_to_ctx(torch)                  # row/col/val were produced on torch's stream
        t0 = time.perf_counter()
        keys, vals, counts = route_device(ctx, torch, capi.SPL_CSR, nrows, ncols, row, col, val, starts)
        t1 = time.perf_counter()
        rk, rv, _ = exchange_routed(dist, torch, keys, vals, counts, group)   # route ended with a stream sync
        torch.cuda.current_stream().synchronize()     # NCCL ran on torch's stream, assembly runs on ctx's
        t2 = time.perf_counter()
        nloc = starts[rank + 1] - starts[rank]
        h = C.c_void_p()
        dtype = np.float32 if val.dtype == torch.float32 else np.float64
        ctx.check(ctx._lib.spl_mat_from_packed_dev(
            ctx._h, capi.SPL_CSR, _dtype_code(dtype), max(nloc, 1), ncols, int(rk.numel()),
            C.c_void_p(rk.data_ptr()), C.c_void_p(rv.data_ptr()), int(dedup), int(dropzero), C.byref(h)))
        if timing:
            ctx.sync()
            t3 = time.perf_counter()
            print(f"[spl dist] sharded assembly on rank 0: route {1e3 * (t1 - t0):.2f} ms, all-to-all "
                  f"{1e3 * (t2 - t1):.2f} ms, shard assembly {1e3 * (t3 - t2):.2f} ms "
                  f"({int(val.numel())} triplets in, {int(rk.numel())} received)", flush=True)
        return cls(CsrMatrix._wrap(ctx, h), starts, rank, nrows, ncols)

    # add / sub / neg: rank-local on a shared partition (SURVEY.md 8e, "sharded add/sub")
    def _same_partition(self, rhs):
        if (self._nrows, self._ncols) != (rhs._nrows, rhs._ncols):
            raise Panic("assertion `left == right` failed: shapes differ")
        if self.starts != rhs.starts or self.rank != rhs.rank:
            raise Panic("operands of a sharded add/sub must share the row partition")

    def __add__(self, rhs):
        self._same_partition(rhs)
        return DistCsrMatrix(self.local + rhs.local, self.starts, self.rank, self._nrows, self._ncols)

    def __sub__(self, rhs):
        self._same_partition(rhs)
        return DistCsrMatrix(self.local - rhs.local, self.starts, self.rank, self._nrows, self._ncols)

    def __neg__(self):
        return DistCsrMatrix(-self.local, self.starts, self.rank, self._nrows, self._ncols)

    def mul(self, rhs: "DistCsrMatrix", dist, torch, group=None) -> "DistCsrMatrix":
        """Sharded `&A * &B` (impl Mul for &CsrMatrix, src/csr/ops/mul.rs:5-60): this rank's rows of A·B, with A's
        row partition and rhs.ncols() columns; rhs may have any row partition.  The rows of B this shard needs are
        gathered from their owners over peer memory (spl_peer_gather_rows), then multiplied locally: bit for bit the
        rows of the unsharded product.  Collective."""
        if self._ncols != rhs._nrows:
            raise Panic("assertion `left == right` failed: self.ncols() == rhs.nrows()")
        shard = _PeerShard(rhs, dist, torch, group)
        try:
            gathered = shard.gather(self.local)
        finally:
            shard.close()
        return DistCsrMatrix(self.local * gathered, self.starts, self.rank, self._nrows, rhs._ncols)

    def nnz_global(self, dist, torch, group=None):
        t = torch.tensor([self.local.nnz()], dtype=torch.int64,
                         device="cuda" if torch.cuda.is_available() else "cpu")
        dist.all_reduce(t, group=group)
        return int(t.item())

    def to_csc(self, dist, torch, group=None, exchange: Optional["PeerExchange"] = None) -> "DistCscMatrix":
        """Sharded From<&CsrMatrix> for CscMatrix (src/csc/conv/csr.rs:3-53): row-sharded CSR in,
        column-sharded CSC out (rank g gets columns [cstarts[g], cstarts[g+1]), global row indices).
        The stored entries are routed to the owner of their column with the same device partition as
        sharded assembly (spl_coo_route_dev, format CSC), one all-to-all, and a (column, row) sort on
        the receiver with no duplicate sum and no zero drop: bit-exact columns of the whole matrix's
        CSC form."""
        from .synthetic_device import device_view
        ctx = self.local._ctx
        world, rank = self.world, self.rank
        cstarts = partition_starts(self._ncols, world)
        r0, r1 = self.local_rows()
        nnz = self.local.nnz()
        tdt = torch.float32 if self.local.dtype == np.float32 else torch.float64
        ctx.sync()        # the matrix may still have tail kernels queued on the context's stream; torch reads it below
        p_ptr, p_ind, p_val = self.local.device_ptrs()
        ptr = device_view(torch, p_ptr, r1 - r0 + 1, torch.int32)
        if nnz:
            col = device_view(torch, p_ind, nnz, torch.int32)
            val = device_view(torch, p_val, nnz, tdt)
            counts = (ptr[1:] - ptr[:-1]).to(torch.int64)
            row = torch.repeat_interleave(torch.arange(r0, r1, device=ptr.device, dtype=torch.int32), counts)
        else:
            col = torch.empty(0, dtype=torch.int32, device=ptr.device)
            val = torch.empty(0, dtype=tdt, device=ptr.device)
            row = torch.empty(0, dtype=torch.int32, device=ptr.device)
        torch.cuda.current_stream().synchronize()
        from .matrix import CscMatrix
        if exchange is not None:                  # routing and exchange fused over peer memory
            h, cstarts = _assemble_over_peers(dist, torch, capi.SPL_CSC, self._nrows, self._ncols, row, col, val,
                                              exchange, False, False)
            return DistCscMatrix(CscMatrix._wrap(ctx, h), cstarts, rank, self._nrows, self._ncols)
        keys, vals, cnts = route_device(ctx, torch, capi.SPL_CSC, self._nrows, self._ncols, row, col, val, cstarts)
        rk, rv, _ = exchange_routed(dist, torch, keys, vals, cnts, group)
        torch.cuda.current_stream().synchronize()
        h = C.c_void_p()
        from .matrix import CscMatrix
        ncl = cstarts[rank + 1] - cstarts[rank]
        ctx.check(ctx._lib.spl_mat_from_packed_dev(
            ctx._h, capi.SPL_CSC, _dtype_code(self.local.dtype), self._nrows, max(ncl, 1), int(rk.numel()),
            C.c_void_p(rk.data_ptr()), C.c_void_p(rv.data_ptr()), 0, 0, C.byref(h)))
        return DistCscMatrix(CscMatrix._wrap(ctx, h), cstarts, rank, self._nrows, self._ncols)

    def spmv_peer(self, x: "PeerVector", y_dev: int):
        """y_local = A_local x with x gathered from its owners' slices (spl_spmv_peer)."""
        ctx = self.local._ctx
        st = (C.c_uint64 * (self.world + 1))(*x.starts)
        sl = (C.c_void_p * self.world)(*x.ptrs)
        ctx.check(ctx._lib.spl_spmv_peer(ctx._h, self.local._h, self.world, self.rank,
                                         C.cast(st, C.c_void_p), C.cast(sl, C.c_void_p), C.c_void_p(y_dev)))


    def halo_widths(self, dist, torch, group=None):
        """(left, right): how far the shards' stored columns reach outside their owners' slices, maximised
        over the ranks (spl_spmv_footprint + one all-reduce): the `halo` a PeerVector needs for spmv_halo."""
        ctx = self.local._ctx
        lo, hi = C.c_uint64(), C.c_uint64()
        ctx.check(ctx._lib.spl_spmv_footprint(ctx._h, self.local._h, C.byref(lo), C.byref(hi)))
        r0, r1 = self.local_rows()                    # square partition: the slice of x has the rows' bounds
        left = max(0, r0 - lo.value) if self.local.nnz() else 0
        right = max(0, hi.value + 1 - r1) if self.local.nnz() else 0
        t = torch.tensor([left, right], dtype=torch.int64, device="cuda" if torch.cuda.is_available() else "cpu")
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
        return int(t[0].item()), int(t[1].item())

    def spmv_halo(self, x: "PeerVector", y_dev: int):
        """y_local = A_local x against the rank's own slice of the published x plus its halo (filled by
        x.publish(halo=True) / x.barrier_halo()): one local array, the plain kernels (spl_spmv_window)."""
        ctx = self.local._ctx
        r0, r1 = x.starts[self.rank], x.starts[self.rank + 1]
        w0 = max(0, r0 - x.halo[0])
        w1 = min(x.n, r1 + x.halo[1])
        item = x.dtype.itemsize
        ctx.check(ctx._lib.spl_spmv_window(ctx._h, self.local._h, C.c_void_p(x.published_ptr - (r0 - w0) * item),
                                           w0, w1 - w0, C.c_void_p(y_dev)))

    def prepare_transpose(self, dist, torch, col_starts: Optional[Sequence[int]] = None, group=None):
        """One-time set-up of spmv_transpose (collective).  Every rank's footprint window [col_min, col_max + 1)
        (spl_spmv_footprint; empty for a shard without entries) travels in one all-gather; two PeerBuffers of the
        longest window hold the partials and a flag block carries the barrier.  col_starts is the column partition
        y is left in: default partition_starts(ncols, world), which is `starts` for a square matrix, so that y can
        be written straight into a PeerVector of x's partition."""
        ctx = self.local._ctx
        world = self.world
        cs = list(col_starts) if col_starts is not None else partition_starts(self._ncols, world)
        if len(cs) != world + 1 or cs[0] != 0 or cs[-1] != self._ncols or any(a > b for a, b in zip(cs, cs[1:])):
            raise ValueError("col_starts must rise from 0 to ncols in world + 1 steps")
        lo, hi = C.c_uint64(), C.c_uint64()
        ctx.check(ctx._lib.spl_spmv_footprint(ctx._h, self.local._h, C.byref(lo), C.byref(hi)))
        r0, r1 = self.local_rows()
        mine = [lo.value, hi.value + 1] if r1 > r0 and self.local.nnz() else [0, 0]
        dev = "cuda" if torch.cuda.is_available() else "cpu"
        allw = torch.empty(2 * world, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(allw, torch.tensor(mine, dtype=torch.int64, device=dev), group=group)
        windows = [int(v) for v in allw.tolist()]
        longest = max(windows[2 * g + 1] - windows[2 * g] for g in range(world))
        item = np.dtype(self.local.dtype).itemsize
        self._transpose = {"col_starts": cs, "windows": windows, "epoch": 0,
                           "parts": [PeerBuffer(ctx, dist, max(longest, 1) * item, group) for _ in range(2)],
                           "flags": PeerBuffer(ctx, dist, 4 * capi.SPL_MAX_PEERS, group)}
        dist.barrier(group=group)              # every flag block exists (and is zero) before first use

    def spmv_transpose(self, x_local_dev: int, y_local_dev: int, timeout_ms: int = 2000):
        """y = A^T x, sharded: x_local_dev holds this rank's rows' slice of x, y_local_dev receives the columns
        [col_starts[rank], col_starts[rank+1]) of y (e.g. a PeerVector's local_ptr).  Two launches on the context's
        stream, no host synchronisation: this rank's partial A_local^T x_local over its footprint window
        (spl_spmv_transpose_window), then the barrier and the sum of the ranks' partials of the own columns in
        ascending rank (spl_peer_reduce_windows).  Call prepare_transpose once first; check() reports a barrier
        that timed out (y then holds NaN).
        Product t writes partial buffer t % 2.  That buffer was last read by the peers' reduces of product t - 2,
        which every peer finished before it arrived at barrier t - 1 (stream order), and this rank passed barrier
        t - 1 before it got here: so one barrier per product is enough, as for PeerVector."""
        T = self._transpose
        ctx, world = self.local._ctx, self.world
        T["epoch"] += 1
        part = T["parts"][T["epoch"] % 2]
        ctx.check(ctx._lib.spl_spmv_transpose_window(ctx._h, self.local._h, C.c_void_p(x_local_dev),
                                                     C.c_void_p(part.local)))
        cs = (C.c_uint64 * (world + 1))(*T["col_starts"])
        win = (C.c_uint64 * (2 * world))(*T["windows"])
        pp = (C.c_void_p * world)(*part.ptrs)
        fl = (C.c_void_p * world)(*T["flags"].ptrs)
        ctx.check(ctx._lib.spl_peer_reduce_windows(
            ctx._h, _dtype_code(self.local.dtype), world, self.rank, C.cast(cs, C.c_void_p), C.cast(win, C.c_void_p),
            C.cast(pp, C.c_void_p), C.cast(fl, C.c_void_p), T["epoch"], int(timeout_ms), C.c_void_p(y_local_dev)))

    def check(self):
        """Raises if a device barrier of this rank's context timed out (synchronises the stream)."""
        t = C.c_int()
        self.local._ctx.check(self.local._ctx._lib.spl_peer_barrier_status(self.local._ctx._h, C.byref(t)))

    def close_transpose(self, dist=None, group=None):
        """Frees what prepare_transpose set up (collective when dist is given)."""
        T = getattr(self, "_transpose", None)
        if T is None:
            return
        self.local._ctx.sync()
        for b in T["parts"] + [T["flags"]]:
            b.close(dist, group)
        self._transpose = None

    @staticmethod
    def gather_groups(world: int):
        """Default blocking of a shard for spmv_gather: ring offsets where blocks begin.  One block per rank (own
        columns, then rank+1, rank+2, ...): the finest overlap of transfer and product (fastest measured on 8 GPUs).
        SPL_GATHER_GROUPS=1,1,2,4 (widths) groups consecutive peers into wider blocks (fewer passes over the rows,
        coarser overlap)."""
        env = os.environ.get("SPL_GATHER_GROUPS")
        widths = [1] * world
        if env:
            widths = [int(t) for t in env.split(",")]
            if widths[0] != 1 or sum(widths) != world or min(widths) < 1:
                raise ValueError("SPL_GATHER_GROUPS must be widths 1,... that sum to the world size")
        first = [0]
        for w in widths:
            first.append(first[-1] + w)
        return first

    def prepare_gather(self, torch, block_first=None):
        """One-time layout for spmv_gather: the shard's entries blocked by the rank that owns their column,
        own block first, then the peers in ring order (rank+1, rank+2, ...) one by one or grouped
        (block_first: ring offsets where blocks begin, default gather_groups), row order kept inside a
        block; one row-pointer array per block.  Device-side plumbing (a stable sort by block id and
        one row histogram per block); the arrays stay with the matrix."""
        from .synthetic_device import device_view
        ctx = self.local._ctx
        ctx.sync()
        r0, r1 = self.local_rows()
        nloc, nnz, G = r1 - r0, self.local.nnz(), self.world
        first = list(block_first) if block_first is not None else self.gather_groups(G)
        if first[0] != 0 or first[-1] != G or (G > 1 and first[1] != 1) or any(a >= b for a, b in zip(first, first[1:])):
            raise ValueError("block_first must increase from 0 through 1 to the world size")
        nb = len(first) - 1
        tdt = torch.float32 if self.local.dtype == np.float32 else torch.float64
        p_ptr, p_ind, p_val = self.local.device_ptrs()
        ptr = device_view(torch, p_ptr, nloc + 1, torch.int32).long()
        col = device_view(torch, p_ind, max(nnz, 1), torch.int32)[:nnz]
        val = device_view(torch, p_val, max(nnz, 1), tdt)[:nnz]
        lay = gather_block_layout(torch, ptr, col, val, self.starts, self.rank, first)
        self._gather = {"bptr": lay["bptr"], "bind": lay["bind"], "bval": lay["bval"], "first": first,
                        "stride": lay["stride"], "caps": lay["caps"],
                        "ready": torch.zeros(capi.SPL_MAX_PEERS, dtype=torch.int32, device=col.device), "epoch": 0}
        torch.cuda.current_stream().synchronize()

    def spmv_gather(self, x: "PeerVector", x_full_dev: int, y_dev: int, barrier: bool = False, timeline_dev: int = 0,
                    timeout_ms: int = 2000):
        """y_local = A_local x for a general shard with the all-gather of x fused into the product
        (spl_spmv_gather_fused): call prepare_gather once, then per product publish x and call this.
        barrier=True folds x's device-side barrier into the kernel (then do NOT call x.barrier() /
        x.publish() for this product; swap the buffers with x.swap() when the slice was rewritten)."""
        g = self._gather
        g["epoch"] += 1
        fl = None
        if barrier:
            x._epoch += 1
            fl = C.cast((C.c_void_p * self.world)(*x._flags.ptrs), C.c_void_p)
        ctx = self.local._ctx
        st = (C.c_uint64 * (self.world + 1))(*x.starts)
        sl = (C.c_void_p * self.world)(*x.ptrs)
        first = g["first"]
        bf = (C.c_uint32 * len(first))(*first)
        r0, r1 = self.local_rows()
        ctx.check(ctx._lib.spl_spmv_gather_fused(
            ctx._h, _dtype_code(self.local.dtype), r1 - r0, self.world, self.rank, C.cast(st, C.c_void_p),
            C.cast(sl, C.c_void_p), len(first) - 1, C.cast(bf, C.c_void_p), C.c_void_p(g["bptr"].data_ptr()),
            g["stride"], C.cast((C.c_uint32 * 5)(*g["caps"]), C.c_void_p), C.c_void_p(g["bind"].data_ptr()),
            C.c_void_p(g["bval"].data_ptr()), C.c_void_p(x_full_dev), C.c_void_p(y_dev),
            C.c_void_p(g["ready"].data_ptr()), g["epoch"], self.local.nnz(), fl, x._epoch if barrier else 0,
            int(timeout_ms), C.c_void_p(timeline_dev) if timeline_dev else None))

    def matvec_host(self, x: "PeerVector", x_host_local, y_host_local, timeout_ms: int = 2000):
        """`&A * &x` with this rank's slices of x and y in host memory (numpy arrays or raw host
        addresses; pinned memory lets the copies overlap): spl_spmv_peer_host.  The slice is uploaded
        into the unpublished half of `x`, published by the barrier inside the call, and gathered from."""
        ctx = self.local._ctx
        nxt_slices = x._slices[(x._cur + 1) % len(x._data)]
        st = (C.c_uint64 * (self.world + 1))(*x.starts)
        sl = (C.c_void_p * self.world)(*nxt_slices)
        fl = (C.c_void_p * self.world)(*x._flags.ptrs)
        x._epoch += 1
        xp = x_host_local if isinstance(x_host_local, int) else x_host_local.ctypes.data
        yp = y_host_local if isinstance(y_host_local, int) else y_host_local.ctypes.data
        ctx.check(ctx._lib.spl_spmv_peer_host(ctx._h, self.local._h, self.world, self.rank, C.cast(st, C.c_void_p),
                                              C.cast(sl, C.c_void_p), C.cast(fl, C.c_void_p), x._epoch, int(timeout_ms),
                                              C.c_void_p(xp), C.c_void_p(yp)))
        x._cur = (x._cur + 1) % len(x._data)


class DistCscMatrix:
    """Column block of a CSC matrix on this rank (global row indices) plus its column partition."""

    def __init__(self, local, starts: Sequence[int], rank: int, nrows: int, ncols: int):
        self.local, self.starts, self.rank = local, list(starts), int(rank)
        self.world = len(starts) - 1
        self._nrows, self._ncols = int(nrows), int(ncols)

    def nrows(self): return self._nrows
    def ncols(self): return self._ncols
    def local_cols(self): return self.starts[self.rank], self.starts[self.rank + 1]

    def mul(self, rhs: "DistCscMatrix", dist, torch, group=None) -> "DistCscMatrix":
        """Sharded `&A * &B` for column-sharded CSC operands (impl Mul for &CscMatrix, src/csc/ops/mul.rs:5-61):
        this rank's columns of A·B, with rhs's column partition.  The columns of A (this matrix) that rhs's shard's
        row indices name are gathered over peer memory, then gathered * rhs.local: bit for bit the columns of the
        unsharded product.  Collective."""
        if self._ncols != rhs._nrows:
            raise Panic("assertion `left == right` failed: self.ncols() == rhs.nrows()")
        shard = _PeerShard(self, dist, torch, group)
        try:
            gathered = shard.gather(rhs.local)
        finally:
            shard.close()
        return DistCscMatrix(gathered * rhs.local, rhs.starts, rhs.rank, self._nrows, rhs._ncols)

    def spmv(self, dist, torch, x_local, group=None):
        """y = A x with A column-sharded (this rank holds columns [c0, c1) as a CscMatrix with global row
        indices) and x sharded like the columns: the sharded form of `&A * &X` for a CscMatrix
        (src/csc/ops/mul.rs:5-61) — with A the CSC view of a row-sharded CSR matrix B it is y = B^T x.
        Every rank multiplies its column block by its slice of x (spl_spmv on the CSC block: the row
        kernels on its cached CSR form) into a full-length partial y; the partials are summed by one
        reduce-scatter, which leaves rank g with rows [rstarts[g], rstarts[g+1]) of y.  This path has
        a real exchange step (the sum over column blocks), so it uses the collective (NCCL on GPUs).
        Returns (y_rows tensor, rstarts)."""
        world, rank = self.world, self.rank
        c0, c1 = self.local_cols()
        assert x_local.numel() == c1 - c0
        rstarts = partition_starts(self._nrows, world)
        chunk = -(-self._nrows // world)
        part = torch.zeros(chunk * world, dtype=x_local.dtype, device=x_local.device)
        _torch_to_ctx(torch)
        if c1 > c0:
            self.local.spmv_device(x_local.data_ptr(), part.data_ptr())        # rows [0, nrows) of the partial
        self.local._ctx.sync()
        if world == 1:
            return part[:self._nrows], rstarts
        # equal chunks for the collective: rank g's rows are re-cut at g * chunk afterwards
        out = torch.empty(chunk, dtype=x_local.dtype, device=x_local.device)
        dist.reduce_scatter_tensor(out, part, group=group)
        lo, hi = rank * chunk, min((rank + 1) * chunk, self._nrows)
        return out[:max(hi - lo, 0)], [min(g * chunk, self._nrows) for g in range(world)] + [self._nrows]


# ------------------------------------------------------------------------- peer memory
class PeerBuffer:
    """`nbytes` of zeroed device memory on every rank, each mapped into every other rank
    (CUDA IPC; handles travel through torch.distributed's object all-gather)."""

    def __init__(self, ctx: Context, dist, nbytes: int, group=None):
        self.ctx = ctx
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        p = C.c_void_p()
        handle = (C.c_ubyte * capi.SPL_IPC_HANDLE_BYTES)()
        ctx.check(ctx._lib.spl_peer_alloc(ctx._h, int(nbytes), C.byref(p), C.cast(handle, C.c_void_p)))
        self.local = p.value
        handles = [None] * self.world
        dist.all_gather_object(handles, bytes(handle), group=group)
        self.ptrs: List[int] = []
        self._opened: List[int] = []
        for g, hb in enumerate(handles):
            if g == self.rank:
                self.ptrs.append(self.local)
                continue
            q = C.c_void_p()
            buf = (C.c_ubyte * capi.SPL_IPC_HANDLE_BYTES).from_buffer_copy(hb)
            ctx.check(ctx._lib.spl_peer_open(ctx._h, C.cast(buf, C.c_void_p), C.byref(q)))
            self.ptrs.append(q.value)
            self._opened.append(q.value)

    def close(self, dist=None, group=None):
        for q in self._opened:
            self.ctx._lib.spl_peer_close(self.ctx._h, C.c_void_p(q))
        self._opened = []
        if dist is not None:
            dist.barrier(group=group)          # nobody frees a block a peer still has mapped
        if self.local:
            self.ctx._lib.spl_peer_free(self.ctx._h, C.c_void_p(self.local))
            self.local = None


class PeerExchange:
    """Receive buffers for the fused routing + exchange of sharded assembly: every rank owns a key
    buffer (uint64) and a value buffer in peer-visible memory that all ranks can write, plus the flag
    block of the device-side barrier.  Buffers grow collectively (every rank sees the same counts) and
    are reused from call to call."""

    def __init__(self, ctx: Context, dist, group=None):
        self.ctx, self.dist, self.group = ctx, dist, group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.cap = 0
        self.vsize = 0
        self._keys = self._vals = None
        self._flags = PeerBuffer(ctx, dist, 4 * capi.SPL_MAX_PEERS, group)
        self._epoch = 0
        dist.barrier(group=group)

    def ensure(self, capacity: int, vsize: int):
        """Collective: every rank calls it with the same arguments."""
        if capacity <= self.cap and vsize <= self.vsize:
            return
        self.ctx.sync()
        for b in (self._keys, self._vals):
            if b is not None:
                b.close(self.dist, self.group)
        cap = max(int(capacity * 1.25) + 1024, 1 << 16)
        self._keys = PeerBuffer(self.ctx, self.dist, 8 * cap, self.group)
        self._vals = PeerBuffer(self.ctx, self.dist, max(vsize, self.vsize) * cap, self.group)
        self.cap, self.vsize = cap, max(vsize, self.vsize)
        self.dist.barrier(group=self.group)

    def barrier(self, timeout_ms: int = 5000):
        self._epoch += 1
        fl = (C.c_void_p * self.world)(*self._flags.ptrs)
        self.ctx.check(self.ctx._lib.spl_peer_barrier(self.ctx._h, self.world, self.rank,
                                                      C.cast(fl, C.c_void_p), self._epoch, int(timeout_ms)))

    def check(self):
        t = C.c_int()
        self.ctx.check(self.ctx._lib.spl_peer_barrier_status(self.ctx._h, C.byref(t)))

    def close(self):
        for b in (self._keys, self._vals, self._flags):
            if b is not None:
                b.close(self.dist, self.group)
        self._keys = self._vals = self._flags = None


class _PeerShard:
    """The sharded product's exchange: a major-sharded matrix (DistCsrMatrix by rows, DistCscMatrix by columns)
    published in peer memory.  __init__ is collective: one all-gather of every rank's (pointers, entries) sizes
    the three buffers (the largest shard) and gives the entry counts spl_peer_gather_rows checks the pointers
    against; the own shard is copied in with plain device-to-device copies.  gather(by) brackets
    spl_peer_gather_rows with the flag barrier: before (every shard is in place), after (nobody closes a buffer
    a peer still reads).  Nothing is kept between products."""

    def __init__(self, mat, dist, torch, group=None):
        from .synthetic_device import device_view
        L = mat.local
        self.ctx, self.dist, self.group = L._ctx, dist, group
        self.world, self.rank = mat.world, mat.rank
        self.starts = list(mat.starts)
        self.fmt, self.dtype = L._FORMAT, L.dtype
        self.nmajor = mat._nrows if self.fmt == capi.SPL_CSR else mat._ncols
        self.nminor = mat._ncols if self.fmt == capi.SPL_CSR else mat._nrows
        nloc = self.starts[self.rank + 1] - self.starts[self.rank]      # 0: the local matrix is a phantom major
        nnz = L.nnz() if nloc else 0
        dev = "cuda" if torch.cuda.is_available() else "cpu"
        mine = torch.tensor([nloc + 1, nnz], dtype=torch.int64, device=dev)
        sizes = torch.empty(2 * self.world, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(sizes, mine, group=group)
        sizes = sizes.view(self.world, 2).tolist()
        self.shard_nnz = [int(e) for _, e in sizes]
        most_p, most_e = max(p for p, _ in sizes), max(max(self.shard_nnz), 1)
        item = np.dtype(self.dtype).itemsize
        self.ex = PeerExchange(self.ctx, dist, group)                   # flag block of the barrier
        self.bufs = [PeerBuffer(self.ctx, dist, n, group) for n in (4 * most_p, 4 * most_e, item * most_e)]
        self.ctx.sync()                          # L's arrays are final on the context's stream; torch copies below
        tdt = torch.float32 if self.dtype == np.float32 else torch.float64
        p_ptr, p_ind, p_val = L.device_ptrs()
        device_view(torch, self.bufs[0].local, nloc + 1, torch.int32).copy_(device_view(torch, p_ptr, nloc + 1, torch.int32))
        if nnz:
            device_view(torch, self.bufs[1].local, nnz, torch.int32).copy_(device_view(torch, p_ind, nnz, torch.int32))
            device_view(torch, self.bufs[2].local, nnz, tdt).copy_(device_view(torch, p_val, nnz, tdt))
        torch.cuda.current_stream().synchronize()

    def gather(self, by):
        """The majors named by `by`'s minor indices, as a new local matrix of the shard's format and full height."""
        ctx, W = self.ctx, self.world
        self.ex.barrier()
        st = (C.c_uint64 * (W + 1))(*self.starts)
        nz = (C.c_uint64 * W)(*self.shard_nnz)
        sl = [(C.c_void_p * W)(*b.ptrs) for b in self.bufs]
        h = C.c_void_p()
        ctx.check(ctx._lib.spl_peer_gather_rows(
            ctx._h, self.fmt, _dtype_code(self.dtype), self.nmajor, self.nminor, W, self.rank, C.cast(st, C.c_void_p),
            C.cast(nz, C.c_void_p), C.cast(sl[0], C.c_void_p), C.cast(sl[1], C.c_void_p), C.cast(sl[2], C.c_void_p),
            by._h, C.byref(h)))
        self.ex.barrier()
        return type(by)._wrap(ctx, h)

    def close(self):
        self.ctx.sync()
        self.ex.check()                          # a barrier that gave up is reported, not a half-gathered result
        for b in self.bufs:
            b.close(self.dist, self.group)
        self.ex.close()


class PeerVector:
    """x sharded conformally with the columns: rank g's slice holds x[starts[g]:starts[g+1]] in
    peer-visible memory.  Two buffers per rank: peers read the PUBLISHED one (`ptrs`, what
    spl_spmv_peer gathers from) while the rank fills the other (`local_ptr`, e.g. as the y of its own
    product: y_t becomes x_{t+1} without a copy); `publish()` runs the device-side barrier and swaps
    them.  That is what makes one barrier per iteration enough: rank A may write its next slice while a
    slower rank B is still gathering the current one, because they are different buffers, and the
    buffer A writes at iteration t+1 is the one read at t-1, which every rank left before it arrived
    at barrier t (stream order).  With a single buffer a second, read-side barrier would be needed.
    `barrier()` is the same barrier without the swap, for products that re-read an unchanged x."""

    def __init__(self, ctx: Context, dist, n: int, dtype, starts: Optional[Sequence[int]] = None, group=None,
                 buffers: int = 2, halo: Sequence[int] = (0, 0)):
        """halo = (left, right): room for that many values before and after every rank's slice (same on all
        ranks), filled by publish(halo=True) / barrier_halo() from the neighbouring slices, so that a banded or
        stencil shard multiplies against ONE local array (DistCsrMatrix.spmv_halo)."""
        self.ctx, self.dtype = ctx, np.dtype(dtype)
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.starts = list(starts) if starts is not None else partition_starts(n, self.world)
        self.n = int(n)
        self.halo = (int(halo[0]), int(halo[1]))
        longest = max(self.starts[g + 1] - self.starts[g] for g in range(self.world))
        assert buffers in (1, 2)
        item = self.dtype.itemsize
        pad = -(-self.halo[0] * item // 256) * 256             # keeps the slices 256-byte aligned
        self._pad = pad
        self._data = [PeerBuffer(ctx, dist, pad + (max(longest, 1) + self.halo[1]) * item, group) for _ in range(buffers)]
        self._slices = [[p + pad for p in d.ptrs] for d in self._data]       # &x[starts[g]] on every rank
        self._flags = PeerBuffer(ctx, dist, 4 * capi.SPL_MAX_PEERS, group)
        self._cur = 0                          # the published buffer
        self.local_len = self.starts[self.rank + 1] - self.starts[self.rank]
        self._epoch = 0
        dist.barrier(group=group)              # every flag block exists (and is zero) before first use

    @property
    def ptrs(self) -> List[int]:
        """Every rank's slice of the published x (own slice included): what the products read."""
        return self._slices[self._cur]

    @property
    def published_ptr(self) -> int:
        return self._slices[self._cur][self.rank]

    @property
    def local_ptr(self) -> int:
        """This rank's slice of the NEXT x: write here, then publish()."""
        return self._slices[(self._cur + 1) % len(self._data)][self.rank]

    def barrier(self, timeout_ms: int = 2000):
        """Device-side barrier on the context's stream (no host synchronisation), no swap."""
        self._epoch += 1
        fl = (C.c_void_p * self.world)(*self._flags.ptrs)
        self.ctx.check(self.ctx._lib.spl_peer_barrier(self.ctx._h, self.world, self.rank,
                                                      C.cast(fl, C.c_void_p), self._epoch, int(timeout_ms)))

    def publish(self, timeout_ms: int = 2000, halo: bool = False):
        """The slice at `local_ptr` is final: barrier, then it becomes the published buffer.  halo=True also
        fills the padding around it from the neighbouring ranks' new slices (same launch as the barrier)."""
        nxt = (self._cur + 1) % len(self._data)
        if halo:
            self._barrier_halo(nxt, timeout_ms)
        else:
            self.barrier(timeout_ms)
        self._cur = nxt

    def swap(self):
        """Make the buffer at `local_ptr` the published one WITHOUT a barrier of its own: for products that carry
        the barrier themselves (DistCsrMatrix.spmv_gather(barrier=True))."""
        self._cur = (self._cur + 1) % len(self._data)

    def barrier_halo(self, timeout_ms: int = 2000):
        """Barrier + halo refresh of the published buffer, no swap."""
        self._barrier_halo(self._cur, timeout_ms)

    def _barrier_halo(self, which: int, timeout_ms: int):
        self._epoch += 1
        fl = (C.c_void_p * self.world)(*self._flags.ptrs)
        st = (C.c_uint64 * (self.world + 1))(*self.starts)
        sl = (C.c_void_p * self.world)(*self._slices[which])
        self.ctx.check(self.ctx._lib.spl_peer_barrier_halo(
            self.ctx._h, self.world, self.rank, C.cast(fl, C.c_void_p), self._epoch, int(timeout_ms),
            _dtype_code(self.dtype), C.cast(st, C.c_void_p), C.cast(sl, C.c_void_p), self.halo[0], self.halo[1]))

    def pull(self, x_full_dev: int):
        """All-gather by pulling: copies every peer's slice of the published x into the local
        full-length vector at `x_full_dev` (device address, n elements).  The own slice is left to
        the caller."""
        st = (C.c_uint64 * (self.world + 1))(*self.starts)
        sl = (C.c_void_p * self.world)(*self.ptrs)
        self.ctx.check(self.ctx._lib.spl_peer_pull(self.ctx._h, _dtype_code(self.dtype), self.world, self.rank,
                                                   C.cast(st, C.c_void_p), C.cast(sl, C.c_void_p),
                                                   C.c_void_p(x_full_dev)))

    def check(self):
        """Raises if a barrier timed out (synchronises the stream).  A product launched behind a
        barrier that timed out writes NaN, never a result computed from a half-written x."""
        t = C.c_int()
        self.ctx.check(self.ctx._lib.spl_peer_barrier_status(self.ctx._h, C.byref(t)))

    def close(self, dist=None, group=None):
        for d in self._data:
            d.close(dist, group)
        self._flags.close(dist, group)


# ------------------------------------------------------------------------- numpy stand-ins (tests)
def route_numpy(nrows: int, ncols: int, row, col, val, starts):
    """What spl_coo_route_dev computes, in numpy (CSR): used by the CPU gloo tests to drive the
    host logic, and by the GPU tests as the checker of the device routing."""
    row = np.asarray(row, np.uint64)
    col = np.asarray(col, np.uint64)
    b = np.asarray(starts[1:-1], np.uint64)
    owner = np.searchsorted(b, row, side="right")
    order = np.argsort(owner, kind="stable")
    base = np.asarray(starts, np.uint64)[owner]
    keys = ((row - base) << np.uint64(bits_for(ncols))) | col
    counts = np.bincount(owner, minlength=len(starts) - 1).tolist()
    return keys[order].astype(np.uint64), np.asarray(val)[order], counts


def reduce_windows_numpy(col_starts, windows, partials, rank: int, dtype):
    """What spl_peer_reduce_windows writes on `rank`, in numpy: for every column c of the rank's slice, the partials
    of the ranks whose window [windows[2g], windows[2g+1]) holds c, folded in ascending rank (the first copied, the
    others added in `dtype`), +0.0 where no window holds c.  partials[g][j] is rank g's value of column
    windows[2g] + j."""
    c0, c1 = int(col_starts[rank]), int(col_starts[rank + 1])
    y = np.zeros(c1 - c0, dtype)
    have = np.zeros(c1 - c0, bool)
    for g in range(len(col_starts) - 1):
        lo, hi = int(windows[2 * g]), int(windows[2 * g + 1])
        a, b = max(lo, c0), min(hi, c1)
        if a >= b:
            continue
        seg = np.asarray(partials[g], dtype)[a - lo:b - lo]
        s = slice(a - c0, b - c0)
        with np.errstate(invalid="ignore", over="ignore"):
            y[s] = np.where(have[s], y[s] + seg, seg)
        have[s] = True
    return y


def unpack_keys(keys, ncols: int):
    mb = np.uint64(bits_for(ncols))
    keys = np.asarray(keys, np.uint64)
    return keys >> mb, keys & ((np.uint64(1) << mb) - np.uint64(1))
