"""The exchange of the row-sharded sparse product (spl_peer_gather_rows) on one GPU, and the DistCsrMatrix /
DistCscMatrix `mul` front end with a one-rank NCCL group.

The ranks are emulated with plain device tensors as the "peer" slices: the call waits on nobody, so every rank's
gather runs on its own.  Each rank's gathered matrix must equal a numpy selection of the whole matrix's majors bit
for bit, and the local product with it must equal that rank's block of the oracle's product of the whole problem
bit for bit."""
import ctypes as C
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist

import oracle as orc
from spalinalg_b200 import dist as spd

pytestmark = pytest.mark.gpu

CSR, CSC = 0, 1


def _t(a, dt):
    return torch.from_numpy(np.ascontiguousarray(a).astype(dt)).cuda()


def _compress(nmajor, nminor, rows, cols, vals):
    """CSR arrays of (rows = majors, cols = minors), duplicates summed (oracle assembly)."""
    return orc.compress_from_coo(nmajor, nminor, orc.make_triplets(rows, cols, vals), "row")


def banded(nmaj, nmin, half, dtype, seed):
    """Major i holds minors around i * nmin / nmaj: one long run per shard, a halo across the owner boundaries."""
    rng = np.random.default_rng(seed)
    i = np.repeat(np.arange(nmaj), 2 * half + 1)
    c = (i * nmin) // nmaj + np.tile(np.arange(-half, half + 1), nmaj)
    keep = (c >= 0) & (c < nmin)
    return _compress(nmaj, nmin, i[keep], c[keep], rng.standard_normal(int(keep.sum())).astype(dtype))


def random_sparse(nmaj, nmin, per, dtype, seed, empty_every=0):
    """`per` random minors per major; every `empty_every`-th major empty."""
    rng = np.random.default_rng(seed)
    i = np.repeat(np.arange(nmaj), per)
    c = rng.integers(0, nmin, len(i))
    if empty_every:
        keep = i % empty_every != 0
        i, c = i[keep], c[keep]
    return _compress(nmaj, nmin, i, c, rng.standard_normal(len(i)).astype(dtype))


def power_law(nmaj, nmin, dtype, seed):
    """Major lengths from a power law: some majors hold many ring chunks (tens of thousands of entries)."""
    rng = np.random.default_rng(seed)
    lens = np.minimum((rng.pareto(1.1, nmaj) * 3).astype(np.int64) + 1, nmin // 2)
    lens[rng.integers(0, nmaj, 4)] = nmin // 2
    i = np.repeat(np.arange(nmaj), lens)
    c = rng.integers(0, nmin, len(i))                       # duplicates summed: lengths shrink a little
    return _compress(nmaj, nmin, i, c, rng.standard_normal(len(i)).astype(dtype))


def special_values(val, dtype):
    """-0.0, NaN payloads and subnormals scattered over the values (copied bit for bit, never computed with)."""
    v = val.copy()
    u = v.view(np.uint32 if dtype == np.float32 else np.uint64)
    nan = np.array([0x7fc00123, 0xffc00abc] if dtype == np.float32 else
                   [0x7ff8000000000123, 0xfff0000000000abc], dtype=u.dtype)
    sub = np.array([1, 0x80000005] if dtype == np.float32 else [1, 0x8000000000000007], dtype=u.dtype)
    u[0::7] = nan[0]
    u[3::11] = nan[1]
    u[5::13] = sub[0]
    u[6::17] = sub[1]
    v[2::19] = -0.0
    return v


def shard(full, starts, g):
    ptr, ind, val = full
    a, b = starts[g], starts[g + 1]
    lo, hi = int(ptr[a]), int(ptr[b])
    return (ptr[a:b + 1] - ptr[a]).astype(np.uint64), ind[lo:hi], val[lo:hi]


class Slices:
    """Every rank's shard of a major-sharded matrix in separate device tensors (uint32 pointers, uint32 indices,
    values), the index and value slices starting `shift[g]` elements into their allocation so that the sources sit at
    every alignment modulo 16 bytes."""

    def __init__(self, full, starts, dtype, shift=None):
        W = len(starts) - 1
        self.starts, self.keep = list(starts), []
        self.ptr, self.ind, self.val, self.nnz = [], [], [], []
        for g in range(W):
            p, i, v = shard(full, starts, g)
            s = shift[g] if shift else 0
            pt = _t(p, np.int32)
            it = torch.zeros(len(i) + s + 4, dtype=torch.int32, device="cuda")
            vt = torch.zeros(len(v) + s + 4, dtype=torch.float32 if dtype == np.float32 else torch.float64, device="cuda")
            it[s:s + len(i)] = _t(i, np.int32)
            vt[s:s + len(v)] = torch.from_numpy(v.copy()).cuda()
            self.keep += [pt, it, vt]
            self.ptr.append(pt.data_ptr())
            self.ind.append(it[s:].data_ptr())
            self.val.append(vt[s:].data_ptr())
            self.nnz.append(len(i))

    def snapshot(self):
        return [t.cpu().numpy().tobytes() for t in self.keep]


def gather(ctx, fmt, dtype, nmajor, nminor, world, rank, sl, by, starts=None, nnz=None, ptrs=None):
    """spl_peer_gather_rows; returns (status, handle)."""
    from spalinalg_b200 import _capi as capi
    starts = sl.starts if starts is None else starts
    nnz = sl.nnz if nnz is None else nnz
    W = max(world, 1)
    arr = lambda xs: C.cast((C.c_void_p * W)(*(list(xs) + [None] * W)[:W]), C.c_void_p)
    st = (C.c_uint64 * (len(starts)))(*starts)
    nz = (C.c_uint64 * max(len(nnz), 1))(*nnz)
    h = C.c_void_p(0xdead)
    status = ctx._lib.spl_peer_gather_rows(
        ctx._h, fmt, capi.SPL_F32 if dtype == np.float32 else capi.SPL_F64, nmajor, nminor, world, rank,
        C.cast(st, C.c_void_p), C.cast(nz, C.c_void_p), arr(ptrs[0] if ptrs else sl.ptr),
        arr(ptrs[1] if ptrs else sl.ind), arr(ptrs[2] if ptrs else sl.val), by._h if by is not None else None,
        C.byref(h))
    return status, h


def expected_gather(full, nmajor, named):
    """Full-height arrays holding the named majors of `full`, every other major empty."""
    ptr, ind, val = full
    mark = np.zeros(nmajor, bool)
    mark[np.asarray(named, np.int64)] = True
    lens = np.where(mark, np.diff(ptr.astype(np.int64)), 0)
    sel = np.repeat(mark, np.diff(ptr.astype(np.int64)))
    return np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64), ind[sel], val[sel]


def same_bits(got, want):
    """Bit for bit, except that a NaN may carry another payload: IEEE arithmetic on a NaN operand (the products
    here) does not fix the payload of its result, on the device or in the oracle.  The gathered matrices, which are
    copies, are compared on every bit."""
    nan = np.isnan(want)
    return bool(np.array_equal(np.isnan(got), nan) and got[~nan].tobytes() == want[~nan].tobytes())


def check_product(fmt, dtype, m, k, n, A, B, a_starts, b_starts, b_shift=None):
    """A (m x k) and B (k x n) as CSR arrays (fmt CSR: row-sharded, A's rows by a_starts, B's by b_starts) or as
    CSC arrays (fmt CSC: column-sharded, A's columns by a_starts, B's by b_starts).  Every rank gathers what its
    shard of the local operand names and multiplies; gathered matrix and block of C are compared bit for bit."""
    import spalinalg_b200 as sp
    ctx = sp.default_context()
    W = len(a_starts) - 1
    Mat = sp.CsrMatrix if fmt == CSR else sp.CscMatrix
    if fmt == CSR:
        whole = orc.csr_mul(m, k, n, A, B)
        src, src_major, src_minor, by_full, by_starts = B, k, n, A, a_starts
    else:
        whole = orc.csr_mul(n, k, m, B, A)                       # CSC(A*B) arrays = CSR(B^T A^T) arrays
        src, src_major, src_minor, by_full, by_starts = A, k, m, B, b_starts
    sl = Slices(src, b_starts if fmt == CSR else a_starts, dtype, b_shift)
    before = sl.snapshot()
    for g in range(W):
        bp, bi, bv = shard(by_full, by_starts, g)
        nloc = by_starts[g + 1] - by_starts[g]
        if nloc == 0:                                           # the phantom major of a rank that owns nothing
            bp = np.zeros(2, np.uint64)
        loc = Mat.new(max(nloc, 1), k, bp, bi, bv) if fmt == CSR else Mat.new(k, max(nloc, 1), bp, bi, bv)
        status, h = gather(ctx, fmt, dtype, src_major, src_minor, W, g, sl, loc)
        ctx.check(status)
        got = Mat._wrap(ctx, h)
        assert got.shape() == ((src_major, src_minor) if fmt == CSR else (src_minor, src_major))
        wp, wi, wv = expected_gather(src, src_major, bi)
        gp, gi, gv = got._download()
        assert np.array_equal(gp, wp) and np.array_equal(gi, wi) and gv.tobytes() == wv.tobytes()
        prod = loc * got if fmt == CSR else got * loc
        cp, ci, cv = prod._download()
        if nloc:
            ep, ei, ev = shard(whole, by_starts, g)
            assert np.array_equal(cp, ep) and np.array_equal(ci, ei)
            assert same_bits(cv, ev)
        else:
            assert prod.nnz() == 0
    ctx.sync()
    assert sl.snapshot() == before                              # the shards are only read


@pytest.mark.parametrize("fmt", [CSR, CSC])
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("shape", ["banded", "random", "power_law"])
def test_gather_rows_matches_oracle(fmt, dtype, world, shape):
    """S = the gathered operand (B for CSR, A for CSC: k majors), Y = the operand whose minor indices name them (A
    for CSR, B for CSC), generated the same way for both formats.  Non-square: A is m x k, B is k x n."""
    m, k, n = 20011, 30011, 17011
    s_min, y_maj = (n, m) if fmt == CSR else (m, n)
    if shape == "banded":
        Y = banded(y_maj, k, 3, dtype, 1)
        S = banded(k, s_min, 4, dtype, 2)
    elif shape == "random":
        Y = random_sparse(y_maj, k, 1 if world < 3 else 2, dtype, 3)     # few named majors: runs of one
        S = random_sparse(k, s_min, 12, dtype, 4, empty_every=5)        # some named majors are empty
    else:
        Y = random_sparse(y_maj, k, 3, dtype, 5)
        S = power_law(k, s_min, dtype, 6)
    S = (S[0], S[1], special_values(S[2], dtype))
    Y = (Y[0], Y[1], special_values(Y[2], dtype))
    A, B = (Y, S) if fmt == CSR else (S, Y)
    a_major, b_major = (m, k) if fmt == CSR else (k, n)
    a_starts = spd.partition_starts(a_major, world)
    b_starts = spd.partition_starts(b_major, world)
    if world == 3:                                              # a rank that owns nothing, on both sides
        a_starts = [0, 0, a_major // 3, a_major]
        b_starts = [0, b_major // 2, b_major // 2, b_major]
    per = 4 if dtype == np.float32 else 2                       # slices at every 16-byte alignment
    check_product(fmt, dtype, m, k, n, A, B, a_starts, b_starts, [g % per for g in range(world)])


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_gather_rows_every_misalignment(dtype):
    """Long runs whose source and output positions take every pair of offsets modulo 16 bytes (the bulk-copy path
    stores each landed stage at the shift between the two), from slices that start at every alignment."""
    rng = np.random.default_rng(7)
    k, n = 600, 400000
    i = np.repeat(np.arange(k), rng.integers(4300, 9000, k))
    B = _compress(k, n, i, rng.integers(0, n, len(i)), rng.standard_normal(len(i)).astype(dtype))
    B = (B[0], B[1], special_values(B[2], dtype))
    lens = np.diff(B[0].astype(np.int64))
    assert lens.min() >= 4096                                   # every row is a long run
    named = np.arange(0, k, 2)                                  # no two adjacent: every named row a run of its own
    per = 4 if dtype == np.float32 else 2
    pairs = set()
    src_pos, dst_pos = B[0][named].astype(np.int64), np.concatenate([[0], np.cumsum(lens[named])[:-1]])
    for s in range(per):
        pairs |= set(zip(((src_pos + s) % per).tolist(), (dst_pos % per).tolist()))
    assert len(pairs) == per * per                              # every relative misalignment occurs
    m = 3
    A = _compress(m, k, np.repeat(np.arange(m), 100), named.reshape(m, 100).ravel(), np.ones(300, dtype))
    for s in range(per):
        check_product(CSR, dtype, m, k, n, A, B, [0, m], [0, k], [s])
        check_product(CSR, dtype, m, k, n, A, B, [0, 1, m], [0, 250, k], [s, (s + 1) % per])


def test_gather_rows_empty_by():
    """`by` without entries: the result has nnz 0 and an all-zero pointer array."""
    import spalinalg_b200 as sp
    ctx = sp.default_context()
    B = banded(5000, 3000, 2, np.float64, 1)
    sl = Slices(B, [0, 2500, 5000], np.float64)
    by = sp.CsrMatrix.new(7, 5000, np.zeros(8, np.uint64), np.zeros(0, np.uint64), np.zeros(0))
    status, h = gather(ctx, CSR, np.float64, 5000, 3000, 2, 1, sl, by)
    ctx.check(status)
    g = sp.CsrMatrix._wrap(ctx, h)
    assert g.shape() == (5000, 3000) and g.nnz() == 0 and not g.rowptr().any()


def test_gather_rows_refusals(monkeypatch):
    """Every refusal: the status, *out NULL, and nothing written to the shards or to `by`."""
    import spalinalg_b200 as sp
    from spalinalg_b200 import _capi as capi
    ctx = sp.default_context()
    k, n = 4000, 3000
    B = random_sparse(k, n, 5, np.float64, 9)
    starts = [0, 1500, k]
    sl = Slices(B, starts, np.float64)
    A = random_sparse(50, k, 4, np.float64, 10)
    by = sp.CsrMatrix.new(50, k, *A)
    by32 = sp.CsrMatrix.new(50, k, A[0], A[1], A[2].astype(np.float32))
    by_csc = sp.CscMatrix.new(k, 50, *A)                      # CSC k x 50: minor dimension k, like `by`
    before, by_before = sl.snapshot(), by._download()
    E = capi
    cases = [
        (E.SPL_ERR_SHAPE, dict(nmajor=k + 1, starts=[0, 1500, k + 1])),       # by's minor dimension != nmajor
        (E.SPL_ERR_SHAPE, dict(starts=[0, 1500, k - 1])),                     # starts[world] != nmajor
        (E.SPL_ERR_ARG, dict(world=0, starts=[0])),
        (E.SPL_ERR_ARG, dict(world=9, starts=[0] * 9 + [k], nnz=[0] * 9)),
        (E.SPL_ERR_ARG, dict(rank=2)),
        (E.SPL_ERR_ARG, dict(rank=-1)),
        (E.SPL_ERR_ARG, dict(starts=[0, 3000, 1500, k], world=3, nnz=sl.nnz + [0])),   # decreasing
        (E.SPL_ERR_ARG, dict(ptrs=(sl.ptr, [sl.ind[0], None], sl.val))),      # NULL slice of an owner
        (E.SPL_ERR_ARG, dict(by=by32)),                                       # another scalar type
        (E.SPL_ERR_ARG, dict(by=by_csc)),                                     # another format
    ]
    for want, kw in cases:
        args = dict(fmt=CSR, dtype=np.float64, nmajor=k, nminor=n, world=2, rank=0, by=by)
        args.update({key: kw[key] for key in ("nmajor", "world", "rank", "by") if key in kw})
        status, h = gather(ctx, args["fmt"], args["dtype"], args["nmajor"], args["nminor"], args["world"],
                           args["rank"], sl, args["by"], starts=kw.get("starts"), nnz=kw.get("nnz"),
                           ptrs=kw.get("ptrs"))
        assert status == want, (kw, status)
        assert h.value is None, kw
    # a corrupted shard pointer array (found on the device, before any index or value is read): a descending pair
    # and a pointer past the shard's entry count, each on a named row
    named = int(A[1][0])
    owner = 0 if named < 1500 else 1
    local = named - starts[owner]
    for bad in ("descend", "past"):
        p = sl.keep[3 * owner]
        saved = p.clone()
        if bad == "descend":
            p[local + 1] = max(int(p[local].item()) - 1, 0)
            p[local] = int(saved[local + 1].item())
        else:
            p[local + 1] = sl.nnz[owner] + 1
        snap = sl.snapshot()
        status, h = gather(ctx, CSR, np.float64, k, n, 2, 0, sl, by)
        assert status == E.SPL_ERR_ARG and h.value is None
        assert sl.snapshot() == snap
        p.copy_(saved)
    # a gathered total of 2^32 - 65536 entries or more: two shards that claim 3e9 entries in one named row each
    # (refused after the counting pass, before anything is copied)
    big = 3_000_000_000
    fake = [_t(np.array([0, big], np.uint64).astype(np.uint32), np.int32) for _ in range(2)]
    tiny = torch.zeros(16, dtype=torch.float64, device="cuda")
    two = sp.CsrMatrix.new(1, 2, np.array([0, 2], np.uint64), np.array([0, 1], np.uint64), np.ones(2))
    status, h = gather(ctx, CSR, np.float64, 2, 5, 2, 0, sl, two, starts=[0, 1, 2], nnz=[big, big],
                       ptrs=([f.data_ptr() for f in fake], [tiny.data_ptr()] * 2, [tiny.data_ptr()] * 2))
    assert status == E.SPL_ERR_UNSUPPORTED and h.value is None
    # a wide `by` (64-bit positions)
    monkeypatch.setenv("SPL_WIDE_MIN_NNZ", "10")
    wide = sp.CsrMatrix.new(50, k, *A)
    assert wide.device_ptr64()
    status, h = gather(ctx, CSR, np.float64, k, n, 2, 0, sl, wide)
    assert status == E.SPL_ERR_UNSUPPORTED and h.value is None
    ctx.sync()
    assert sl.snapshot() == before
    bp, bi, bv = by._download()
    assert np.array_equal(bp, by_before[0]) and np.array_equal(bi, by_before[1]) and bv.tobytes() == by_before[2].tobytes()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_dist_mul_world1_nccl():
    """DistCsrMatrix.mul and DistCscMatrix.mul with a one-rank NCCL group: the same host code as the multi-GPU
    runs (peer buffers, flag barriers, gather, local product), bit for bit against the oracle; each called twice
    (the peer buffers are set up and closed per product)."""
    import spalinalg_b200 as sp
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{_free_port()}", rank=0, world_size=1,
                            device_id=torch.device("cuda", 0))
    try:
        ctx = sp.default_context()
        m, k, n = 3001, 2003, 1501
        A = random_sparse(m, k, 6, np.float64, 11)
        B = power_law(k, n, np.float64, 12)
        whole = orc.csr_mul(m, k, n, A, B)
        dA = spd.DistCsrMatrix(sp.CsrMatrix.new(m, k, *A, ctx=ctx), [0, m], 0, m, k)
        dB = spd.DistCsrMatrix(sp.CsrMatrix.new(k, n, *B, ctx=ctx), [0, k], 0, k, n)
        for _ in range(2):
            P = dA.mul(dB, dist, torch)
            assert (P.nrows(), P.ncols(), P.starts) == (m, n, [0, m])
            p = P.local._download()
            assert np.array_equal(p[0], whole[0]) and np.array_equal(p[1], whole[1]) and p[2].tobytes() == whole[2].tobytes()
        with pytest.raises(sp.Panic):
            dB.mul(dB, dist, torch)
        Ac, Bc = orc.recompress(m, k, *A), orc.recompress(k, n, *B)
        wc = orc.csr_mul(n, k, m, Bc, Ac)
        cA = spd.DistCscMatrix(sp.CscMatrix.new(m, k, *Ac, ctx=ctx), [0, k], 0, m, k)
        cB = spd.DistCscMatrix(sp.CscMatrix.new(k, n, *Bc, ctx=ctx), [0, n], 0, k, n)
        for _ in range(2):
            Q = cA.mul(cB, dist, torch)
            assert (Q.nrows(), Q.ncols(), Q.starts) == (m, n, [0, n])
            q = Q.local._download()
            assert np.array_equal(q[0], wc[0]) and np.array_equal(q[1], wc[1]) and q[2].tobytes() == wc[2].tobytes()
    finally:
        dist.destroy_process_group()
