"""The row-sharded transposed product y = A^T x (spl_spmv_transpose_window + spl_peer_reduce_windows) on one GPU, and
the DistCsrMatrix.spmv_transpose front end with a one-rank NCCL group.

The ranks are emulated one after another with plain device tensors as the "peer" partial buffers and no flag
barrier (flag_ptrs NULL): first every rank's window product, then every rank's reduce.  The result is checked
  * bit for bit against a numpy restatement of the sum order (dist.reduce_windows_numpy over the partials the row
    kernels compute) wherever the row kernels run one lane per row, and against the oracle for world 1;
  * against the oracle's A^T x within the SpMV tolerance everywhere;
  * bit for bit between two runs."""
import ctypes as C
import socket

import numpy as np
import pytest
import torch

import oracle as orc
from spalinalg_b200 import dist as spd

CSR, CSC = 0, 1
RTOL = {np.float64: 1e-12, np.float32: 1e-5}


def _compress(nmajor, nminor, rows, cols, vals):
    return orc.compress_from_coo(nmajor, nminor, orc.make_triplets(rows, cols, vals), "row")


def band9(n, dtype, seed):
    rng = np.random.default_rng(seed)
    i = np.repeat(np.arange(n), 9)
    c = i + np.tile(np.arange(-4, 5), n)
    keep = (c >= 0) & (c < n)
    return _compress(n, n, i[keep], c[keep], rng.standard_normal(int(keep.sum())).astype(dtype))


def random16(m, n, dtype, seed):
    rng = np.random.default_rng(seed)
    i = np.repeat(np.arange(m), 16)
    return _compress(m, n, i, rng.integers(0, n, len(i)), rng.standard_normal(len(i)).astype(dtype))


def power_law(m, n, dtype, seed):
    """Row lengths from a power law, columns crowded towards 0: the transpose has a few very long rows."""
    rng = np.random.default_rng(seed)
    lens = np.minimum((rng.pareto(1.2, m) * 3).astype(np.int64) + 1, n // 4)
    i = np.repeat(np.arange(m), lens)
    c = (n * rng.random(len(i)) ** 2).astype(np.int64)
    return _compress(m, n, i, c, rng.standard_normal(len(i)).astype(dtype))


def scaled_band(m, n, dtype, seed):
    """Non-square: row i holds the 5 columns around i * n / m."""
    rng = np.random.default_rng(seed)
    i = np.repeat(np.arange(m), 5)
    c = (i * n) // m + np.tile(np.arange(-2, 3), m)
    keep = (c >= 0) & (c < n)
    return _compress(m, n, i[keep], c[keep], rng.standard_normal(int(keep.sum())).astype(dtype))


def shard(full, starts, g):
    ptr, ind, val = full
    a, b = starts[g], starts[g + 1]
    lo, hi = int(ptr[a]), int(ptr[b])
    return (ptr[a:b + 1] - ptr[a]).astype(np.uint64), ind[lo:hi], val[lo:hi]


def local_matrix(sp, full, starts, g, ncols, ctx):
    p, i, v = shard(full, starts, g)
    if starts[g + 1] == starts[g]:                              # the phantom row of a rank that owns nothing
        p = np.zeros(2, np.uint64)
    return sp.CsrMatrix.new(max(starts[g + 1] - starts[g], 1), ncols, p, i, v, ctx=ctx)


def window_of(full, starts, g):
    _, i, _ = shard(full, starts, g)
    return (int(i.min()), int(i.max()) + 1) if len(i) else (0, 0)


def window_transpose(full, starts, g, ncols):
    """CSR arrays of the transpose of rank g's shard restricted to its window (rows = columns lo .. hi - 1)."""
    p, i, v = shard(full, starts, g)
    lo, hi = window_of(full, starts, g)
    nloc = starts[g + 1] - starts[g]
    tp, ti, tv = orc.recompress(nloc, ncols, p, i, v)
    a, b = int(tp[lo]), int(tp[hi])
    return (tp[lo:hi + 1] - tp[lo]).astype(np.uint64), ti[a:b], tv[a:b]


def model_partial(full, starts, g, ncols, x):
    """Rank g's partial as the row kernels compute it with one lane per row: every row of the windowed transpose
    summed over ascending rows of A.  Their sums start at +0.0, so a row whose products are all zeros is +0.0
    (the oracle, which copies the first product, keeps a lone -0.0 there)."""
    lo, hi = window_of(full, starts, g)
    if hi == lo:
        return np.zeros(0, x.dtype)
    tp, ti, tv = window_transpose(full, starts, g, ncols)
    p = orc.csr_spmv(hi - lo, tp, ti, tv, x[starts[g]:starts[g + 1]])
    p[p == 0] = 0
    return p


def one_lane(sp, full, starts, g, ncols, ctx):
    """True when the planner runs rank g's windowed transpose with one lane per row (same arrays, same plan)."""
    lo, hi = window_of(full, starts, g)
    if hi == lo:
        return True
    nloc = starts[g + 1] - starts[g]
    T = sp.CsrMatrix.new(hi - lo, nloc, *window_transpose(full, starts, g, ncols), ctx=ctx)
    kernel, lanes = T.spmv_choice()
    return kernel != 3 and lanes == 1                           # 3 = SPL_SPMV_SPLIT


def oracle_transpose(full, nrows, ncols, x):
    """(A^T x, |A|^T |x|) from the oracle's transpose and SpMV."""
    tp, ti, tv = orc.recompress(nrows, ncols, *full)
    y = orc.csr_spmv(ncols, tp, ti, tv, x)
    scale = orc.csr_spmv(ncols, tp, ti, np.abs(tv).astype(np.float64), np.abs(x).astype(np.float64))
    return y, scale


def same_bits(got, want):
    """Bit for bit; a NaN may carry another payload (IEEE arithmetic does not fix it)."""
    nan = np.isnan(want)
    return bool(np.array_equal(np.isnan(got), nan) and got[~nan].tobytes() == want[~nan].tobytes())


def _tdt(dtype):
    return torch.float32 if dtype == np.float32 else torch.float64


def _code(dtype):
    from spalinalg_b200 import _capi as capi
    return capi.SPL_F32 if dtype == np.float32 else capi.SPL_F64


def transpose_window(ctx, a, x_ptr, y_ptr):
    return ctx._lib.spl_spmv_transpose_window(ctx._h, a._h if a is not None else None, C.c_void_p(x_ptr),
                                              C.c_void_p(y_ptr))


def reduce_windows(ctx, dtype, world, rank, col_starts, windows, partials, y_ptr, flags=None, epoch=0):
    W = max(world, 1)
    arr = lambda xs: C.cast((C.c_void_p * W)(*(list(xs) + [None] * W)[:W]), C.c_void_p)
    cs = (C.c_uint64 * max(len(col_starts), 1))(*col_starts)
    win = (C.c_uint64 * max(len(windows), 2))(*windows)
    return ctx._lib.spl_peer_reduce_windows(ctx._h, _code(dtype), world, rank, C.cast(cs, C.c_void_p),
                                            C.cast(win, C.c_void_p), arr(partials), arr(flags) if flags else None,
                                            epoch, 2000, C.c_void_p(y_ptr))


class Emulated:
    """Every rank of a row-sharded matrix on this GPU: its shard, its slice of x, its partial buffer (starting
    `shift` elements into the allocation, so that windows at odd columns are not 16-byte aligned) and its slice of
    y (the same shift)."""

    def __init__(self, sp, ctx, full, nrows, ncols, rs, cs, x, dtype, shift=0, fill=7.0):
        self.sp, self.ctx, self.full, self.rs, self.cs, self.dtype = sp, ctx, full, list(rs), list(cs), dtype
        self.ncols, self.W = ncols, len(rs) - 1
        self.mats = [local_matrix(sp, full, rs, g, ncols, ctx) for g in range(self.W)]
        self.windows = []
        for g in range(self.W):
            lo, hi = C.c_uint64(), C.c_uint64()
            ctx.check(ctx._lib.spl_spmv_footprint(ctx._h, self.mats[g]._h, C.byref(lo), C.byref(hi)))
            self.windows += [lo.value, hi.value + 1] if self.mats[g].nnz() else [0, 0]
        assert self.windows == sum((list(window_of(full, rs, g)) for g in range(self.W)), [])
        tdt = _tdt(dtype)
        self.x = [torch.from_numpy(np.ascontiguousarray(x[rs[g]:rs[g + 1]]).copy()).cuda() if rs[g + 1] > rs[g]
                  else torch.zeros(1, dtype=tdt, device="cuda") for g in range(self.W)]
        self.parts = [torch.full((self.windows[2 * g + 1] - self.windows[2 * g] + shift + 1,), 5.0, dtype=tdt,
                                 device="cuda") for g in range(self.W)]
        self.ys = [torch.full((cs[g + 1] - cs[g] + shift + 1,), fill, dtype=tdt, device="cuda") for g in range(self.W)]
        self.shift = shift

    def part_ptr(self, g):
        return self.parts[g][self.shift:].data_ptr()

    def run(self):
        ctx = self.ctx
        for g in range(self.W):
            ctx.check(transpose_window(ctx, self.mats[g], self.x[g].data_ptr(), self.part_ptr(g)))
        for g in range(self.W):
            ctx.check(reduce_windows(ctx, self.dtype, self.W, g, self.cs, self.windows,
                                     [self.part_ptr(g2) for g2 in range(self.W)], self.ys[g][self.shift:].data_ptr()))
        ctx.sync()
        torch.cuda.synchronize()
        y = np.concatenate([self.ys[g][self.shift:self.shift + self.cs[g + 1] - self.cs[g]].cpu().numpy()
                            for g in range(self.W)])
        parts = [self.parts[g][self.shift:self.shift + self.windows[2 * g + 1] - self.windows[2 * g]].cpu().numpy()
                 for g in range(self.W)]
        return y, parts

    def model(self, x):
        parts = [model_partial(self.full, self.rs, g, self.ncols, x) for g in range(self.W)]
        y = np.concatenate([spd.reduce_windows_numpy(self.cs, self.windows, parts, g, self.dtype) for g in range(self.W)])
        return y, parts

    def one_lane(self):
        return all(one_lane(self.sp, self.full, self.rs, g, self.ncols, self.ctx) for g in range(self.W))


# ----------------------------------------------------------------------------------------------------- CPU
def test_reduce_windows_numpy_by_hand():
    """The restatement of the sum order on a tiny case worked out by hand: columns 0..9, slices [0, 4) [4, 7)
    [7, 10), windows rank 0 [1, 5), rank 1 [3, 8), rank 2 empty.  Ascending rank, first term copied (-0.0 kept),
    no window -> +0.0."""
    cs = [0, 4, 7, 10]
    win = [1, 5, 3, 8, 0, 0]
    p0 = np.array([1.0, -0.0, 0.5, 2.0])                       # columns 1, 2, 3, 4
    p1 = np.array([0.25, -0.0, 3.0, 4.0, 5.0])                 # columns 3, 4, 5, 6, 7
    parts = [p0, p1, np.zeros(0)]
    y = np.concatenate([spd.reduce_windows_numpy(cs, win, parts, g, np.float64) for g in range(3)])
    want = np.array([0.0, 1.0, -0.0, 0.5 + 0.25, 2.0 + -0.0, 3.0, 4.0, 5.0, 0.0, 0.0])
    assert y.tobytes() == want.tobytes()
    assert np.signbit(y[2]) and not np.signbit(y[0]) and not np.signbit(y[8]) and not np.signbit(y[4])
    # the order is the ranks', not the values': (a + b) + c != a + (b + c) in f32 here
    a, b, c = np.float32(1e8), np.float32(-1e8), np.float32(1.0)
    win1 = [0, 1, 0, 1, 0, 1]
    y1 = spd.reduce_windows_numpy([0, 1, 1, 1], win1, [np.array([a]), np.array([b]), np.array([c])], 0, np.float32)
    assert y1[0] == np.float32(1.0)
    y2 = spd.reduce_windows_numpy([0, 1, 1, 1], win1, [np.array([c]), np.array([a]), np.array([b])], 0, np.float32)
    assert y2[0] == np.float32(0.0)


# ----------------------------------------------------------------------------------------------------- GPU
SHAPES = ["band9", "random16", "power_law", "nonsquare", "balanced_empty"]


def make_case(shape, world, dtype):
    n = 20011
    if shape == "band9":
        return band9(n, dtype, 1), n, n, spd.partition_starts(n, world), None
    if shape == "random16":
        return random16(n, n, dtype, 2), n, n, spd.partition_starts(n, world), None
    if shape == "power_law":
        return power_law(n, n, dtype, 3), n, n, spd.partition_starts(n, world), None
    if shape == "nonsquare":
        m, k = 20011, 30011
        return scaled_band(m, k, dtype, 4), m, k, spd.partition_starts(m, world), spd.partition_starts(k, world)
    # power-law rows with an nnz-balanced row partition, then one rank given no rows
    full = power_law(n, n, dtype, 5)
    bins = np.diff(full[0].astype(np.int64))
    rs = spd.balanced_starts(bins, 1, n, max(world - 1, 1))
    if world > 1:
        rs = rs[:1] + [0] + rs[1:] if world == 2 else rs[:2] + [rs[1]] + rs[2:]
    assert len(rs) == world + 1 and (world == 1 or any(a == b for a, b in zip(rs, rs[1:])))
    return full, n, n, rs, None


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("world", [1, 2, 3, 8])
@pytest.mark.parametrize("shape", SHAPES)
def test_spmv_transpose_matches_oracle(shape, world, dtype):
    import spalinalg_b200 as sp
    ctx = sp.default_context()
    full, m, n, rs, cs = make_case(shape, world, dtype)
    cs = cs if cs is not None else rs
    x = np.random.default_rng(9).standard_normal(m).astype(dtype)
    em = Emulated(sp, ctx, full, m, n, rs, cs, x, dtype, shift=world % 2)
    y, parts = em.run()
    want, scale = oracle_transpose(full, m, n, x)
    assert np.all(np.abs(y.astype(np.float64) - want) <= RTOL[dtype] * scale + 1e-300), shape
    y2, parts2 = em.run()
    assert y2.tobytes() == y.tobytes() and all(a.tobytes() == b.tobytes() for a, b in zip(parts, parts2))
    if em.one_lane():
        my, mparts = em.model(x)
        assert all(a.tobytes() == b.tobytes() for a, b in zip(parts, mparts))
        assert y.tobytes() == my.tobytes()
        if world == 1:
            assert y.tobytes() == want.tobytes()
    if shape == "band9":
        assert em.one_lane()                                     # the band runs one lane everywhere


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("shape", ["band9", "random16", "power_law"])
def test_transpose_window_alone(shape, dtype):
    """spl_spmv_transpose_window = rows [col_min, col_max] of spl_spmv on the CSC view of the same arrays
    (within tolerance; bit for bit when both run one lane per row)."""
    import spalinalg_b200 as sp
    ctx = sp.default_context()
    full, m, n, _, _ = make_case(shape, 1, dtype)
    rs = [0, 7000, 16000, m]
    x = np.random.default_rng(10).standard_normal(m).astype(dtype)
    for g in range(3):
        p, i, v = shard(full, rs, g)
        nloc = rs[g + 1] - rs[g]
        A = sp.CsrMatrix.new(nloc, n, p, i, v, ctx=ctx)
        At = sp.CscMatrix.new(n, nloc, p, i, v, ctx=ctx)         # the CSC view: A_g^T
        lo, hi = window_of(full, rs, g)
        xg = torch.from_numpy(x[rs[g]:rs[g + 1]].copy()).cuda()
        yw = torch.full((hi - lo,), 7.0, dtype=_tdt(dtype), device="cuda")
        yf = torch.zeros(n, dtype=_tdt(dtype), device="cuda")
        ctx.check(transpose_window(ctx, A, xg.data_ptr(), yw.data_ptr()))
        At.spmv_device(xg.data_ptr(), yf.data_ptr())
        ctx.sync()
        torch.cuda.synchronize()
        got, full_y = yw.cpu().numpy(), yf.cpu().numpy()
        _, scale = oracle_transpose((p, i, v), nloc, n, x[rs[g]:rs[g + 1]])
        assert np.all(np.abs(got.astype(np.float64) - full_y[lo:hi]) <= 2 * RTOL[dtype] * scale[lo:hi] + 1e-300)
        _, csc_lanes = At.spmv_choice()
        if one_lane(sp, full, rs, g, n, ctx) and csc_lanes == 1 and At.spmv_choice()[0] != 3:
            assert got.tobytes() == full_y[lo:hi].tobytes()
        assert not np.any(full_y[:lo]) and not np.any(full_y[hi:])       # nothing outside the footprint


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_spmv_transpose_special_values(dtype):
    """Two ranks, rows [0, 32) and [32, 64), y cut at the odd column 33.
      column 5: its only entry gives -0.0 (a negative value times x = +0.0);
      columns 10 and 63: no rank stores them (10 lies inside rank 0's window, 63 outside every window): +0.0 over
      a y prefilled with 7.0;
      x[31] = +inf, and row 31's columns 30 and 34 are also in rank 1's window (rows 32, 33 store columns 30, 34);
      a NaN value at (40, 41);
      windows start at the odd columns 1 and 29, partial buffers and y slices one element off 16-byte alignment."""
    import spalinalg_b200 as sp
    ctx = sp.default_context()
    rows, cols, vals = [], [], []
    def put(r, c, v):
        rows.append(r); cols.append(c); vals.append(v)
    put(3, 5, -1.5)
    for r in range(0, 32):
        for c in (r + 1, r + 3):
            if c != 5 and c != 10 and c < 36:
                put(r, c, 0.5 + 0.01 * r)
    put(31, 30, 2.0); put(31, 34, -3.0)
    put(32, 30, 1.25); put(33, 34, 0.75)
    for r in range(34, 64):
        for c in (r - 5, r - 3):
            if c != 10:
                put(r, c, -0.25 - 0.01 * r)
    put(40, 41, np.nan)
    r, c, v = np.array(rows), np.array(cols), np.array(vals, dtype)
    full = _compress(64, 64, r, c, v)
    x = (1.0 + 0.125 * np.arange(64)).astype(dtype)
    x[3] = 0.0
    x[31] = np.inf
    rs, cs = [0, 32, 64], [0, 33, 64]
    em = Emulated(sp, ctx, full, 64, 64, rs, cs, x, dtype, shift=1)
    assert em.windows[0] == 1 and em.windows[2] == 29
    assert em.one_lane()
    y, parts = em.run()
    my, mparts = em.model(x)
    assert all(same_bits(a, b) for a, b in zip(parts, mparts))
    assert same_bits(y, my)
    assert y[5] == 0 and not np.signbit(y[5])                   # the row kernels' sum of one -0.0 is +0.0
    assert y[10].tobytes() == np.zeros(1, dtype).tobytes() and y[63].tobytes() == np.zeros(1, dtype).tobytes()
    assert np.isinf(y[30]) and np.isinf(y[34]) and np.isnan(y[41])
    want, scale = oracle_transpose(full, 64, 64, x)
    fin = np.isfinite(want)
    assert np.array_equal(np.isnan(y), np.isnan(want)) and np.array_equal(y[np.isinf(want)], want[np.isinf(want)])
    assert np.all(np.abs(y[fin].astype(np.float64) - want[fin]) <= RTOL[dtype] * scale[fin])
    # the fold itself: a lone -0.0 partial is copied, -0.0 + -0.0 stays -0.0, -0.0 + +0.0 is +0.0
    tdt = _tdt(dtype)
    p0 = torch.tensor([-0.0, -0.0, -0.0, 1.0], dtype=tdt, device="cuda")
    p1 = torch.tensor([-0.0, 0.0, 2.0], dtype=tdt, device="cuda")
    yy = torch.full((5,), 7.0, dtype=tdt, device="cuda")
    ctx.check(reduce_windows(ctx, dtype, 2, 0, [0, 5, 5], [0, 4, 1, 4], [p0.data_ptr(), p1.data_ptr()],
                             yy.data_ptr()))
    ctx.sync()
    got = yy.cpu().numpy()
    assert got.tobytes() == np.array([-0.0, -0.0, 0.0, 3.0, 0.0], dtype).tobytes()


@pytest.mark.gpu
def test_spmv_transpose_follows_new_values():
    """The cached windowed transpose is dropped when the values change: the next product uses the new values."""
    import spalinalg_b200 as sp
    ctx = sp.default_context()
    n = 5003
    full = band9(n, np.float64, 11)
    rs = [0, 2500, n]
    x = np.random.default_rng(12).standard_normal(n)
    em = Emulated(sp, ctx, full, n, n, rs, rs, x, np.float64)
    y_old, _ = em.run()
    new_val = full[2] * 3.0 - 1.0
    for g in range(2):
        a, b = int(full[0][rs[g]]), int(full[0][rs[g + 1]])
        em.mats[g].set_values(new_val[a:b])
    em.full = (full[0], full[1], new_val)
    y_new, _ = em.run()
    want, scale = oracle_transpose(em.full, n, n, x)
    assert em.one_lane()
    assert y_new.tobytes() == em.model(x)[0].tobytes()
    assert np.all(np.abs(y_new - want) <= 1e-12 * scale)
    assert not np.array_equal(y_new, y_old)


@pytest.mark.gpu
def test_spmv_transpose_refusals(monkeypatch):
    """Every refusal: its status, and y and the partial buffers left as they were."""
    import spalinalg_b200 as sp
    from spalinalg_b200 import _capi as E
    ctx = sp.default_context()
    n = 3000
    full = band9(n, np.float64, 13)
    rs = [0, 1000, n]
    x = np.random.default_rng(14).standard_normal(n)
    em = Emulated(sp, ctx, full, n, n, rs, rs, x, np.float64)
    em.run()
    snap = lambda: [t.cpu().numpy().tobytes() for t in em.parts + em.ys]
    before = snap()
    A = em.mats[0]
    xp, yp = em.x[0].data_ptr(), em.part_ptr(0)
    p, i, v = shard(full, rs, 0)
    csc = sp.CscMatrix.new(n, 1000, p, i, v, ctx=ctx)
    assert transpose_window(ctx, csc, xp, yp) == E.SPL_ERR_UNSUPPORTED
    assert transpose_window(ctx, None, xp, yp) == E.SPL_ERR_ARG
    assert transpose_window(ctx, A, 0, yp) == E.SPL_ERR_ARG
    assert transpose_window(ctx, A, xp, 0) == E.SPL_ERR_ARG
    monkeypatch.setenv("SPL_WIDE_MIN_NNZ", "10")
    wide = sp.CsrMatrix.new(1000, n, p, i, v, ctx=ctx)
    assert wide.device_ptr64()
    assert transpose_window(ctx, wide, xp, yp) == E.SPL_ERR_UNSUPPORTED
    monkeypatch.delenv("SPL_WIDE_MIN_NNZ")
    parts = [em.part_ptr(0), em.part_ptr(1)]
    y0 = em.ys[0].data_ptr()
    ok = dict(world=2, rank=0, cs=rs, win=em.windows, parts=parts)
    cases = [
        dict(world=0, cs=[0], win=[]),
        dict(world=9, cs=[0] * 9 + [n], win=[0, 0] * 9, parts=[None] * 9),
        dict(rank=-1),
        dict(rank=2),
        dict(cs=[1, 1000, n]),                                  # not from 0
        dict(cs=[0, 2000, 1000], world=2),                      # decreasing
        dict(win=[5, 4] + em.windows[2:]),                      # a window that ends before it starts
        dict(win=em.windows[:3] + [n + 1]),                     # past col_starts[world]
        dict(parts=[parts[0], None]),                           # NULL partial of a non-empty window
    ]
    for kw in cases:
        a = dict(ok, **kw)
        st = reduce_windows(ctx, np.float64, a["world"], a["rank"], a["cs"], a["win"], a["parts"], y0)
        assert st == E.SPL_ERR_ARG, (kw, st)
    fl = torch.zeros(8, dtype=torch.int32, device="cuda")
    st = reduce_windows(ctx, np.float64, 2, 0, rs, em.windows, parts, y0, flags=[fl.data_ptr(), None], epoch=1)
    assert st == E.SPL_ERR_ARG                                  # a NULL flag block
    for args in ((None, em.windows, parts), (rs, None, parts), (rs, em.windows, None)):
        cs = (C.c_uint64 * 3)(*rs) if args[0] else None
        win = (C.c_uint64 * 4)(*em.windows) if args[1] else None
        pp = (C.c_void_p * 2)(*parts) if args[2] else None
        st = ctx._lib.spl_peer_reduce_windows(ctx._h, _code(np.float64), 2, 0, C.cast(cs, C.c_void_p) if cs else None,
                                              C.cast(win, C.c_void_p) if win else None,
                                              C.cast(pp, C.c_void_p) if pp else None, None, 0, 2000, C.c_void_p(y0))
        assert st == E.SPL_ERR_ARG
    assert reduce_windows(ctx, np.float64, 2, 0, rs, em.windows, parts, 0) == E.SPL_ERR_ARG     # NULL y
    ctx.sync()
    torch.cuda.synchronize()
    assert snap() == before


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.gpu
def test_dist_spmv_transpose_world1_nccl():
    """DistCsrMatrix.prepare_transpose / spmv_transpose / check with a one-rank NCCL group: the same host code as
    the multi-GPU runs (footprint all-gather, two partial buffers, flag block, both launches), bit for bit against
    the oracle on the band (one lane); three products, so both partial buffers are used and reused."""
    import torch.distributed as dist
    import spalinalg_b200 as sp
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{_free_port()}", rank=0, world_size=1,
                            device_id=torch.device("cuda", 0))
    try:
        ctx = sp.default_context()
        for dtype in (np.float64, np.float32):
            m, n = 20011, 30011
            full = scaled_band(m, n, dtype, 15)
            D = spd.DistCsrMatrix(sp.CsrMatrix.new(m, n, *full, ctx=ctx), [0, m], 0, m, n)
            D.prepare_transpose(dist, torch)
            assert D._transpose["col_starts"] == [0, n]
            for t in range(3):
                x = np.random.default_rng(16 + t).standard_normal(m).astype(dtype)
                xd = torch.from_numpy(x).cuda()
                yd = torch.full((n,), 7.0, dtype=_tdt(dtype), device="cuda")
                D.spmv_transpose(xd.data_ptr(), yd.data_ptr())
                D.check()
                want, _ = oracle_transpose(full, m, n, x)
                assert yd.cpu().numpy().tobytes() == want.tobytes()
            with pytest.raises(ValueError):
                D.prepare_transpose(dist, torch, col_starts=[0, n - 1])
            D.close_transpose(dist)
    finally:
        dist.destroy_process_group()
