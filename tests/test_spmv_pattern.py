"""The row-pattern path of the stream SpMV: tiles whose rows all follow the matrix's row pattern (the column
offsets of one reference row) stream their values only.  Every case compares, with torch.equal, the stream
kernel with the path on, the stream kernel with SPL_STREAM_PATTERN=0 and the vector kernel, and all of them with
the oracle (bit for bit with one lane per row).  Then the first column index of every full-length row is overwritten
with its second column: the CSR path sees that on every such row, the pattern path only on rows of irregular tiles,
which shows that the regular path ran and does not read the index stream."""
import contextlib
import ctypes as C
import os

import numpy as np
import pytest

import oracle as orc
import spalinalg_b200 as sp
from spalinalg_b200 import _capi as capi
from spalinalg_b200 import synthetic as syn
from spalinalg_b200.synthetic_device import device_view

pytestmark = pytest.mark.gpu

SPMV_RTOL = {np.dtype(np.float64): 1e-12, np.dtype(np.float32): 1e-5}


@contextlib.contextmanager
def env(**kv):
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update({k: str(v) for k, v in kv.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def band_rows(r0, r1, n, offsets):
    """(local row, column) of the band rows [r0, r1) of an n x n matrix with the given diagonals, row-major."""
    rows = np.repeat(np.arange(r0, r1, dtype=np.int64), len(offsets))
    cols = rows + np.tile(np.asarray(offsets, np.int64), r1 - r0)
    ok = (cols >= 0) & (cols < n)
    return rows[ok] - r0, cols[ok]


def csr(nrows, rows, cols, rng, dtype):
    ptr = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=nrows))]).astype(np.uint64)
    return ptr, cols.astype(np.uint64), (rng.standard_normal(len(cols)) * 0.5).astype(dtype)


def matrix(shape, dtype, rng):
    if shape.startswith("band") and shape[4:].isdigit():       # band3, band9, band16, band33, band64, band65
        w = int(shape[4:])
        n = 300_001 if w <= 16 else 100_003                    # not a multiple of a tile
        rows, cols = band_rows(0, n, n, range(-(w // 2), w - w // 2))
        return n, csr(n, rows, cols, rng, dtype)
    if shape == "band9_irregular":                             # irregular rows amid regular tiles
        n = 300_001
        rows, cols = band_rows(0, n, n, range(-4, 5))
        keep = np.ones(len(rows), bool)
        m = n // 2 + 777
        keep[(rows == m) & (cols == m + 2)] = False            # a row missing a diagonal
        keep[rows == m + 3000] = False                         # a row of no entries
        cols = cols.copy()
        cols[(rows == m + 6000) & (cols == m + 6004)] = n - 1  # a full-length row with a far column
        rows, cols = rows[keep], cols[keep]
        # one row with an extra far entry (the longest row, before the middle: no row pattern at all)
        x = n // 3
        at = np.searchsorted(rows, x, side="right")
        rows, cols = np.insert(rows, at, x), np.insert(cols, at, n - 2)
        return n, csr(n, rows, cols, rng, dtype)
    if shape == "band9_holes":                                 # the same without the extra entry: a row pattern
        n = 300_001
        rows, cols = band_rows(0, n, n, range(-4, 5))
        keep = np.ones(len(rows), bool)
        m = n // 2 + 777
        keep[(rows == m) & (cols == m + 2)] = False
        keep[rows == m + 3000] = False
        cols = cols.copy()
        cols[(rows == m + 6000) & (cols == m + 6004)] = n - 1
        return n, csr(n, rows[keep], cols[keep], rng, dtype)
    if shape == "laplace":                                     # boundary rows in many tiles
        g = 301
        r, c, v = syn.laplacian_2d(g)
        n = g * g
        order = np.lexsort((c, r))
        return n, (syn.csr_from_sorted_triplets(n, r, c, v)[0], c[order].astype(np.uint64),
                   (rng.standard_normal(len(c)) * 0.5).astype(dtype))
    n = 200_003                                                # random: no regular tile
    lens = rng.integers(0, 21, n)
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    ind = np.concatenate([np.sort(rng.choice(n, l, replace=False)) for l in lens if l]).astype(np.uint64)
    return n, (ptr, ind, (rng.standard_normal(len(ind)) * 0.5).astype(dtype))


def three_products(run, y):
    """y of the stream kernel with the pattern path on, off, and of the vector kernel."""
    import torch
    out = []
    for kernel, pattern in ((capi.SPL_SPMV_STREAM, 1), (capi.SPL_SPMV_STREAM, 0), (capi.SPL_SPMV_VECTOR, 1)):
        y.fill_(7.0)
        torch.cuda.synchronize()
        with env(SPL_STREAM_PATTERN=pattern):
            run(kernel)
        sp.default_context().sync()
        out.append(y.clone())
    return out


def check_oracle(got, n, a, x, lanes, dtype):
    want = orc.csr_spmv(n, *a, x)
    scale = orc.csr_spmv(n, a[0], a[1], np.abs(a[2]), np.abs(x))
    assert np.all(np.abs(got - want) <= SPMV_RTOL[np.dtype(dtype)] * np.maximum(scale, np.finfo(dtype).tiny))
    if lanes == 1:
        assert got.tobytes() == want.tobytes()


def index_probe(A, a, run_stream, y):
    """Overwrites the first column index of every row of the longest length with its second column and returns
    (rows whose y changes with the pattern path on, rows whose y changes with it off, rows overwritten)."""
    import torch

    def product(pattern):
        y.fill_(7.0)
        torch.cuda.synchronize()
        with env(SPL_STREAM_PATTERN=pattern):
            run_stream()
        sp.default_context().sync()
        return y.clone()
    y0 = product(1)
    ptr, cols = a[0].astype(np.int64), a[1].astype(np.int64)
    lens = np.diff(ptr)
    rows = np.nonzero(lens == lens.max())[0]
    _, ind_dev, _ = A.device_ptrs()
    ind = device_view(torch, ind_dev, A.nnz(), torch.int32)
    ind[torch.from_numpy(ptr[rows]).cuda()] = torch.from_numpy(cols[ptr[rows] + 1].astype(np.int32)).cuda()
    torch.cuda.synchronize()
    on, off = product(1), product(0)
    changed = [set((y_ != y0).nonzero().flatten().cpu().tolist()) for y_ in (on, off)]
    assert changed[1] <= set(rows.tolist()) and len(changed[1]) >= 0.99 * len(rows), "the CSR path reads every index"
    assert changed[0] <= changed[1]
    return changed[0], changed[1], rows


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("shape", ["band3", "band9", "band9_irregular", "band9_holes", "band16", "band33", "band64",
                                   "band65", "laplace", "random"])
def test_stream_pattern_same_bits(dtype, shape):
    """band3 (1 lane per row) and band16 (4 lanes) take U = 4 entries per lane and trip, the others U = 8; band64
    is the longest row pattern, band65 and the band with one extra long row have none."""
    import torch
    rng = np.random.default_rng(5)
    n, a = matrix(shape, dtype, rng)
    A = sp.CsrMatrix.new(n, n, *a)
    lanes = A.spmv_choice()[1]
    x = rng.standard_normal(n).astype(dtype)
    xd = torch.from_numpy(x).cuda()
    yd = torch.empty_like(xd)
    run = lambda k: A.spmv_device(xd.data_ptr(), yd.data_ptr(), kernel=k)
    yp, yc, yv = three_products(run, yd)
    assert torch.equal(yp, yc) and torch.equal(yp, yv)
    check_oracle(yp.cpu().numpy(), n, a, x, lanes, dtype)
    on, off, rows = index_probe(A, a, lambda: run(capi.SPL_SPMV_STREAM), yd)
    if shape in ("band9_irregular", "band65", "random"):          # no row pattern (or no regular tile)
        assert on == off
    elif shape in ("band9_holes", "laplace"):                     # regular and irregular tiles
        assert 0 < len(off - on) and len(on) > 0
    else:                                                         # a band: only its first and last tile are irregular
        assert len(on) <= 2 * (256 // lanes), f"{len(on)} of {len(rows)} rows read their indices"


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_stream_pattern_window_shard(dtype):
    """A row shard of a band with local rows and global columns (row pattern shifted by its first row), run
    through spl_spmv_window on its own slice of x plus the halo: every row has the pattern."""
    import torch
    rng = np.random.default_rng(6)
    n, r0, r1 = 1_000_003, 300_001, 700_003
    rows, cols = band_rows(r0, r1, n, range(-4, 5))
    nloc = r1 - r0
    a = csr(nloc, rows, cols, rng, dtype)
    A = sp.CsrMatrix.new(nloc, n, *a)
    x = rng.standard_normal(n).astype(dtype)
    w0, w1 = r0 - 4, r1 + 4
    xw = torch.from_numpy(x[w0:w1].copy()).cuda()
    yd = torch.empty(nloc, dtype=xw.dtype, device="cuda")
    ctx = sp.default_context()

    def run(kernel):
        with env(SPL_SPMV_KERNEL="stream" if kernel == capi.SPL_SPMV_STREAM else "vector"):
            ctx.check(ctx._lib.spl_spmv_window(ctx._h, A._h, C.c_void_p(xw.data_ptr()), w0, w1 - w0,
                                               C.c_void_p(yd.data_ptr())))
    yp, yc, yv = three_products(run, yd)
    assert torch.equal(yp, yc) and torch.equal(yp, yv)
    check_oracle(yp.cpu().numpy(), nloc, a, x, A.spmv_choice()[1], dtype)
    on, off, _ = index_probe(A, a, lambda: run(capi.SPL_SPMV_STREAM), yd)
    assert not on
