"""The band kernel of the stream SpMV: a matrix whose rows, all but a few, follow its row pattern, with values and the
x window of each regular tile staged in shared memory.  Every case compares, with torch.equal (bit patterns where x
holds NaN), the band route, the route off (SPL_STREAM_BAND=0: the stream kernel's row-pattern path) and the vector
kernel, and all of them with the oracle (bit for bit with one lane per row).  torch.profiler shows which kernel ran;
an index probe (the first column index of every full-length row overwritten with its second) shows that the band
route reads no index of a regular tile."""
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


def band_csr(nrows, ncols, offsets, rng, dtype, r0=0, drop=()):
    """Rows [r0, r0 + nrows) of a matrix with the given diagonals (global columns, local rows), without the
    entries (local row, column) in `drop`."""
    rows = np.repeat(np.arange(nrows, dtype=np.int64), len(offsets))
    cols = rows + r0 + np.tile(np.asarray(sorted(offsets), np.int64), nrows)
    ok = (cols >= 0) & (cols < ncols)
    for r, c in drop:
        ok &= ~((rows == r) & (cols == c))
    rows, cols = rows[ok], cols[ok]
    ptr = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=nrows))]).astype(np.uint64)
    return ptr, cols.astype(np.uint64), (rng.standard_normal(len(cols)) * 0.5).astype(dtype)


def kernels_run(fn):
    """Names of the CUDA kernels fn launches."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return " ".join(e.name for e in prof.events())


def same(p, q):
    """bit for bit, NaN included"""
    import torch
    bits = {torch.float64: torch.int64, torch.float32: torch.int32}[p.dtype]
    return p.dtype == q.dtype and torch.equal(p.view(bits), q.view(bits))


def three_products(run, y):
    """y of the band route, of the route off and of the vector kernel, and the kernel names of the first two."""
    import torch
    out, names = [], []
    for kernel, band in ((capi.SPL_SPMV_STREAM, 1), (capi.SPL_SPMV_STREAM, 0), (capi.SPL_SPMV_VECTOR, 1)):
        y.fill_(7.0)
        torch.cuda.synchronize()
        with env(SPL_STREAM_BAND=band):
            names.append(kernels_run(lambda: run(kernel)))
        sp.default_context().sync()
        out.append(y.clone())
    return out, names


def check_oracle(got, n, a, x, lanes, dtype):
    want = orc.csr_spmv(n, *a, x)
    nan = np.isnan(want)
    assert np.array_equal(nan, np.isnan(got))
    g, w = got[~nan], want[~nan]
    scale = orc.csr_spmv(n, a[0], a[1], np.abs(a[2]), np.abs(x))[~nan]
    with np.errstate(invalid="ignore"):
        ok = (g == w) | (np.abs(g - w) <= SPMV_RTOL[np.dtype(dtype)] * np.maximum(scale, np.finfo(dtype).tiny))
    assert np.all(ok)
    if lanes == 1:
        assert got[~nan].tobytes() == want[~nan].tobytes()


def check_routes(run, y, n, a, x, lanes, dtype, band=True):
    (yb, yo, yv), (kb, ko, _) = three_products(run, y)
    assert same(yb, yo) and same(yb, yv)
    assert ("spmv_band_kernel" in kb) == band and "spmv_band_kernel" not in ko
    assert "spmv_stream_kernel" in ko
    check_oracle(yb.cpu().numpy(), n, a, x, lanes, dtype)


def index_probe(A, a, run_stream, y):
    """Overwrites the first column index of every row of the longest length with its second column; returns the rows
    whose y changes with the band route on, and those overwritten."""
    import torch

    def product(band):
        y.fill_(7.0)
        torch.cuda.synchronize()
        with env(SPL_STREAM_BAND=band):
            run_stream()
        sp.default_context().sync()
        return y.clone()
    y0 = product(1)
    ptr, cols = a[0].astype(np.int64), a[1].astype(np.int64)
    lens = np.diff(ptr)
    rows = np.nonzero(lens == lens.max())[0]
    _, ind_dev, _ = A.device_ptrs()
    ind = device_view(torch, ind_dev, A.nnz(), torch.int32)
    saved = ind.clone()
    ind[torch.from_numpy(ptr[rows]).cuda()] = torch.from_numpy(cols[ptr[rows] + 1].astype(np.int32)).cuda()
    torch.cuda.synchronize()
    on = product(1)
    ind.copy_(saved)
    torch.cuda.synchronize()
    return set((on != y0).nonzero().flatten().cpu().tolist()), rows


def device_run(A, x, y):
    return lambda k: A.spmv_device(x.data_ptr(), y.data_ptr(), kernel=k)


BANDS = {"k1": [0], "k3": [-1, 0, 1], "k9": list(range(-4, 5)), "k17": list(range(-8, 9)), "k33": list(range(-16, 17)),
         "k64": list(range(-32, 32)), "upper0_8": list(range(0, 9)), "lower8_0": list(range(-8, 1))}


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("band", list(BANDS) + ["rect_shift"])
def test_band_same_bits(dtype, band):
    """n is a multiple neither of 4 nor of a tile; k64 is the longest row pattern.  rect_shift: 300 001 x 300 041,
    columns r + 20 .. r + 28 (no row off the pattern)."""
    import torch
    rng = np.random.default_rng(7)
    n = 300_001
    if band == "rect_shift":
        ncols, offs = n + 40, list(range(20, 29))
    else:
        ncols, offs = n, BANDS[band]
    a = band_csr(n, ncols, offs, rng, dtype)
    A = sp.CsrMatrix.new(n, ncols, *a)
    lanes = A.spmv_choice()[1]
    x = rng.standard_normal(ncols).astype(dtype)
    xd = torch.from_numpy(x).cuda()
    yd = torch.empty(n, dtype=xd.dtype, device="cuda")
    check_routes(device_run(A, xd, yd), yd, n, a, x, lanes, dtype)
    if len(offs) < 2:                                    # the probe needs a second column to write into the first
        return
    on, rows = index_probe(A, a, lambda: A.spmv_device(xd.data_ptr(), yd.data_ptr(), kernel=capi.SPL_SPMV_STREAM), yd)
    # only the rows of the irregular tiles (the first and last tile) read their indices
    assert len(on) <= 2 * (256 // lanes) and on <= set(rows.tolist())


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_band_broken_rows(dtype):
    """Rows off the pattern (a dropped entry) in the middle of a CTA's range and on both sides of a CTA boundary:
    their tiles take the global path, the tiles around them the staged one."""
    import torch
    rng = np.random.default_rng(8)
    n, offs = 1_000_003, list(range(-4, 5))
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    grid = sms * 2                                       # SPL_STREAM_CTAS=2 below
    a0 = band_csr(n, n, offs, rng, dtype)

    def first_row(ptr, b):                               # stream_partition_kernel's CTA start
        target = (int(ptr[-1]) + n) * b // grid
        return int(np.searchsorted(ptr[:-1].astype(np.int64) + np.arange(n), target, side="left")) & ~3
    mid = (first_row(a0[0], 10) + first_row(a0[0], 11)) // 2 + 1
    q = first_row(a0[0], grid // 2)
    for _ in range(8):                                   # the dropped entries may move the boundary: follow it
        a = band_csr(n, n, offs, rng, dtype, drop=[(mid, mid + 2), (q - 1, q + 3), (q, q - 1)])
        if first_row(a[0], grid // 2) == q:
            break
        q = first_row(a[0], grid // 2)
    assert first_row(a[0], grid // 2) == q               # rows q - 1 and q sit on either side of a CTA boundary
    A = sp.CsrMatrix.new(n, n, *a)
    x = rng.standard_normal(n).astype(dtype)
    xd = torch.from_numpy(x).cuda()
    yd = torch.empty_like(xd)
    with env(SPL_STREAM_CTAS=2):
        check_routes(device_run(A, xd, yd), yd, n, a, x, A.spmv_choice()[1], dtype)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_band_inf_nan(dtype):
    """x holds inf and NaN in columns rows touch and in columns no row touches."""
    import torch
    rng = np.random.default_rng(9)
    n, ncols = 300_001, 300_001 + 30                     # columns n + 9 .. n + 29: no row touches them
    a = band_csr(n, ncols, list(range(0, 9)), rng, dtype)
    A = sp.CsrMatrix.new(n, ncols, *a)
    x = rng.standard_normal(ncols).astype(dtype)
    x[[2, 150_000, n + 4, n + 15]] = np.inf
    x[[5, 150_100, n + 16, n + 29]] = np.nan
    xd = torch.from_numpy(x).cuda()
    yd = torch.empty(n, dtype=xd.dtype, device="cuda")
    check_routes(device_run(A, xd, yd), yd, n, a, x, A.spmv_choice()[1], dtype)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("shift", [1, 3])
def test_band_window_shard(dtype, shift):
    """A row shard at global rows [4e9, 4e9 + 300 001) through spl_spmv_window: large column offsets, a window
    buffer that starts `shift` elements past a 16-byte boundary and ends exactly at the footprint, inside a tensor
    whose other elements are NaN."""
    import torch
    rng = np.random.default_rng(10)
    r0, nloc, ncols = 4_000_000_000, 300_001, 4_294_000_000
    offs = list(range(-4, 5))
    a = band_csr(nloc, ncols, offs, rng, dtype, r0=r0)
    A = sp.CsrMatrix.new(nloc, ncols, *a)
    w0, w1 = r0 - 4, r0 + nloc + 4                       # the footprint
    xw = rng.standard_normal(w1 - w0).astype(dtype)
    big = torch.full((w1 - w0 + 2 * shift + 8,), float("nan"), dtype=getattr(torch, np.dtype(dtype).name), device="cuda")
    view = big[shift:shift + (w1 - w0)]
    view.copy_(torch.from_numpy(xw))
    assert view.data_ptr() % 16 != 0
    yd = torch.empty(nloc, dtype=view.dtype, device="cuda")
    ctx = sp.default_context()

    def run(kernel):
        with env(SPL_SPMV_KERNEL="stream" if kernel == capi.SPL_SPMV_STREAM else "vector"):
            ctx.check(ctx._lib.spl_spmv_window(ctx._h, A._h, C.c_void_p(view.data_ptr()), w0, w1 - w0,
                                               C.c_void_p(yd.data_ptr())))
    rebased = (a[0], a[1] - np.uint64(w0), a[2])         # the same rows on the window's columns, for the oracle
    check_routes(run, yd, nloc, rebased, xw, A.spmv_choice()[1], dtype)
    assert not torch.isnan(yd).any()


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_band_iteration_back_to_back(dtype):
    """x_{t+1} = A x_t for 30 products launched back to back (programmatic dependent launch between them), bit for
    bit against the same iteration on the vector kernel: an x copy issued before griddepcontrol.wait would read the
    previous product's output before it is final."""
    import torch
    rng = np.random.default_rng(11)
    n = 2_000_003
    a = band_csr(n, n, list(range(-4, 5)), rng, dtype)
    a = (a[0], a[1], (a[2] * 0.6).astype(dtype))
    A = sp.CsrMatrix.new(n, n, *a)
    x0 = torch.from_numpy(rng.standard_normal(n).astype(dtype)).cuda()

    def iterate(kernel):
        v = [x0.clone(), torch.empty_like(x0)]
        torch.cuda.synchronize()
        for t in range(30):
            A.spmv_device(v[t % 2].data_ptr(), v[(t + 1) % 2].data_ptr(), kernel=kernel)
        sp.default_context().sync()
        return v[0]
    names = kernels_run(lambda: iterate(capi.SPL_SPMV_STREAM))
    assert "spmv_band_kernel" in names
    yb, yv = iterate(capi.SPL_SPMV_STREAM), iterate(capi.SPL_SPMV_VECTOR)
    assert torch.isfinite(yb).all() and torch.equal(yb, yv)


@pytest.mark.parametrize("shape", ["laplace", "stencil27", "random"])
def test_band_not_taken(shape):
    """Boundary rows in many tiles (2-D Laplacian, 27-point stencil) or no row pattern (random): the stream kernel,
    with the row-pattern path where it had one."""
    import torch
    dtype = np.float64
    rng = np.random.default_rng(12)
    if shape == "laplace":
        g = 301
        r, c, v = syn.laplacian_2d(g)
        n = g * g
    elif shape == "stencil27":
        g, n = 50, 50 ** 3
        idx = np.arange(n)
        i, j, k = idx // (g * g), (idx // g) % g, idx % g
        rs, cs = [], []
        for di in (-1, 0, 1):
            for dj in (-1, 0, 1):
                for dk in (-1, 0, 1):
                    ok = (i + di >= 0) & (i + di < g) & (j + dj >= 0) & (j + dj < g) & (k + dk >= 0) & (k + dk < g)
                    rs.append(idx[ok])
                    cs.append(idx[ok] + di * g * g + dj * g + dk)
        r, c = np.concatenate(rs), np.concatenate(cs)
    else:
        n = 200_003
        lens = rng.integers(0, 21, n)
        r = np.repeat(np.arange(n), lens)
        c = np.concatenate([np.sort(rng.choice(n, l, replace=False)) for l in lens if l])
    order = np.lexsort((c, r))
    r, c = r[order], c[order]
    a = (np.concatenate([[0], np.cumsum(np.bincount(r, minlength=n))]).astype(np.uint64), c.astype(np.uint64),
         (rng.standard_normal(len(c)) * 0.5).astype(dtype))
    A = sp.CsrMatrix.new(n, n, *a)
    x = rng.standard_normal(n).astype(dtype)
    xd = torch.from_numpy(x).cuda()
    yd = torch.empty_like(xd)
    check_routes(device_run(A, xd, yd), yd, n, a, x, A.spmv_choice()[1], dtype, band=False)
