"""COO -> CSR / CSC assembly in buckets of whole majors, the route of lists with 2^32 - 65536 triplets or
more (wide_assemble.cu).  At oracle sizes SPL_ASSEMBLE_BUCKET_MAX sends short lists down the same route;
the result must equal the oracle's restatement of src/csr/conv/coo.rs:3-116 bit for bit and the direct
32-bit route's output.  At full size: a scrambled band of 4.36 G cells with order-sensitive duplicates on
both sides of position 2^32, checked against its analytic assembly."""
import ctypes as C

import numpy as np
import pytest

import oracle as orc
import spalinalg_b200 as sp
from spalinalg_b200 import _capi as capi
from spalinalg_b200 import synthetic as syn

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

KNOB = "SPL_ASSEMBLE_BUCKET_MAX"
CLS = {"row": sp.CsrMatrix, "col": sp.CscMatrix}


def sd():
    from spalinalg_b200 import synthetic_device
    return synthetic_device


def arrays(m):
    if isinstance(m, sp.CsrMatrix):
        return m.rowptr(), m.colind(), m.values()
    return m.colptr(), m.rowind(), m.values()


def same(got, want, what=""):
    gp, gi, gv = got
    wp, wi, wv = want
    assert gp.dtype == np.uint64 and gi.dtype == np.uint64
    assert np.array_equal(gp, np.asarray(wp, np.uint64)), f"{what}: ptr differs"
    assert np.array_equal(gi, np.asarray(wi, np.uint64)), f"{what}: ind differs"
    wv = np.asarray(wv, gv.dtype)
    assert gv.tobytes() == wv.tobytes(), f"{what}: values differ (bitwise)"


def dev_arrays(A):
    p, i, v = A.device_ptrs()
    nmajor = A.nrows() if isinstance(A, sp.CsrMatrix) else A.ncols()
    tdt = torch.float32 if A.dtype == np.float32 else torch.float64
    view = sd().device_view
    return (view(torch, p, nmajor + 1, torch.int32), view(torch, i, max(A.nnz(), 1), torch.int32)[:A.nnz()],
            view(torch, v, max(A.nnz(), 1), tdt)[:A.nnz()])


def same_device(A, B):
    """torch.equal on the device arrays (values compared as bit patterns)."""
    torch.cuda.synchronize()
    assert A.nnz() == B.nnz() and A.device_ptr64() is None and B.device_ptr64() is None
    (ap, ai, av), (bp, bi, bv) = dev_arrays(A), dev_arrays(B)
    it = torch.int32 if av.dtype == torch.float32 else torch.int64
    assert torch.equal(ap, bp) and torch.equal(ai, bi) and torch.equal(av.view(it), bv.view(it))


def case(seed, nr, nc, major, dtype, dedup, long_len=2000):
    """Random triplets with >= 3-way duplicates spread over the whole list, exact cancellations, -0.0, a
    run of empty majors, one major longer than a bucket and one long major whose every cell cancels (an
    empty part).  With dedup == 0 the keys are unique (DokMatrix semantics, explicit zeros kept)."""
    rng = np.random.default_rng(seed)
    n = 20000
    r, c, v = syn.random_coo(rng, nr, nc, n, dtype, dup_frac=0.3, cancel_frac=0.05)
    mj, mn = (r, c) if major == "row" else (c, r)
    nmaj, nmin = (nr, nc) if major == "row" else (nc, nr)
    keep = ((mj < 100) | (mj >= 400)) & (mj != 7) & (mj != 9)        # majors 100..399 empty
    mj, mn, v = mj[keep], mn[keep], v[keep]
    # one major longer than any bucket below
    lm = np.full(long_len, 7, np.uint64)
    ln = rng.integers(0, nmin, long_len).astype(np.uint64)
    lv = rng.uniform(-1, 1, long_len).astype(dtype)
    # one long major whose cells all cancel: (x, -x) pushed far apart
    half = long_len // 2
    zn = rng.choice(nmin, half, replace=False).astype(np.uint64)
    zv = rng.uniform(-1, 1, half).astype(dtype)
    zm = np.full(long_len, 9, np.uint64)
    # three-way duplicates: first push near the start, the others in the middle and at the end
    t = 300
    tm = rng.integers(400, nmaj, t).astype(np.uint64)
    tn = rng.integers(0, nmin, t).astype(np.uint64)
    tv = (rng.standard_normal((3, t)) * 10.0 ** rng.integers(-6, 6, (3, t))).astype(dtype)
    tv[2, :50] = -(tv[0, :50] + tv[1, :50])                           # some of them cancel (or nearly)
    negz = np.full(40, -0.0, dtype)
    nzm = rng.integers(400, nmaj, 40).astype(np.uint64)
    nzn = rng.integers(0, nmin, 40).astype(np.uint64)
    m = len(v)
    parts_m = [tm, mj[:m // 3], lm, zm[:half], nzm, mj[m // 3:2 * m // 3], tm, zm[half:], mj[2 * m // 3:], tm]
    parts_n = [tn, mn[:m // 3], ln, zn, nzn, mn[m // 3:2 * m // 3], tn, zn, mn[2 * m // 3:], tn]
    parts_v = [tv[0], v[:m // 3], lv, zv, negz, v[m // 3:2 * m // 3], tv[1], -zv, v[2 * m // 3:], tv[2]]
    mj, mn, v = np.concatenate(parts_m), np.concatenate(parts_n), np.concatenate(parts_v).astype(dtype)
    if not dedup:                                                     # DOK: first occurrence of each key
        _, first = np.unique(mj * np.uint64(nmin) + mn, return_index=True)
        first.sort()
        mj, mn, v = mj[first], mn[first], v[first]
    r, c = (mj, mn) if major == "row" else (mn, mj)
    return r, c, v


def from_device(major, nr, nc, r, c, v, dedup, dropzero):
    rd = torch.from_numpy(r.astype(np.int64)).to(torch.int32).cuda()
    cd = torch.from_numpy(c.astype(np.int64)).to(torch.int32).cuda()
    vd = torch.from_numpy(v).cuda()
    torch.cuda.synchronize()
    M = CLS[major].from_device_triplets(nr, nc, len(v), rd.data_ptr(), cd.data_ptr(), vd.data_ptr(), v.dtype,
                                        dedup=dedup, dropzero=dropzero)
    sp.default_context().sync()
    return M


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("major", ["row", "col"])
@pytest.mark.parametrize("flags", [(1, 1), (0, 0)])
@pytest.mark.parametrize("shape", [(3000, 5000), (3000, 1 << 30)])       # keys of 25 bits / of 42 bits
@pytest.mark.parametrize("bucket", [300, 7000])
def test_bucketed_device_triplets_match_oracle_and_direct(monkeypatch, dtype, major, flags, shape, bucket):
    dedup, dropzero = flags
    nr, nc = shape if major == "row" else shape[::-1]
    r, c, v = case(shape[1] % 9973 + 2 * (major == "row") + dedup, nr, nc, major, dtype, dedup)
    assert len(v) > bucket
    monkeypatch.delenv(KNOB, raising=False)
    direct = from_device(major, nr, nc, r, c, v, dedup, dropzero)
    monkeypatch.setenv(KNOB, str(bucket))
    got = from_device(major, nr, nc, r, c, v, dedup, dropzero)
    want = orc.compress_from_coo(nr, nc, orc.make_triplets(r, c, v), major, dedup, dropzero)
    same(arrays(got), want, "bucketed vs oracle")
    same_device(got, direct)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("major", ["row", "col"])
def test_bucketed_host_and_builder_fronts(monkeypatch, dtype, major):
    nr, nc = 4000, 2500
    r, c, v = case(11, nr, nc, major, dtype, 1)
    want = orc.compress_from_coo(nr, nc, orc.make_triplets(r, c, v), major)
    monkeypatch.setenv(KNOB, "500")
    coo = sp.CooMatrix.with_triplets(nr, nc, r, c, v)
    same(arrays(CLS[major].from_coo(coo)), want, "spl_mat_from_coo")
    pinned = sp.PinnedCooMatrix.with_triplets(nr, nc, r, c, v)
    same(arrays(CLS[major].from_coo(pinned)), want, "builder")
    # DokMatrix: unique keys, explicit zeros kept (src/csr/conv/dok.rs:3-76)
    rd, cd, vd = case(12, nr, nc, major, dtype, 0)
    dok = sp.DokMatrix.with_entries(nr, nc, zip(rd.tolist(), cd.tolist(), vd.tolist()), dtype=dtype)
    dr, dc, dv = dok.triplets()
    same(arrays(CLS[major].from_dok(dok)),
         orc.compress_from_coo(nr, nc, orc.make_triplets(dr, dc, dv), major, False, False), "from_dok")


def test_bucketed_out_of_bounds_in_last_bucket(monkeypatch):
    nr, nc = 2000, 2000
    rng = np.random.default_rng(5)
    r = np.sort(rng.integers(0, nr, 5000)).astype(np.int64)
    c = rng.integers(0, nc, 5000).astype(np.int64)
    c[-1] = nc                                                        # last triplet, last row: column out of range
    v = rng.uniform(-1, 1, 5000)
    rd, cd, vd = (torch.from_numpy(x).cuda() for x in (r.astype(np.int32), c.astype(np.int32), v))
    torch.cuda.synchronize()
    monkeypatch.setenv(KNOB, "256")
    ctx = sp.default_context()
    for fmt in (capi.SPL_CSR, capi.SPL_CSC):
        h = C.c_void_p()
        st = ctx._lib.spl_mat_from_coo_dev(ctx._h, fmt, capi.SPL_F64, nr, nc, len(v), C.c_void_p(rd.data_ptr()),
                                           C.c_void_p(cd.data_ptr()), C.c_void_p(vd.data_ptr()), 1, 1, C.byref(h))
        assert st == capi.SPL_ERR_ARG and not h.value
    h = C.c_void_p()
    ru, cu = r.astype(np.uint64), c.astype(np.uint64)
    st = ctx._lib.spl_mat_from_coo(ctx._h, capi.SPL_CSR, capi.SPL_F64, nr, nc, len(v), ru.ctypes.data, cu.ctypes.data,
                                   v.ctypes.data, 1, 1, C.byref(h))
    assert st == capi.SPL_ERR_ARG and not h.value


# ------------------------------------------------------------------ beyond 2^32 triplets
def test_bucketed_beyond_2_pow_32_triplets():
    """f32 band, n = 2^26, 65 diagonals: 4.36 G distinct cells in scrambled order, so the output is wide.
    Some cells are pushed three times, the first push in place (anywhere in the list) and two more at the
    end, beyond position 2^32: (2^24, 1, -2^24) sums to 0 in f32 and the cell is dropped, (2^24, -2^24, 1)
    sums to 1 and it is kept."""
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    sp.default_context().trim()
    free, _ = torch.cuda.mem_get_info()
    if free < 150 * 2 ** 30:
        pytest.skip(f"needs ~150 GB of free device memory, {free / 2 ** 30:.0f} GB available")
    g = sd()
    n, half, k = 1 << 26, 32, 64                              # k cells dropped, k kept
    row, col, val, cells = g.scrambled_band_coo_device(torch, n, half, torch.float32, spare=4 * k)
    assert cells > 2 ** 32
    # the 2k split cells: their first push at positions spread over the whole list, both sides of 2^32
    at = torch.linspace(1000, cells - 1000, 2 * k, device="cuda").long()
    assert int(at[-1]) > 2 ** 32 and int(at[0]) < 2 ** 32
    big = float(2 ** 24)
    val[at] = big
    drop, kept = at[:k], at[k:]
    second = torch.cat([torch.full((k,), 1.0), torch.full((k,), -big)]).cuda()
    third = torch.cat([torch.full((k,), -big), torch.full((k,), 1.0)]).cuda()
    tail = slice(cells, cells + 4 * k)
    row[tail] = torch.cat([row[at], row[at]])
    col[tail] = torch.cat([col[at], col[at]])
    val[tail] = torch.cat([second, third])
    cell_drop = (row[drop].long(), col[drop].long())
    cell_keep = (row[kept].long(), col[kept].long())
    length = cells + 4 * k
    torch.cuda.synchronize()
    A = sp.CsrMatrix.from_device_triplets(n, n, length, row.data_ptr(), col.data_ptr(), val.data_ptr(), np.float32)
    sp.default_context().sync()
    nnz = cells - k
    assert A.nnz() == nnz and A.device_ptr64() is not None           # wide
    del row, col, val, at, drop, kept, second, third
    gc.collect()
    torch.cuda.empty_cache()
    # expectation, row slice by row slice: the band's cells in column order, the dropped ones removed, the
    # kept split cells equal to 1
    offs = torch.arange(-half, half + 1, device="cuda", dtype=torch.int64)
    counts = torch.full((n,), 2 * half + 1, device="cuda", dtype=torch.int64)
    edge = torch.arange(half, device="cuda", dtype=torch.int64)
    counts[:half] -= half - edge
    counts[n - half:] -= edge + 1
    counts.index_add_(0, cell_drop[0], torch.full_like(cell_drop[0], -1))
    ptr = torch.zeros(n + 1, device="cuda", dtype=torch.int64)
    ptr[1:] = torch.cumsum(counts, 0)
    del counts
    p64 = g.device_view(torch, A.device_ptr64(), n + 1, torch.int64)
    assert torch.equal(p64, ptr)
    _, ai, av = A.device_ptrs()
    chunk = 1 << 21
    for s in range(0, n, chunk):
        e = min(n, s + chunk)
        i = torch.arange(s, e, device="cuda", dtype=torch.int64)[:, None].expand(-1, offs.numel())
        d = offs[None, :].expand(e - s, -1)
        j = i + d
        ok = (j >= 0) & (j < n)
        v = g.band_value(torch, i, d).float()
        for (rr, cc), kind in ((cell_drop, "drop"), (cell_keep, "keep")):
            sel = (rr >= s) & (rr < e)
            li, ld = rr[sel] - s, cc[sel] - rr[sel] + half
            if kind == "drop":
                ok[li, ld] = False
            else:
                v[li, ld] = 1.0
        want_i, want_v = j[ok].to(torch.int32), v[ok]
        lo, hi = int(ptr[s]), int(ptr[e])
        assert hi - lo == want_i.numel()
        assert torch.equal(g.device_view(torch, ai + 4 * lo, hi - lo, torch.int32), want_i), s
        assert torch.equal(g.device_view(torch, av + 4 * lo, hi - lo, torch.int32), want_v.view(torch.int32)), s
        del i, d, j, ok, v, want_i, want_v
