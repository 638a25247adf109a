"""Wide matrices (64-bit positions, wide.cu / wide_assemble.cu) at oracle sizes.  SPL_WIDE_MIN_NNZ makes every
matrix created with that many stored entries or more wide, so each wide kernel runs on small inputs and is
compared with the oracle and with the narrow kernel it mirrors:
- structure, transposes, conversions, downloads and assembly bit for bit with the oracle;
- SpMV within rtol * sum|a||x| of the oracle, and bit for bit with the narrow vector kernel at the same lanes
  per row (same lane order, same U = 4); with one lane per row bit for bit with the oracle too;
- the refusals (SPL_ERR_UNSUPPORTED) of everything the wide form does not support.
Every test first checks that the matrix it means to be wide is wide, so a knob that does nothing fails."""
import ctypes as C
import gc

import numpy as np
import pytest

import oracle as orc
import spalinalg_b200 as sp
from spalinalg_b200 import _capi as capi
from tests.test_wide_assembly import case, from_device, same

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

KNOB = "SPL_WIDE_MIN_NNZ"
BUCKET = "SPL_ASSEMBLE_BUCKET_MAX"
DTYPES = [np.float64, np.float32]
SPMV_RTOL = {np.dtype(np.float64): 1e-12, np.dtype(np.float32): 1e-5}
CLS = {"row": sp.CsrMatrix, "col": sp.CscMatrix}
TORCH = {np.dtype(np.float32): torch.float32, np.dtype(np.float64): torch.float64}
UNSUPPORTED = capi.SPL_ERR_UNSUPPORTED
U = 4                                                    # entries in flight per lane in the vector kernels


@pytest.fixture
def wide(monkeypatch):
    """set(True): matrices created from now on with >= 1 stored entry are wide; set(False): the default."""
    def set_wide(on, min_nnz=1):
        if on:
            monkeypatch.setenv(KNOB, str(min_nnz))
        else:
            monkeypatch.delenv(KNOB, raising=False)
    return set_wide


def ctx():
    return sp.default_context()


def is_wide(m):
    return m.device_ptr64() is not None


def arrays(m):
    m._host = None                                       # download again: the device arrays are under test
    if isinstance(m, sp.CsrMatrix):
        return m.rowptr(), m.colind(), m.values()
    return m.colptr(), m.rowind(), m.values()


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)


def wide_lanes(mean):
    """Lanes per row of wide_spmv_t (wide.cu): 1 up to a mean row length of 10, 2 up to 12, then 4 .. 32."""
    lanes = 4 if mean > 12.0 else 1
    while lanes < 32 and lanes * 10 < mean:
        lanes *= 2
    return lanes


def scatter_lanes(mean):
    """Lanes per input major of wide_minor_scatter_kernel (wide.cu)."""
    return 1 if mean <= 2.0 else 4 if mean <= 12.0 else 8 if mean <= 64.0 else 32


def repair_shape(longest):
    """<lanes per segment, entries per lane> of wide_segment_repair_kernel (wide.cu); None: no repair."""
    if longest <= 1:
        return None
    for cap, shape in ((16, (8, 2)), (32, (16, 2)), (64, (32, 2)), (128, (32, 4)), (256, (32, 8))):
        if longest <= cap:
            return shape
    raise ValueError("longer than the repair pass ranks")


def random_values(rng, n, dtype):
    """Magnitudes over 20 binades: the summation order shows in the last bits."""
    return (rng.standard_normal(n) * 2.0 ** rng.integers(-10, 10, n)).astype(dtype)


def csr_from_lengths(rng, lengths, ncols, dtype, last_col_rows=()):
    """Rows of the given lengths with distinct sorted columns below ncols - 1; the rows in last_col_rows end
    at column ncols - 1, which no other row uses."""
    ind = []
    for r, n in enumerate(lengths):
        if r in last_col_rows:
            ind.append(np.append(np.sort(rng.choice(ncols - 1, n - 1, replace=False)), ncols - 1))
        else:
            ind.append(np.sort(rng.choice(ncols - 1, n, replace=False)))
    ptr = np.zeros(len(lengths) + 1, np.uint64)
    ptr[1:] = np.cumsum(lengths)
    ind = np.concatenate(ind).astype(np.uint64)
    return ptr, ind, random_values(rng, len(ind), dtype)


# ------------------------------------------------------------------ SpMV
def spmv_case(seed, mean, lanes, dtype):
    """CSR with a mean row length of exactly `mean`: every 9th row empty, a ragged last row (length not a multiple
    of U * lanes), and one row (`inf_row`) of length U * lanes + 1 whose last entry is the only use of column
    ncols - 1: that entry is the first slot of a lane whose other U - 1 slots are masked and read it again."""
    rng = np.random.default_rng(seed)
    nrows = max(120000 // mean, 300)
    ncols = 1200
    lengths = rng.integers(1, 2 * mean, nrows)
    lengths[::9] = 0
    inf_row = nrows // 2 + 1
    lengths[inf_row] = U * lanes + 1
    lengths[-1] = U * lanes + 3
    fixed = np.zeros(nrows, bool)
    fixed[[inf_row, nrows - 1]] = True
    grow = np.flatnonzero((lengths > 0) & ~fixed)
    short = mean * nrows - int(lengths.sum())
    assert short > 0
    np.add.at(lengths, rng.choice(grow, short), 1)
    assert lengths.sum() == mean * nrows and lengths.max() < ncols
    ptr, ind, val = csr_from_lengths(rng, lengths, ncols, dtype, last_col_rows=(inf_row,))
    x = random_values(rng, ncols, dtype)
    x[ncols - 1] = np.inf
    return nrows, ncols, ptr, ind, val, x, lengths, inf_row


def device_spmv(A, x, kernel=capi.SPL_SPMV_AUTO, lanes=0):
    """y = A x through spl_spmv_ex, y filled with 7.0 first (rows the kernel skipped would show)."""
    xd = torch.from_numpy(x).cuda()
    yd = torch.full((A.nrows(),), 7.0, dtype=TORCH[x.dtype], device="cuda")
    torch.cuda.synchronize()
    A.spmv_device(xd.data_ptr(), yd.data_ptr(), kernel=kernel, lanes=lanes)
    ctx().sync()
    return yd.cpu().numpy()


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("mean,lanes", [(5, 1), (11, 2), (20, 4), (50, 8), (100, 16), (400, 32)])
def test_wide_spmv_every_lane_count(wide, dtype, mean, lanes):
    nrows, ncols, ptr, ind, val, x, lengths, inf_row = spmv_case(7 * lanes + (dtype == np.float32), mean, lanes, dtype)
    assert wide_lanes(float(ptr[-1]) / nrows) == lanes
    wide(True)
    A = sp.CsrMatrix.new(nrows, ncols, ptr, ind, val)
    assert is_wide(A)
    wide(False)
    N = sp.CsrMatrix.new(nrows, ncols, ptr, ind, val)
    assert not is_wide(N)

    y = device_spmv(A, x)
    # the narrow vector kernel on the same arrays at the same lanes: same lane order, same U, same bits
    y_narrow = device_spmv(N, x, kernel=capi.SPL_SPMV_VECTOR, lanes=lanes)
    assert np.array_equal(bits(y), bits(y_narrow))
    # the oracle: same non-finite positions, the rest within the componentwise bound
    want = orc.csr_spmv(nrows, ptr, ind, val, x)
    scale = orc.csr_spmv(nrows, ptr, ind, np.abs(val), np.abs(x))
    assert np.array_equal(np.isnan(y), np.isnan(want)) and np.array_equal(np.isposinf(y), np.isposinf(want))
    assert np.array_equal(np.isneginf(y), np.isneginf(want))
    assert not np.isfinite(y[inf_row]) and np.isfinite(np.delete(y, inf_row)).all()
    ok = np.isfinite(want)
    assert np.all(np.abs(y[ok] - want[ok]) <= SPMV_RTOL[np.dtype(dtype)] * scale[ok])
    assert np.array_equal(bits(y[lengths == 0]), np.zeros(int((lengths == 0).sum()), bits(y).dtype))   # +0.0
    if lanes == 1:                                        # one lane per row sums in ascending column order
        assert np.array_equal(bits(y), bits(want))
    # spl_spmv_host, pageable and pinned vectors
    assert np.array_equal(bits(A.matvec(x)), bits(y))
    xp = sp.pinned_empty(ncols, dtype)
    xp[:] = x
    yp = sp.pinned_empty(nrows, dtype)
    A.matvec(xp, out=yp)
    assert np.array_equal(bits(yp), bits(y))
    assert A.spmv_choice() == (capi.SPL_SPMV_VECTOR, 0)
    # the kernel argument is ignored on a wide matrix: every kernel and lanes value gives the same bytes
    for kernel in (capi.SPL_SPMV_AUTO, capi.SPL_SPMV_VECTOR, capi.SPL_SPMV_MERGE, capi.SPL_SPMV_SPLIT,
                   capi.SPL_SPMV_SLICED, capi.SPL_SPMV_STREAM, capi.SPL_SPMV_SCATTER, 0x7f):
        for forced in (0, 1, 32):
            assert np.array_equal(bits(device_spmv(A, x, kernel, forced)), bits(y)), (kernel, forced)


# ------------------------------------------------------------------ transpose / CSR <-> CSC
def by_minor_counts(seed, nmajor, nminor, longest, dtype):
    """Compressed arrays (major = row of a CSR) whose longest minor segment (output segment of a transpose) has
    exactly `longest` entries: minor j gets a random count in [0, longest] (every 11th none, the middle one
    `longest`) of distinct majors; every 13th major stays empty when there are enough."""
    rng = np.random.default_rng(seed)
    counts = rng.integers(0, longest + 1, nminor)
    counts[::11] = 0
    counts[nminor // 2] = longest
    empty = np.arange(0, nmajor, 13) if nmajor >= 2 * 13 else np.array([], np.int64)
    avail = np.setdiff1d(np.arange(nmajor), empty)
    maj = np.concatenate([rng.choice(avail, c, replace=False) for c in counts])
    mn = np.repeat(np.arange(nminor), counts)
    order = np.lexsort((mn, maj))
    maj, mn = maj[order], mn[order]
    ptr = np.zeros(nmajor + 1, np.uint64)
    ptr[1:] = np.cumsum(np.bincount(maj, minlength=nmajor))
    val = random_values(rng, len(mn), dtype)
    val[::17] = -0.0
    return ptr, mn.astype(np.uint64), val


# (nmajor, nminor, longest output segment) -> scatter lanes, repair shape
TRANSPOSE_CASES = {
    "scatter1-norepair": ((3000, 4000, 1), 1, None),
    "scatter1-repair8x2": ((5000, 1000, 16), 1, (8, 2)),
    "scatter4-repair8x2": ((1000, 1000, 16), 4, (8, 2)),
    "scatter8-repair16x2": ((500, 1500, 32), 8, (16, 2)),
    "scatter32-repair32x2": ((400, 2000, 64), 32, (32, 2)),
    "scatter8-repair32x4": ((300, 200, 128), 8, (32, 4)),
    "scatter32-repair32x8": ((300, 200, 256), 32, (32, 8)),
    "one-major": ((1, 500, 1), 32, None),
    "one-minor": ((400, 1, 256), 1, (32, 8)),
}


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("fmt", ["row", "col"])
@pytest.mark.parametrize("name", list(TRANSPOSE_CASES))
def test_wide_transpose_and_convert(wide, dtype, fmt, name):
    (nmajor, nminor, longest), lanes, shape = TRANSPOSE_CASES[name]
    ptr, ind, val = by_minor_counts(nmajor * 7 + nminor + (dtype == np.float32), nmajor, nminor, longest, dtype)
    assert scatter_lanes(float(ptr[-1]) / nmajor) == lanes
    assert int(np.bincount(ind.astype(np.int64), minlength=nminor).max()) == longest and repair_shape(longest) == shape
    cls = CLS[fmt]
    nr, nc = (nmajor, nminor) if fmt == "row" else (nminor, nmajor)
    wide(True)
    A = cls.new(nr, nc, ptr, ind, val)
    assert is_wide(A)
    want = orc.recompress(nmajor, nminor, ptr, ind, val)
    B = A.to_csc() if fmt == "row" else A.to_csr()                      # other format, same matrix
    assert is_wide(B) and B.shape() == (nr, nc)
    same(arrays(B), want, "convert")
    same(arrays(B.to_csr() if fmt == "row" else B.to_csc()), (ptr, ind, val), "convert back")
    T = A.transpose()                                                  # same format, dims swapped
    assert is_wide(T) and type(T) is cls and T.shape() == (nc, nr)
    same(arrays(T), want, "transpose")
    TT = T.transpose()
    assert is_wide(TT)
    same(arrays(TT), (ptr, ind, val), "transpose twice")
    # the same format: a wide copy that outlives the original
    copy = A._convert(cls)
    assert is_wide(copy)
    del A
    gc.collect()
    ctx().sync()
    same(arrays(copy), (ptr, ind, val), "copy")
    same(arrays(copy.transpose()), want, "transpose of the copy")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("fmt", ["row", "col"])
@pytest.mark.parametrize("dims", [(400, 1), (300, 600)])
def test_wide_transpose_refuses_segments_above_256(wide, dtype, fmt, dims):
    nmajor, nminor = dims
    ptr, ind, val = by_minor_counts(nmajor + nminor, nmajor, nminor, 257, dtype)
    cls = CLS[fmt]
    nr, nc = (nmajor, nminor) if fmt == "row" else (nminor, nmajor)
    wide(True)
    A = cls.new(nr, nc, ptr, ind, val)
    assert is_wide(A)
    lib = ctx()._lib
    for call in (lambda h: lib.spl_mat_transpose(ctx()._h, A._h, C.byref(h)),
                 lambda h: lib.spl_mat_convert(ctx()._h, A._h, 1 - cls._FORMAT, C.byref(h))):
        h = C.c_void_p(0x1234)
        assert call(h) == UNSUPPORTED and h.value is None
    same(arrays(A), (ptr, ind, val), "input after the refusal")


# ------------------------------------------------------------------ construction and validation
def test_wide_new_panics_match_oracle(wide, goldens):
    """The reference's #[should_panic] constructions through the host constructor with every nonempty matrix
    wide: the same failing assertion as the oracle's."""
    wide(True)
    for cls, major, key in ((sp.CsrMatrix, "row", "csr"), (sp.CscMatrix, "col", "csc")):
        for m in goldens["valid_constructions"][key]:
            assert is_wide(cls.new(*m))
        for name, (nr, nc, ptr, ind, val) in goldens[f"{key}_new_panics"]["cases"].items():
            with pytest.raises(sp.Panic):
                cls.new(nr, nc, ptr, ind, val)
            assert ctx().invalid_reason() == orc.validate_compressed(nr, nc, ptr, ind, len(val), major), name


# nrows, ncols, ptr, ind (CSR layout; the CSC cases swap the dims) -> failing assertion, 0 = valid
VALIDATION_CASES = {
    "unsorted-ptr": (3, 6, [0, 3, 2, 4], [0, 2, 4, 1], 7),
    "index-out-of-range": (3, 6, [0, 2, 3, 4], [1, 6, 0, 5], 8),
    "repeated-index": (3, 6, [0, 1, 4, 4], [2, 1, 1, 3], 9),
    "descent-on-row-boundary-after-empty-rows": (6, 6, [0, 2, 2, 2, 2, 4, 5], [3, 5, 0, 1, 0], 0),
    "descent-inside-row-after-empty-rows": (6, 6, [0, 2, 2, 2, 2, 4, 5], [3, 5, 1, 0, 0], 9),
}


def major_of(cls):
    return "row" if cls is sp.CsrMatrix else "col"


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("cls", [sp.CsrMatrix, sp.CscMatrix])
@pytest.mark.parametrize("name", list(VALIDATION_CASES))
def test_wide_validation_host_and_device_constructors(wide, dtype, cls, name):
    nmajor, nminor, ptr, ind, reason = VALIDATION_CASES[name]
    nr, nc = (nmajor, nminor) if cls is sp.CsrMatrix else (nminor, nmajor)
    ptr, ind = np.array(ptr, np.uint64), np.array(ind, np.uint64)
    val = np.arange(1, len(ind) + 1, dtype=dtype)
    assert orc.validate_compressed(nr, nc, ptr, ind, len(val), major_of(cls)) == reason
    wide(True, min_nnz=len(ind))                                       # nnz >= n: wide
    one_major = np.concatenate([[0], np.full(nmajor, len(ind))]).astype(np.uint64)
    assert is_wide(cls.new(nr, nc, one_major, np.arange(len(ind), dtype=np.uint64), val))
    # host constructor
    if reason:
        with pytest.raises(sp.Panic):
            cls.new(nr, nc, ptr, ind, val)
        assert ctx().invalid_reason() == reason
    else:
        A = cls.new(nr, nc, ptr, ind, val)
        assert is_wide(A)
        same(arrays(A), (ptr, ind, val))
    # device constructor with 64-bit pointers, validating
    pd = torch.from_numpy(ptr.astype(np.int64)).cuda()
    idd = torch.from_numpy(ind.astype(np.int32)).cuda()
    vd = torch.from_numpy(val).cuda()
    torch.cuda.synchronize()
    make = lambda nnz, p=pd: cls.from_device_arrays64(nr, nc, nnz, p.data_ptr(), idd.data_ptr(), vd.data_ptr(), dtype)
    if reason:
        with pytest.raises(sp.Panic):
            make(len(ind))
        assert ctx().invalid_reason() == reason
    else:
        A = make(len(ind))
        assert is_wide(A)
        same(arrays(A), (ptr, ind, val))
    # ptr[0] != 0 (4) and ptr[n] != nnz (5): spl_mat_from_compressed_dev64 checks both before it chooses wide or
    # narrow storage, so these pin the device constructor's reasons, not wide.cu's validation
    bad = pd.clone()
    bad[0] = 1
    torch.cuda.synchronize()
    with pytest.raises(sp.Panic):
        make(len(ind), bad)
    assert ctx().invalid_reason() == 4
    with pytest.raises(sp.Panic):
        make(len(ind) + 1)
    assert ctx().invalid_reason() == 5


@pytest.mark.parametrize("cls", [sp.CsrMatrix, sp.CscMatrix])
def test_wide_host_constructor_index_beyond_2_pow_32(wide, cls):
    ptr = np.array([0, 2, 3], np.uint64)
    ind = np.array([0, (1 << 32) + 1, 1], np.uint64)                 # narrows to a valid-looking index
    val = np.ones(3)
    nr, nc = (2, 4) if cls is sp.CsrMatrix else (4, 2)
    assert orc.validate_compressed(nr, nc, ptr, ind, 3, major_of(cls)) == 8
    wide(True)
    assert is_wide(cls.new(nr, nc, ptr, np.array([0, 3, 1], np.uint64), val))
    with pytest.raises(sp.Panic):
        cls.new(nr, nc, ptr, ind, val)
    assert ctx().invalid_reason() == 8


def test_knob_threshold(wide):
    """SPL_WIDE_MIN_NNZ=n: n stored entries or more -> wide, fewer -> narrow, at each of the three places that
    choose the storage of a new matrix.  A value that is not a number leaves the default (narrow)."""
    rng = np.random.default_rng(3)
    ptr, ind, val = csr_from_lengths(rng, [3, 0, 5, 1], 9, np.float64)
    nnz = int(ptr[-1])
    pd = torch.from_numpy(ptr.astype(np.int64)).cuda()
    idd = torch.from_numpy(ind.astype(np.int32)).cuda()
    vd = torch.from_numpy(val).cuda()
    r = np.repeat(np.arange(4), np.diff(ptr).astype(np.int64)).astype(np.uint64)
    torch.cuda.synchronize()
    for n, expect in ((nnz, True), (nnz + 1, False), (0, True), (1 << 40, False), ("off", False), ("4x", False)):
        wide(True, min_nnz=n)
        A = sp.CsrMatrix.new(4, 9, ptr, ind, val)
        B = sp.CsrMatrix.from_device_arrays64(4, 9, nnz, pd.data_ptr(), idd.data_ptr(), vd.data_ptr(), np.float64)
        with pytest.MonkeyPatch.context() as mp:
            mp.setenv(BUCKET, "2")
            D = sp.CsrMatrix.from_coo(sp.CooMatrix.with_triplets(4, 9, r, ind, val))
        for m in (A, B, D):
            assert is_wide(m) == expect, n
            same(arrays(m), (ptr, ind, val))
    wide(True)                                                         # a matrix without entries is never wide
    assert not is_wide(sp.CsrMatrix.new(2, 3, np.zeros(3, np.uint64), np.zeros(0, np.uint64), np.zeros(0)))
    # SPL_ASSEMBLE_BUCKET_MAX that is not a number: the direct 32-bit route, whose output is never wide
    with pytest.MonkeyPatch.context() as mp:
        mp.setenv(BUCKET, "off")
        D = sp.CsrMatrix.from_coo(sp.CooMatrix.with_triplets(4, 9, r, ind, val))
    assert not is_wide(D)
    same(arrays(D), (ptr, ind, val))


# ------------------------------------------------------------------ download and entry chunks
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("fmt", ["row", "col"])
def test_wide_download_and_entry_chunks(wide, dtype, fmt):
    rng = np.random.default_rng(11 + (fmt == "col"))
    lengths = rng.integers(1, 12, 120)
    lengths[1:4] = 0                                                   # row 4 follows three empty rows
    lengths[50:53] = 0
    lengths[4] = 9
    ptr, ind, val = csr_from_lengths(rng, lengths, 40, dtype)
    nmajor, nminor = len(lengths), 40
    nnz = int(ptr[-1])
    cls = CLS[fmt]
    nr, nc = (nmajor, nminor) if fmt == "row" else (nminor, nmajor)
    wide(True)
    A = cls.new(nr, nc, ptr, ind, val)
    assert is_wide(A) and A.nnz() == nnz
    same(arrays(A), (ptr, ind, val), "download")
    trip = orc.expand_to_coo(nmajor, ptr, ind, val, fmt)
    chunks = [(int(ptr[4]) + 3, 20),                                   # starts mid-row
              (int(ptr[4]), 15),                                       # starts at a row after empty rows
              (int(ptr[53]), 7),                                       # the same after the second run
              (nnz - 1, 1),                                            # the last entry
              (0, nnz),                                                # everything
              (nnz, 0)]                                                # nothing, at the end
    for start, count in chunks:
        r, c, v = A.read_entries(start, count)
        t = trip[start:start + count]
        assert np.array_equal(r, t["row"]) and np.array_equal(c, t["col"]), (start, count)
        assert v.tobytes() == np.ascontiguousarray(t["val"]).tobytes(), (start, count)
    lib = ctx()._lib
    buf = np.empty(4, np.uint64), np.empty(4, np.uint64), np.empty(4, dtype)
    for start, count in ((nnz - 2, 3), (nnz + 1, 0), (1 << 40, 1)):
        st = lib.spl_mat_read_entries(ctx()._h, A._h, start, count, *(b.ctypes.data for b in buf))
        assert st == capi.SPL_ERR_ARG, (start, count)
    A.ITER_CHUNK = 7
    want = list(zip(trip["row"].tolist(), trip["col"].tolist(), trip["val"].tolist()))
    assert list(A.iter()) == want


# ------------------------------------------------------------------ assembly with a wide output
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("major", ["row", "col"])
@pytest.mark.parametrize("flags", [(1, 1), (0, 0)])
def test_wide_assembly_device_triplets(wide, monkeypatch, dtype, major, flags):
    """Buckets of 300 triplets (a major of 2000 spans many), duplicates spread over the whole list: the stitch
    writes ptr64; the result equals the oracle and the same list assembled narrow."""
    dedup, dropzero = flags
    nr, nc = (3000, 5000) if major == "row" else (5000, 3000)
    r, c, v = case(21 + (major == "row") + 2 * dedup, nr, nc, major, dtype, dedup)
    want = orc.compress_from_coo(nr, nc, orc.make_triplets(r, c, v), major, dedup, dropzero)
    monkeypatch.setenv(BUCKET, "300")
    wide(False)
    narrow = from_device(major, nr, nc, r, c, v, dedup, dropzero)
    assert not is_wide(narrow)
    wide(True)
    got = from_device(major, nr, nc, r, c, v, dedup, dropzero)
    assert is_wide(got)
    same(arrays(got), want, "wide stitch vs oracle")
    same(arrays(got), arrays(narrow), "wide stitch vs narrow stitch")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("major", ["row", "col"])
def test_wide_assembly_host_and_builder_fronts(wide, monkeypatch, dtype, major):
    nr, nc = 4000, 2500
    r, c, v = case(31, nr, nc, major, dtype, 1)
    want = orc.compress_from_coo(nr, nc, orc.make_triplets(r, c, v), major)
    monkeypatch.setenv(BUCKET, "500")
    wide(False)
    narrow = CLS[major].from_coo(sp.CooMatrix.with_triplets(nr, nc, r, c, v))
    assert not is_wide(narrow)
    wide(True)
    host = CLS[major].from_coo(sp.CooMatrix.with_triplets(nr, nc, r, c, v))
    builder = CLS[major].from_coo(sp.PinnedCooMatrix.with_triplets(nr, nc, r, c, v))
    for what, m in (("spl_mat_from_coo", host), ("builder", builder)):
        assert is_wide(m), what
        same(arrays(m), want, what)
        same(arrays(m), arrays(narrow), what + " vs narrow")


# ------------------------------------------------------------------ refusals
@pytest.mark.parametrize("dtype", DTYPES)
def test_wide_refusals_leave_the_operand_intact(wide, dtype):
    rng = np.random.default_rng(41)
    n = 300
    ptr, ind, val = csr_from_lengths(rng, rng.integers(0, 20, n), n, dtype)
    nnz = int(ptr[-1])
    x = random_values(rng, n, dtype)
    wide(True)
    A = sp.CsrMatrix.new(n, n, ptr, ind, val)
    Ac = A.to_csc()
    assert is_wide(A) and is_wide(Ac)
    wide(False)
    N = sp.CsrMatrix.new(n, n, ptr, ind, val)
    assert not is_wide(N)
    y0 = device_spmv(A, x)
    lib, h_ctx = ctx()._lib, ctx()._h
    tdt = TORCH[np.dtype(dtype)]
    xd = torch.from_numpy(x).cuda()
    yd = torch.full((n,), 7.0, dtype=tdt, device="cuda")
    coo_d = [torch.full((nnz,), 5, dtype=torch.int32, device="cuda"), torch.full((nnz,), 5, dtype=torch.int32, device="cuda"),
             torch.full((nnz,), 5.0, dtype=tdt, device="cuda")]
    torch.cuda.synchronize()
    coo_h = [np.full(nnz, 5, np.uint64), np.full(nnz, 5, np.uint64), np.full(nnz, 5.0, dtype)]
    y_host = np.full(n, 7.0, dtype)
    col_starts = np.array([0, n], np.uint64)
    slices = (C.c_void_p * 1)(xd.data_ptr())
    flags = torch.zeros(64, dtype=torch.int32, device="cuda")
    flag_ptrs = (C.c_void_p * 1)(flags.data_ptr())
    lo, hi = C.c_uint64(99), C.c_uint64(99)
    new_vals = np.zeros(nnz, dtype)

    def with_out(fn, *ops):
        h = C.c_void_p(0x1234)                                         # must come back NULL
        st = fn(h_ctx, *(m._h for m in ops), C.byref(h))
        return st if h.value is None else f"output {h.value:#x}"

    calls = {}
    for name in ("add", "sub", "mul"):
        fn = getattr(lib, f"spl_mat_{name}")
        calls[f"{name}(wide, wide)"] = lambda fn=fn: with_out(fn, A, A)
        calls[f"{name}(wide, narrow)"] = lambda fn=fn: with_out(fn, A, N)
        calls[f"{name}(narrow, wide)"] = lambda fn=fn: with_out(fn, N, A)
    calls["neg"] = lambda: with_out(lib.spl_mat_neg, A)
    calls["set_values"] = lambda: lib.spl_mat_set_values(h_ctx, A._h, new_vals.ctypes.data)
    calls["to_coo"] = lambda: lib.spl_mat_to_coo(h_ctx, A._h, *(b.ctypes.data for b in coo_h))
    calls["to_coo_dev"] = lambda: lib.spl_mat_to_coo_dev(h_ctx, A._h, *(b.data_ptr() for b in coo_d))
    calls["spmv_window"] = lambda: lib.spl_spmv_window(h_ctx, A._h, xd.data_ptr(), 0, n, yd.data_ptr())
    calls["spmv_footprint"] = lambda: lib.spl_spmv_footprint(h_ctx, A._h, C.byref(lo), C.byref(hi))
    calls["spmv_peer"] = lambda: lib.spl_spmv_peer(h_ctx, A._h, 1, 0, col_starts.ctypes.data,
                                                   C.cast(slices, C.c_void_p), yd.data_ptr())
    calls["spmv_peer_host"] = lambda: lib.spl_spmv_peer_host(h_ctx, A._h, 1, 0, col_starts.ctypes.data,
                                                             C.cast(slices, C.c_void_p), C.cast(flag_ptrs, C.c_void_p),
                                                             1, 1000, x.ctypes.data, y_host.ctypes.data)
    calls["spmv of a wide CSC"] = lambda: lib.spl_spmv_ex(h_ctx, Ac._h, xd.data_ptr(), yd.data_ptr(), 0)
    calls["spmv_host of a wide CSC"] = lambda: lib.spl_spmv_host(h_ctx, Ac._h, x.ctypes.data, y_host.ctypes.data)
    for what, call in calls.items():
        assert call() == UNSUPPORTED, what
        ctx().sync()
        torch.cuda.synchronize()
        assert np.array_equal(bits(device_spmv(A, x)), bits(y0)), what
    # nothing was written anywhere
    assert (yd.cpu().numpy() == 7.0).all() and (y_host == 7.0).all() and lo.value == 99 and hi.value == 99
    assert all((b == 5).all() for b in coo_h) and all(bool((b == 5).all()) for b in coo_d)
    same(arrays(A), (ptr, ind, val), "operand after the refusals")
    with pytest.raises(sp.DeviceError):
        Ac.matvec(x)
