"""One-byte value codes in the band kernel: a band matrix with at most 256 distinct values (by bit pattern) streams a
code per entry and reads the value from a dictionary in shared memory (spmv_band_codes_kernel).  Every case compares,
bit for bit (NaN included), the code route, the route off (SPL_STREAM_BAND_CODES=0: the band kernel on the values)
and the vector kernel, and all of them with the oracle (bit for bit with one lane per row).  torch.profiler shows which
kernel ran."""
import ctypes as C

import numpy as np
import pytest

import spalinalg_b200 as sp
from spalinalg_b200 import _capi as capi
from tests.test_spmv_band import band_csr, check_oracle, env, kernels_run, same

pytestmark = pytest.mark.gpu

K9 = list(range(-4, 5))


def with_dictionary(a, rng, count, dtype, special=()):
    """a with its values drawn from `count` distinct values (each of them used), `special` among them"""
    while True:
        d = np.concatenate([np.asarray(special, dtype), (rng.standard_normal(count - len(special)) * 0.5).astype(dtype)])
        if len(np.unique(d.view(np.uint64 if d.dtype.itemsize == 8 else np.uint32))) == count:
            break
    idx = rng.integers(0, count, len(a[2]))
    idx[:count] = np.arange(count)
    return a[0], a[1], d[idx]


def nan_with_payload(dtype, payload):
    if np.dtype(dtype) == np.float64:
        return np.array([0x7FF8000000000000 | payload], np.uint64).view(np.float64)[0]
    return np.array([0x7FC00000 | payload], np.uint32).view(np.float32)[0]


def all_ones(dtype):
    """the NaN with every bit set"""
    if np.dtype(dtype) == np.float64:
        return np.array([0xFFFFFFFFFFFFFFFF], np.uint64).view(np.float64)[0]
    return np.array([0xFFFFFFFF], np.uint32).view(np.float32)[0]


def three_products(run, y):
    """y of the code route, of the route off and of the vector kernel, and the kernel names of the first two"""
    import torch
    out, names = [], []
    for kernel, codes in ((capi.SPL_SPMV_STREAM, 1), (capi.SPL_SPMV_STREAM, 0), (capi.SPL_SPMV_VECTOR, 1)):
        y.fill_(7.0)
        torch.cuda.synchronize()
        with env(SPL_STREAM_BAND_CODES=codes):
            names.append(kernels_run(lambda: run(kernel)))
        sp.default_context().sync()
        out.append(y.clone())
    return out, names


def check_routes(run, y, n, a, x, lanes, dtype, codes=True):
    (yc, yo, yv), (kc, ko, _) = three_products(run, y)
    assert same(yc, yo) and same(yc, yv)
    assert ("spmv_band_codes_kernel" in kc) == codes and "spmv_band_codes_kernel" not in ko
    assert "spmv_band_kernel" in ko and (codes or "spmv_band_kernel" in kc)
    check_oracle(yc.cpu().numpy(), n, a, x, lanes, dtype)


def device_run(A, x, y):
    return lambda k: A.spmv_device(x.data_ptr(), y.data_ptr(), kernel=k)


def band_with_values(n, count, dtype, seed, offs=K9, ncols=None, special=()):
    import torch
    rng = np.random.default_rng(seed)
    ncols = ncols or n
    a = with_dictionary(band_csr(n, ncols, offs, rng, dtype), rng, count, dtype, special)
    A = sp.CsrMatrix.new(n, ncols, *a)
    x = rng.standard_normal(ncols).astype(dtype)
    xd = torch.from_numpy(x).cuda()
    yd = torch.empty(n, dtype=xd.dtype, device="cuda")
    return a, A, x, xd, yd


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("count", [1, 35, 256, 257])
def test_codes_distinct_counts(dtype, count):
    """Up to 256 distinct values take the code route, 257 do not."""
    n = 300_001
    a, A, x, xd, yd = band_with_values(n, count, dtype, 20 + count)
    check_routes(device_run(A, xd, yd), yd, n, a, x, A.spmv_choice()[1], dtype, codes=count <= 256)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("offs", ["k3", "k33"])
def test_codes_band_widths(dtype, offs):
    """Other row lengths: 3 entries (one code group per entry is 32 bytes) and 33 (four lanes per row)."""
    n = 300_001
    o = {"k3": [-1, 0, 1], "k33": list(range(-16, 17))}[offs]
    a, A, x, xd, yd = band_with_values(n, 40, dtype, 30, offs=o)
    check_routes(device_run(A, xd, yd), yd, n, a, x, A.spmv_choice()[1], dtype)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("kind", ["zeros", "nans"])
@pytest.mark.parametrize("count", [256, 257])
def test_codes_count_by_bits(dtype, kind, count):
    """Values count by bit pattern: +0.0 and -0.0 are two values, and so are NaNs that differ in their payload (the
    NaN with every bit set among them).  With them, `count` distinct values in all: a dictionary that merged any of
    them would hold 256 or fewer at 257 and take the code route."""
    n = 300_001
    special = [0.0, -0.0] if kind == "zeros" else [nan_with_payload(dtype, 1), nan_with_payload(dtype, 2),
                                                   all_ones(dtype)]
    rng = np.random.default_rng(45)
    a = band_csr(n, n, K9, rng, dtype)
    a = with_dictionary(a, rng, count, dtype, special)
    if kind == "nans":                                   # few NaN entries, so that most rows stay finite
        v = a[2].copy()
        nan = np.isnan(v)
        nan[np.nonzero(nan)[0][:len(special)]] = False   # each NaN once at least
        keep = np.nonzero(~np.isnan(v))[0]
        v[nan] = v[keep[rng.integers(0, len(keep), int(nan.sum()))]]
        a = (a[0], a[1], v)
    assert len(np.unique(a[2].view(np.uint64 if np.dtype(dtype).itemsize == 8 else np.uint32))) == count
    A = sp.CsrMatrix.new(n, n, *a)
    import torch
    x = rng.standard_normal(n).astype(dtype)
    xd = torch.from_numpy(x).cuda()
    yd = torch.empty(n, dtype=xd.dtype, device="cuda")
    check_routes(device_run(A, xd, yd), yd, n, a, x, A.spmv_choice()[1], dtype, codes=count <= 256)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_codes_wide_pattern(dtype):
    """A pattern kBandWidthMax = 4096 columns wide (n x (n + 4096), columns r and r + 4096, no row off it): in f64
    eight stages of the code kernel do not fit next to the x window, so it runs with fewer."""
    n = 300_001
    a, A, x, xd, yd = band_with_values(n, 3, dtype, 47, offs=[0, 4096], ncols=n + 4096)
    check_routes(device_run(A, xd, yd), yd, n, a, x, A.spmv_choice()[1], dtype)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_codes_special_values(dtype):
    """+0.0 and -0.0 (two codes), NaNs with two payloads, the NaN with every bit set (in f64 the empty slot of the
    value sets, counted apart), +-inf and a subnormal in the dictionary.  y cannot tell +0.0 from -0.0 nor one NaN
    from another (test_codes_count_by_bits can); a wrong code for any of them shows as a finite row against a NaN one
    or the other way round."""
    n = 300_001
    tiny = np.finfo(dtype).tiny
    special = [0.0, -0.0, nan_with_payload(dtype, 1), nan_with_payload(dtype, 2), all_ones(dtype), np.inf, -np.inf,
               tiny / 4]
    rng = np.random.default_rng(40)
    a = band_csr(n, n, K9, rng, dtype)
    # few special entries, so that most rows stay finite: the dictionary holds them all the same
    d = np.concatenate([np.asarray(special, dtype), (rng.standard_normal(20) * 0.5).astype(dtype)])
    idx = rng.integers(len(special), len(d), len(a[2]))
    idx[:len(special)] = np.arange(len(special))
    idx[rng.integers(0, len(idx), 200)] = rng.integers(0, len(special), 200)
    a = (a[0], a[1], d[idx])
    A = sp.CsrMatrix.new(n, n, *a)
    import torch
    x = rng.standard_normal(n).astype(dtype)
    xd = torch.from_numpy(x).cuda()
    yd = torch.empty(n, dtype=xd.dtype, device="cuda")
    check_routes(device_run(A, xd, yd), yd, n, a, x, A.spmv_choice()[1], dtype)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_codes_many_values_late(dtype):
    """Few values in the first rows and many in the last ones: no codes (the count covers the whole matrix)."""
    n = 300_001
    rng = np.random.default_rng(50)
    a = band_csr(n, n, K9, rng, dtype)
    v = a[2].copy()
    head = len(v) - 3000
    v[:head] = np.asarray([0.25, -0.5, 1.5], dtype)[rng.integers(0, 3, head)]
    a = (a[0], a[1], v)
    A = sp.CsrMatrix.new(n, n, *a)
    import torch
    x = rng.standard_normal(n).astype(dtype)
    xd = torch.from_numpy(x).cuda()
    yd = torch.empty(n, dtype=xd.dtype, device="cuda")
    check_routes(device_run(A, xd, yd), yd, n, a, x, A.spmv_choice()[1], dtype, codes=False)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_codes_set_values(dtype):
    """set_values on a coded matrix, to more than 256 values and then to another set of at most 256: the next
    product follows the new values each time."""
    n = 300_001
    rng = np.random.default_rng(60)
    a, A, x, xd, yd = band_with_values(n, 35, dtype, 61)
    lanes = A.spmv_choice()[1]
    check_routes(device_run(A, xd, yd), yd, n, a, x, lanes, dtype)
    many = (rng.standard_normal(len(a[2])) * 0.5).astype(dtype)
    A.set_values(many)
    check_routes(device_run(A, xd, yd), yd, n, (a[0], a[1], many), x, lanes, dtype, codes=False)
    few = with_dictionary(a, rng, 200, dtype)[2]
    A.set_values(few)
    check_routes(device_run(A, xd, yd), yd, n, (a[0], a[1], few), x, lanes, dtype)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_codes_broken_rows(dtype):
    """Rows off the pattern in the middle of a CTA's range and on both sides of a CTA boundary (their tiles run on
    the CSR arrays), with CTAs that do not start on a 32-row code group."""
    import torch
    rng = np.random.default_rng(70)
    n = 1_000_003
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    grid = sms * 3                                       # SPL_STREAM_CTAS=3 below

    def first_row(ptr, b):                               # stream_partition_kernel's CTA start
        target = (int(ptr[-1]) + n) * b // grid
        return int(np.searchsorted(ptr[:-1].astype(np.int64) + np.arange(n), target, side="left")) & ~3
    a0 = band_csr(n, n, K9, rng, dtype)
    mid = (first_row(a0[0], 10) + first_row(a0[0], 11)) // 2 + 1
    q = first_row(a0[0], grid // 2)
    for _ in range(8):                                   # the dropped entries may move the boundary: follow it
        a = band_csr(n, n, K9, rng, dtype, drop=[(mid, mid + 2), (q - 1, q + 3), (q, q - 1)])
        if first_row(a[0], grid // 2) == q:
            break
        q = first_row(a[0], grid // 2)
    assert first_row(a[0], grid // 2) == q
    assert any(first_row(a[0], b) % 32 for b in range(1, grid))
    a = with_dictionary(a, rng, 35, dtype)
    A = sp.CsrMatrix.new(n, n, *a)
    x = rng.standard_normal(n).astype(dtype)
    xd = torch.from_numpy(x).cuda()
    yd = torch.empty_like(xd)
    with env(SPL_STREAM_CTAS=3):
        check_routes(device_run(A, xd, yd), yd, n, a, x, A.spmv_choice()[1], dtype)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("shift", [1, 3])
def test_codes_window_shard(dtype, shift):
    """A row shard at global rows [4e9, 4e9 + 300 001) through spl_spmv_window, with a window buffer that starts
    `shift` elements past a 16-byte boundary, ends at the footprint and sits between NaNs."""
    import torch
    rng = np.random.default_rng(80)
    r0, nloc, ncols = 4_000_000_000, 300_001, 4_294_000_000
    a = with_dictionary(band_csr(nloc, ncols, K9, rng, dtype, r0=r0), rng, 35, dtype)
    A = sp.CsrMatrix.new(nloc, ncols, *a)
    w0, w1 = r0 - 4, r0 + nloc + 4
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
    rebased = (a[0], a[1] - np.uint64(w0), a[2])
    check_routes(run, yd, nloc, rebased, xw, A.spmv_choice()[1], dtype)
    assert not torch.isnan(yd).any()


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_codes_iteration_back_to_back(dtype):
    """x_{t+1} = A x_t for 30 products launched back to back, bit for bit against the vector kernel: the dictionary
    is read before griddepcontrol.wait, x after it."""
    import torch
    rng = np.random.default_rng(90)
    n = 2_000_003
    a = with_dictionary(band_csr(n, n, K9, rng, dtype), rng, 35, dtype)
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
    assert "spmv_band_codes_kernel" in names
    yc, yv = iterate(capi.SPL_SPMV_STREAM), iterate(capi.SPL_SPMV_VECTOR)
    assert torch.isfinite(yc).all() and torch.equal(yc, yv)
