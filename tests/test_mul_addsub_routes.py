"""A * B (spgemm.cu) and A + B / A - B (addsub.cu) on every kernel route, at the route boundaries, bit for bit
against the oracle.

Both operations choose their kernels from the operands' shapes.  Each case below is built for one route, and
before it runs it checks with a numpy restatement of the C++ rule (`mul_route`, `addsub_plan`) that it takes
that route, so a case that drifts off its route fails instead of quietly testing another one.
`test_cases_claim_their_routes` checks every case on the CPU at 148 SMs (a B200); the GPU tests check them again
at the device's SM count, and `test_mirrors_agree_with_the_launched_kernels` reads the launched kernels, their
grids and their shared memory from a profiler trace to check the mirrors themselves.

Routes of the product, with both operands read as CSR (CSC operands swapped, as `spgemm()` does):
- small_hash: every row of A has at most 128 products; a warp per row, 256-slot table (8 warps per CTA);
- large_hash: at most 1 024 products; 2 048-slot table (6 warps per CTA for f64, 8 for f32);
- sort32 / sort64: a row above 1 024 products; expand, radix sort on (row, column) keys of 32 or 64 bits;
- n_by_1: B has one column; expand, no sort.
A hash route also needs B to have more than one column and A at least one stored entry.
"""
import json
import math
import os
import re
import tempfile
from collections import namedtuple

import numpy as np
import pytest

import oracle as orc

DTYPES = [np.float64, np.float32]
B200_SMS = 148
HS_SMALL, HS_LARGE = 128, 1024            # products per row of the two hash tables
HS_SLOT_BITS = {"small_hash": 8, "large_hash": 11}
HS_HASH = 2654435761                      # hs_hash: (j * HS_HASH mod 2^32) >> (32 - SLOT_BITS)
ROUTER_THREADS = 256                      # row_products_kernel's block
GRID_PER_SM = 8                           # both spgemm grids are capped at 8 CTAs per SM


# ------------------------------------------------------------------ route mirrors (spgemm.cu, addsub.cu)
def bits_for(count):
    """common.cuh bits_for: bits needed for values in [0, count)."""
    return 0 if count <= 1 else int(count - 1).bit_length()


Mat = namedtuple("Mat", "nrows ncols fmt ptr ind val")     # fmt "csr" or "csc"; ptr / ind uint64


def nmajor(M):
    return M.nrows if M.fmt == "csr" else M.ncols


def nminor(M):
    return M.ncols if M.fmt == "csr" else M.nrows


def hash_warps(route, dtype):
    return 6 if route == "large_hash" and np.dtype(dtype).itemsize == 8 else 8


class MulRoute(namedtuple("MulRoute", "route an bn max_products products hash_grid warps router_grid")):
    @property
    def key_bits(self):
        return bits_for(self.an) + bits_for(self.bn)

    @property
    def hash_passes(self):
        """Rows a warp of the hash kernel takes (the grid-stride loop runs more than once above 1)."""
        return math.ceil(self.an / (self.hash_grid * self.warps))

    @property
    def router_passes(self):
        return math.ceil(self.an / (self.router_grid * ROUTER_THREADS))


def products_per_row(l, r):
    """Products of each row of l (CSR reading) against r: sum over its entries of r's row lengths."""
    rlen = np.diff(r.ptr.astype(np.int64))
    per_entry = rlen[l.ind.astype(np.int64)]
    cs = np.concatenate([[0], np.cumsum(per_entry)])
    p = l.ptr.astype(np.int64)
    return cs[p[1:]] - cs[p[:-1]]


def mul_route(a, b, sms, dtype):
    """spgemm() / spgemm_impl(): the route of a * b and the grids of the hash and row_products kernels."""
    assert a.fmt == b.fmt
    l, r = (a, b) if a.fmt == "csr" else (b, a)
    an, bn = nmajor(l), nminor(r)
    prods = products_per_row(l, r)
    maxp = int(prods.max()) if an else 0
    route = None
    if len(l.ind):                               # row_products and the hash routes need an entry of A
        if maxp <= HS_SMALL and bn > 1:
            route = "small_hash"
        elif maxp <= HS_LARGE and bn > 1:
            route = "large_hash"
    if route is None:
        route = "n_by_1" if bits_for(bn) == 0 else "sort64" if bits_for(an) + bits_for(bn) > 32 else "sort32"
    warps = hash_warps(route, dtype)
    return MulRoute(route, an, bn, maxp, prods, min(math.ceil(an / warps), GRID_PER_SM * sms), warps,
                    min(math.ceil(an / ROUTER_THREADS), GRID_PER_SM * sms))


AddsubPlan = namedtuple("AddsubPlan", "rows cap_a cap_b smem_numeric staged")


def addsub_plan(aptr, bptr):
    """plan_blocks() and each CTA's `staged` flag in union_block_kernel."""
    aptr, bptr = aptr.astype(np.int64), bptr.astype(np.int64)
    n = len(aptr) - 1
    ma, mb = float(aptr[-1]) / n, float(bptr[-1]) / n
    for rows in (128, 32):
        ca, cb = int(ma * rows * 1.25) + 64, int(mb * rows * 1.25) + 64
        in_words = (ca + ca // 32 + 1) + (cb + cb // 32 + 1)
        out_words = (ca + cb) + (ca + cb) // 32 + 1
        smem = in_words * 4 + out_words * 8 + 16
        if smem <= 64 * 1024 and ca + cb < 0xFFFF:
            break
    else:                                        # very long segments: every CTA merges from global memory
        ca, cb, smem = 0, 0, 64
    m0 = np.arange(0, n, rows)
    m1 = np.minimum(m0 + rows, n)
    staged = (aptr[m1] - aptr[m0] <= ca) & (bptr[m1] - bptr[m0] <= cb)
    return AddsubPlan(rows, ca, cb, smem, staged)


def hs_hash(j, slot_bits):
    return (np.asarray(j, np.uint32) * np.uint32(HS_HASH)) >> np.uint32(32 - slot_bits)


# ------------------------------------------------------------------ building blocks
def random_values(rng, n, dtype):
    """Magnitudes over 20 binades: the summation order shows in the last bits."""
    return (rng.standard_normal(n) * 2.0 ** rng.integers(-10, 10, n)).astype(dtype)


def csr(nrows, ncols, r, c, v):
    """CSR arrays of the entries (r, c, v); no cell twice."""
    r, c = np.asarray(r, np.int64), np.asarray(c, np.int64)
    order = np.lexsort((c, r))
    r, c, v = r[order], c[order], np.asarray(v)[order]
    assert not np.any((np.diff(r) == 0) & (np.diff(c) == 0)), "a cell twice"
    assert len(r) == 0 or (r[-1] < nrows and c.max() < ncols and c.min() >= 0)
    ptr = np.zeros(nrows + 1, np.uint64)
    ptr[1:] = np.cumsum(np.bincount(r, minlength=nrows))
    return ptr, c.astype(np.uint64), v


def random_entries(rng, rows, lengths, col_lo, col_hi):
    """About lengths[t] distinct columns in [col_lo, col_hi) for each row rows[t] (duplicates dropped)."""
    rr = np.repeat(np.asarray(rows, np.int64), lengths)
    cc = rng.integers(col_lo, col_hi, len(rr))
    key = np.unique(rr * (col_hi + 1) + cc)
    return key // (col_hi + 1), key % (col_hi + 1)


def concat(*parts):
    return tuple(np.concatenate([p[i] for p in parts]) for i in range(2))


class MulCase(namedtuple("MulCase", "n k m a b expect csc")):
    """C = A B with A n x k and B k x m given as CSR arrays.  csc = "mirror": the CSC run multiplies the CSC
    matrices whose arrays are b and a (the kernels see the very same arrays, so the route is the same);
    "native": it also multiplies the CSC forms of A and B themselves."""

    def forms(self):
        """(label, A, B, oracle arguments (an, ak, bn, l, r)) for every run of the case."""
        n, k, m, a, b = self.n, self.k, self.m, self.a, self.b
        yield "csr", Mat(n, k, "csr", *a), Mat(k, m, "csr", *b), (n, k, m, a, b)
        yield "csc", Mat(m, k, "csc", *b), Mat(k, n, "csc", *a), (n, k, m, a, b)
        if self.csc == "native":
            ac, bc = orc.recompress(n, k, *a), orc.recompress(k, m, *b)
            yield "csc-native", Mat(n, k, "csc", *ac), Mat(k, m, "csc", *bc), (m, k, n, bc, ac)


def check_mul_claims(case, sms, dtype, what):
    """Every form of the case takes the route it was built for, with the stated stride conditions."""
    e = case.expect
    for label, A, B, args in case.forms():
        rt = mul_route(A, B, sms, dtype)
        tag = f"{what} [{label}]"
        assert rt.route == e["route"], f"{tag}: route {rt.route}, built for {e['route']}"
        if "max_products" in e:
            assert rt.max_products == e["max_products"], f"{tag}: max products {rt.max_products}"
        if "key_bits" in e:
            assert rt.key_bits == e["key_bits"], f"{tag}: {rt.key_bits} key bits"
        if e.get("hash_strides"):                # warps take a second and third row; the limit row is in the last,
            per_pass = rt.hash_grid * rt.warps   # partial pass
            assert rt.hash_passes >= 3 and rt.an % per_pass, f"{tag}: {rt.hash_passes} hash passes"
            assert rt.products[-1] == e["max_products"], tag
        if "heavy_row" in e:                     # the one row above 1 024 products, where the router strides
            heavy = np.flatnonzero(rt.products > HS_LARGE)
            assert heavy.tolist() == [e["heavy_row"](rt.an)], f"{tag}: rows above 1024 products: {heavy[:5]}"
            assert rt.router_passes >= 2 and rt.router_grid == GRID_PER_SM * sms, tag
            if heavy[0]:
                assert heavy[0] >= rt.router_grid * ROUTER_THREADS, f"{tag}: the heavy row is in the first pass"
        if "probe_wrap" in e:                    # one row's columns all hash into the last slots and wrap to 0
            cols, slot_bits = e["probe_wrap"]
            h = hs_hash(cols, slot_bits)
            slots = 1 << slot_bits
            assert HS_SLOT_BITS[rt.route] == slot_bits and len(cols) == slots // 2, tag
            assert h.min() >= slots - 8 and int(h.min()) + len(cols) > slots, f"{tag}: no wrap (min slot {h.min()})"
        if "out_nnz" in e:
            assert len(orc.csr_mul(*args)[1]) == e["out_nnz"], tag


# ------------------------------------------------------------------ product cases
def grid_stride_case(sms, dtype, table):
    """About 3.5 x the rows one pass of the hash grid covers, so warps reset their table and take more rows.  Rows
    of B: 0-63 empty ("dead"), 64-127 64 entries (large table only), 128-159 32 entries from a small pool of
    columns (the limit rows), the rest 1-8 entries.  Rows of A: every 7th empty; rows whose 40 entries all hit
    dead rows of B (two 32-entry trips that yield no product), one of them followed by live entries; rows 0 and
    n - 1 at exactly the table's limit, n - 1 in the last, partial pass; for the large table every 13th row
    with three 64-entry rows of B."""
    route = "small_hash" if table == "small" else "large_hash"
    limit = HS_SMALL if table == "small" else HS_LARGE
    rng = np.random.default_rng(11 + 2 * (table == "large") + (dtype == np.float32))
    n = GRID_PER_SM * sms * hash_warps(route, dtype) * 7 // 2
    k = m = 4096
    live = np.arange(160, k)
    b_parts = [random_entries(rng, live, rng.integers(1, 9, len(live)), 0, m)]
    pool = rng.choice(m, 40 if table == "small" else 300, replace=False)
    b_parts.append((np.repeat(np.arange(128, 160), 32), np.concatenate([rng.choice(pool, 32, replace=False) for _ in range(32)])))
    if table == "large":
        b_parts.append(random_entries(rng, np.arange(64, 128), np.full(64, 64), 0, m))
    br, bc = concat(*b_parts)
    lens = rng.integers(0, 7, n)
    lens[::7] = 0
    dead_only, dead_then_live = [5, n // 2 + 1, n - 2], n // 2
    lens[[0, n - 1] + dead_only] = 0
    a_parts = [random_entries(rng, np.arange(n), lens, 160, k)]
    for i in dead_only + [dead_then_live]:
        a_parts.append((np.full(40, i), rng.choice(64, 40, replace=False)))
    per_limit_row = limit // 32
    for i in (0, n - 1):
        a_parts.append((np.full(per_limit_row, i), np.arange(128, 128 + per_limit_row)))
    if table == "large":
        fat = np.setdiff1d(np.arange(1, n - 1, 13), dead_only + [dead_then_live])
        a_parts.append((np.repeat(fat, 3), np.concatenate([rng.choice(np.arange(64, 128), 3, replace=False) for _ in fat])))
    ar, ac = concat(*a_parts)
    a = csr(n, k, ar, ac, random_values(rng, len(ar), dtype))
    b = csr(k, m, br, bc, random_values(rng, len(br), dtype))
    return MulCase(n, k, m, a, b, {"route": route, "max_products": limit, "hash_strides": True}, "mirror")


def router_case(sms, dtype, heavy):
    """More rows than row_products_kernel's grid covers in one pass, one entry per row; the only row above 1 024
    products is the last one (seen only by the grid-stride loop) or the first one."""
    rng = np.random.default_rng(21 + (heavy == "last") + 2 * (dtype == np.float32))
    stride = GRID_PER_SM * sms * ROUTER_THREADS
    n, k, m = stride + stride // 2 + 3, 4096, 2048
    h = n - 1 if heavy == "last" else 0
    br, bc = concat(random_entries(rng, np.arange(1, k), rng.integers(1, 4, k - 1), 0, m),
                    (np.zeros(1100, np.int64), rng.choice(m, 1100, replace=False)))
    ac = rng.integers(1, k, n)
    ac[h] = 0
    a = csr(n, k, np.arange(n), ac, random_values(rng, n, dtype))
    b = csr(k, m, br, bc, random_values(rng, len(br), dtype))
    heavy_row = (lambda an: an - 1) if heavy == "last" else (lambda an: 0)
    return MulCase(n, k, m, a, b, {"route": "sort32", "heavy_row": heavy_row, "key_bits": 30}, "mirror")


def boundary_case(dtype, products, way):
    """The most products of a row is exactly `products`, reached by row 1234 of A in one of two ways.  long: one
    entry of A against a row of B with `products` columns (1 024 of them are 32 product batches of one step).
    many: `products` entries of A against one-entry rows of B, all in column 77: a `products`-term sum in one
    entry of C.  Other rows have at most 24 products."""
    rng = np.random.default_rng(products * 2 + (way == "many") + 7 * (dtype == np.float32))
    n, k, m, i0 = 3000, 2048, 2048, 1234
    bg = np.arange(1100, k)
    b_parts = [random_entries(rng, bg, rng.integers(1, 7, len(bg)), 0, m)]
    lens = rng.integers(0, 5, n)
    lens[i0] = 0
    a_parts = [random_entries(rng, np.arange(n), lens, 1100, k)]
    if way == "long":
        a_parts.append((np.array([i0]), np.array([0])))
        b_parts.append((np.zeros(products, np.int64), rng.choice(m, products, replace=False)))
    else:
        a_parts.append((np.full(products, i0), np.arange(1, products + 1)))
        b_parts.append((np.arange(1, products + 1), np.full(products, 77)))
    ar, ac = concat(*a_parts)
    br, bc = concat(*b_parts)
    route = ("small_hash" if products <= HS_SMALL else "large_hash" if products <= HS_LARGE else "sort32")
    a = csr(n, k, ar, ac, random_values(rng, len(ar), dtype))
    b = csr(k, m, br, bc, random_values(rng, len(br), dtype))
    return MulCase(n, k, m, a, b, {"route": route, "max_products": products}, "mirror")


def key_width_case(dtype, n):
    """n x 4096 times 4096 x 65 536: (row, column) keys of 32 bits with the top bit in use (n = 65 536) or of 64
    bits (n = 65 537).  Row n - 1 of A takes rows 0-1099 of B, each of which ends at column 65 535, so the sort
    runs and the highest key is formed; the other rows are light.  The CSC forms of A and B cross the same line
    with their roles swapped (B^T's row 65 535 has the 1 100 products)."""
    rng = np.random.default_rng(n + 3 * (dtype == np.float32))
    k, m, h = 4096, 65536, n - 1
    br, bc = concat(random_entries(rng, np.arange(1100), rng.integers(1, 4, 1100), 0, m - 1),
                    (np.arange(1100), np.full(1100, m - 1)),
                    random_entries(rng, np.arange(1100, k), rng.integers(1, 4, k - 1100), 0, m))
    rows = np.arange(0, h, 4)
    ar, ac = concat(random_entries(rng, rows, rng.integers(1, 4, len(rows)), 1100, k),
                    (np.full(1100, h), np.arange(1100)))
    a = csr(n, k, ar, ac, random_values(rng, len(ar), dtype))
    b = csr(k, m, br, bc, random_values(rng, len(br), dtype))
    bits = bits_for(n) + bits_for(m)
    return MulCase(n, k, m, a, b, {"route": "sort64" if bits > 32 else "sort32", "key_bits": bits}, "native")


def probe_columns(slot_bits, ncols):
    """The half-table's worth of columns below ncols whose hash slots are the highest."""
    j = np.arange(ncols, dtype=np.uint32)
    h = hs_hash(j, slot_bits).astype(np.int64)
    order = np.lexsort((j, -h))
    return np.sort(j[order[:(1 << slot_bits) // 2]]).astype(np.int64)


def probe_case(dtype, table):
    """Row 0 inserts 128 (small table) or 1 024 (large table) columns that all hash into the table's last slots:
    the probe chains are as long as the table allows and wrap to slot 0.  Row 1 reaches the same limit through
    4 (8) rows of B holding overlapping subsets of those columns, so values accumulate along the chains."""
    slot_bits = 8 if table == "small" else 11
    cols = probe_columns(slot_bits, 1 << 16 if table == "small" else 1 << 20)
    m = int(cols.max()) + 1
    count, steps = len(cols), 4 if table == "small" else 8
    rng = np.random.default_rng(slot_bits + 5 * (dtype == np.float32))
    n = k = 64
    b_parts = [(np.zeros(count, np.int64), cols)]
    for t in range(1, steps + 1):
        b_parts.append((np.full(count // steps, t), rng.choice(cols, count // steps, replace=False)))
    bg = np.arange(steps + 1, k)
    b_parts.append(random_entries(rng, bg, rng.integers(1, 5, len(bg)), 0, m))
    lens = rng.integers(0, 5, n)
    lens[:2] = 0
    ar, ac = concat(random_entries(rng, np.arange(n), lens, steps + 1, k), (np.array([0]), np.array([0])),
                    (np.ones(steps, np.int64), np.arange(1, steps + 1)))
    br, bc = concat(*b_parts)
    a = csr(n, k, ar, ac, random_values(rng, len(ar), dtype))
    b = csr(k, m, br, bc, random_values(rng, len(br), dtype))
    route = "small_hash" if table == "small" else "large_hash"
    return MulCase(n, k, m, a, b, {"route": route, "max_products": count, "probe_wrap": (cols, slot_bits)}, "mirror")


def payload_nan(dtype, negative=False):
    """A quiet NaN with a payload (and the sign bit when negative)."""
    if np.dtype(dtype) == np.float32:
        return np.array([0xFFC01234 if negative else 0x7FC05678], np.uint32).view(np.float32)[0]
    return np.array([0xFFF8000000012345 if negative else 0x7FF800000006789A], np.uint64).view(np.float64)[0]


def fma_pair(dtype):
    """(c, a): c * 1 + a * a is 0 with the product rounded before the add and 2^-60 (f64) / 2^-26 (f32) when the
    two are contracted into a fused multiply-add; no rounding tie either way."""
    e = 2.0 ** (-13 if np.dtype(dtype) == np.float32 else -30)
    return -(1.0 + 2.0 * e), 1.0 + e


def special_rows(dtype):
    """Rows of C with one entry each, in column 0: the (A, B) value pairs of its products in ascending k."""
    f32 = np.dtype(dtype) == np.float32
    c, a = fma_pair(dtype)
    big = 2.0 ** (24 if f32 else 53)
    tiny = 2.0 ** (-70 if f32 else -530)            # tiny * tiny is subnormal and exact
    under = 2.0 ** (-80 if f32 else -600)           # under * under rounds to zero
    inf, mx = np.inf, float(np.finfo(dtype).max)
    nan, nneg = payload_nan(dtype), payload_nan(dtype, True)
    return [
        [(c, 1.0), (a, a)],                          # fused multiply-add detector
        [(big, 1.0), (1.0, 1.0), (-big, 1.0)],       # ascending k gives 0, any other order 1
        [(-0.0, 1.0)],                               # a first product of -0.0 is copied, not added to +0.0
        [(1.0, -0.0), (-0.0, 1.0)],
        [(-0.0, 1.0), (0.0, 1.0)],
        [(under, -under)],                           # a product that underflows to -0.0
        [(tiny, tiny)], [(tiny, tiny), (-tiny, 2.0 * tiny)], [(-tiny, tiny), (1.0, 0.0)],
        [(inf, 1.0)], [(-inf, 1.0)], [(inf, 0.0)], [(inf, 1.0), (-inf, 1.0)], [(1.0, 1.0), (inf, 1.0)],
        [(mx, 2.0)], [(mx, 1.0), (mx, 1.0)],
        [(0.0, 1.0)], [(1.0, 0.0)], [(3.0, 1.0), (-3.0, 1.0)], [(0.0, 5.0), (0.0, -5.0)],   # zeros stay stored
        [(nan, 1.0)], [(1.0, nneg)], [(nan, 1.0), (inf, 1.0)], [(1.0, 1.0), (nneg, 1.0)],
    ]


def values_case(dtype, route):
    """special_rows, each product k on a row of B of its own, plus one row of A that sizes the route: a row of B
    with 200 (large table) or 1 100 (sort) columns.  For n_by_1, B is k x 1."""
    rows = special_rows(dtype)
    pad = {"small_hash": 0, "large_hash": 200, "sort32": 1100, "n_by_1": 0}[route]
    ar, av, bv = [], [], []
    for i, prods in enumerate(rows):
        for x, y in prods:
            ar.append(i)
            av.append(x)
            bv.append(y)
    kk = len(ar)
    ac = list(range(kk))
    br, bc = list(range(kk)), [0] * kk
    n, m = len(rows) + 1, 1 if route == "n_by_1" else 2048
    if pad:
        rng = np.random.default_rng(pad)
        ar.append(len(rows)); ac.append(kk); av.append(1.5)
        br += [kk] * pad; bc += list(range(1, pad + 1)); bv += list(random_values(rng, pad, dtype))
        kk += 1
    a = csr(n, kk, ar, ac, np.array(av, dtype))
    b = csr(kk, m, br, bc, np.array(bv, dtype))
    return MulCase(n, kk, m, a, b, {"route": route}, "mirror")


def degenerate_case(dtype, name):
    rng = np.random.default_rng(len(name))
    empty = (np.array([], np.int64), np.array([], np.int64))

    def rand(nr, nc, lo=0, hi=None):
        r, c = random_entries(rng, np.arange(nr), rng.integers(0, 5, nr), lo, nc if hi is None else hi)
        return csr(nr, nc, r, c, random_values(rng, len(r), dtype))

    if name == "a_empty":                            # no product count at all: the sort route with nothing to sort
        n, k, m = 50, 40, 30
        a, b, route = csr(n, k, *empty, np.zeros(0, dtype)), rand(k, m), "sort32"
    elif name == "b_empty":
        n, k, m = 50, 40, 30
        a, b, route = rand(n, k), csr(k, m, *empty, np.zeros(0, dtype)), "small_hash"
    elif name == "dead_rows":                        # every entry of A meets an empty row of B
        n, k, m = 60, 40, 30
        bb = rand(20, m)
        b = (np.concatenate([np.zeros(20, np.uint64), bb[0]]), bb[1], bb[2])
        a, route = rand(n, k, 0, 20), "small_hash"
    elif name == "one_by_one":
        n = k = m = 1
        a = csr(1, 1, [0], [0], np.array([3.0], dtype))
        b = csr(1, 1, [0], [0], np.array([-0.5], dtype))
        route = "n_by_1"
    else:                                            # x_empty: A times an empty k x 1 X
        n, k, m = 300, 200, 1
        a, b, route = rand(n, k), csr(k, 1, *empty, np.zeros(0, dtype)), "n_by_1"
    expect = {"route": route}
    if name != "one_by_one":
        expect["out_nnz"] = 0
    return MulCase(n, k, m, a, b, expect, "mirror")


MUL_CASES = {
    "grid_stride_small": lambda s, d: grid_stride_case(s, d, "small"),
    "grid_stride_large": lambda s, d: grid_stride_case(s, d, "large"),
    "router_stride_heavy_last": lambda s, d: router_case(s, d, "last"),
    "router_stride_heavy_first": lambda s, d: router_case(s, d, "first"),
    **{f"boundary_{p}_{w}": (lambda s, d, p=p, w=w: boundary_case(d, p, w))
       for p in (128, 129, 1024, 1025) for w in ("long", "many")},
    "key_bits_32": lambda s, d: key_width_case(d, 65536),
    "key_bits_64": lambda s, d: key_width_case(d, 65537),
    "probe_wrap_small": lambda s, d: probe_case(d, "small"),
    "probe_wrap_large": lambda s, d: probe_case(d, "large"),
    **{f"values_{r}": (lambda s, d, r=r: values_case(d, r)) for r in ("small_hash", "large_hash", "sort32", "n_by_1")},
    **{f"degenerate_{x}": (lambda s, d, x=x: degenerate_case(d, x))
       for x in ("a_empty", "b_empty", "dead_rows", "one_by_one", "x_empty")},
}


# ------------------------------------------------------------------ add / sub cases
AddsubCase = namedtuple("AddsubCase", "n m a b expect")       # n segments (rows of a CSR) over m; CSR arrays


def addsub_specials(dtype):
    """(a, b) pairs stored in both operands, then values stored only in A, then only in B."""
    x, tiny, mx = 1.375, float(np.finfo(dtype).smallest_subnormal), float(np.finfo(dtype).max)
    nan, nneg, inf = payload_nan(dtype), payload_nan(dtype, True), np.inf
    both = [(-0.0, -0.0), (-0.0, 0.0), (0.0, -0.0), (0.0, 0.0), (x, x), (x, -x), (-x, -x), (inf, -inf), (inf, inf),
            (-inf, inf), (inf, 1.0), (nan, 1.0), (1.0, nan), (nneg, nan), (tiny, tiny), (tiny, -tiny), (mx, mx),
            (-mx, mx)]
    single = [nan, nneg, -0.0, 0.0, inf, -inf, tiny, -tiny]
    return both, single


def addsub_case(dtype, name):
    rng = np.random.default_rng(len(name) + 100 * (dtype == np.float32))

    def pattern(n, m, lens_a, lens_b, shared):
        """A's cells, and B's: a `shared` share of A's plus cells of its own."""
        ar, ac = random_entries(rng, np.arange(n), lens_a, 0, m)
        keep = rng.random(len(ar)) < shared
        br, bc = random_entries(rng, np.arange(n), lens_b, 0, m)
        key = np.unique(np.concatenate([ar[keep] * m + ac[keep], br * m + bc]))
        return (ar, ac), (key // m, key % m)

    def pack(n, m, pa, pb, va=None, vb=None):
        va = random_values(rng, len(pa[0]), dtype) if va is None else va
        vb = random_values(rng, len(pb[0]), dtype) if vb is None else vb
        return AddsubCase(n, m, csr(n, m, *pa, va), csr(n, m, *pb, vb), expect)

    expect = {}
    if name == "skewed":                 # short rows, one 5 000-entry row in A and one in B, in other CTAs
        n, m = 20000, 8000
        lens_a, lens_b = rng.integers(0, 7, n), rng.integers(0, 7, n)
        lens_a[[300, 9000]] = 0
        lens_b[9000] = 0
        pa, pb = pattern(n, m, lens_a, lens_b, 0.5)
        pa = concat(pa, (np.full(5000, 300), rng.choice(m, 5000, replace=False)))
        pb = concat(pb, (np.full(5000, 9000), rng.choice(m, 5000, replace=False)))
        expect.update(rows=128, global_ctas=[300 // 128, 9000 // 128])
        return pack(n, m, pa, pb)
    if name == "rows_32":                # mean A + B row length 60: the 32-row plan, every CTA staged
        n, m = 3000, 4000
        pa, pb = pattern(n, m, rng.integers(20, 41, n), rng.integers(15, 26, n), 0.3)
        expect.update(rows=32, global_ctas=[])
        return pack(n, m, pa, pb)
    if name == "all_global":             # mean A + B row length 160: Caps{0, 0}, every CTA merges from global memory
        n, m = 2000, 3000
        pa, pb = pattern(n, m, rng.integers(60, 101, n), rng.integers(50, 81, n), 0.3)
        expect.update(rows=32, caps=(0, 0), global_ctas="all")
        return pack(n, m, pa, pb)
    if name.startswith(("a_dense", "b_dense")):     # one operand dense, the other without entries
        n, m = (2003, 20) if name.endswith("staged") else (301, 200)
        full = (np.repeat(np.arange(n), m), np.tile(np.arange(m), n))
        none = (np.array([], np.int64), np.array([], np.int64))
        pa, pb = (full, none) if name.startswith("a_dense") else (none, full)
        if name.endswith("staged"):
            expect.update(rows=128, global_ctas=[])
        else:
            expect.update(caps=(0, 0), global_ctas="all")
        return pack(n, m, pa, pb)
    if name == "same_pattern":           # identical patterns, half of B's values equal to A's: x - x
        n, m = 5000, 3000
        pa, _ = pattern(n, m, rng.integers(0, 17, n), np.zeros(n, np.int64), 0.0)
        va = random_values(rng, len(pa[0]), dtype)
        vb = np.where(rng.random(len(va)) < 0.5, va, random_values(rng, len(va), dtype)).astype(dtype)
        expect.update(rows=128, global_ctas=[])
        return pack(n, m, pa, pa, va, vb)
    # specials_staged / specials_global: the special values in rows 10 and 11 (CTA 0); a 5 000-entry row of A
    # makes CTA 0 merge from global memory (row 5) or leaves it staged (row 900, CTA 7)
    n, m = 1000, 6000
    lens = rng.integers(0, 7, n)
    lens[[5, 10, 11, 900]] = 0
    pa, pb = pattern(n, m, lens, lens, 0.5)
    heavy = 5 if name == "specials_global" else 900
    pa = concat(pa, (np.full(5000, heavy), np.arange(5000)))
    both, single = addsub_specials(dtype)
    nb, ns = len(both), len(single)
    va = [random_values(rng, len(pa[0]), dtype)]
    vb = [random_values(rng, len(pb[0]), dtype)]
    for row, pairs in ((10, both), (11, [(y, x) for x, y in both])):
        cols = np.arange(nb)
        pa, pb = concat(pa, (np.full(nb, row), cols)), concat(pb, (np.full(nb, row), cols))
        va.append(np.array([x for x, _ in pairs], dtype))
        vb.append(np.array([y for _, y in pairs], dtype))
        pa = concat(pa, (np.full(ns, row), nb + np.arange(ns)))
        va.append(np.array(single, dtype))
        pb = concat(pb, (np.full(ns, row), nb + ns + np.arange(ns)))
        vb.append(np.array(single, dtype))
    expect.update(rows=128, global_ctas=[0] if name == "specials_global" else [900 // 128])
    return pack(n, m, pa, pb, np.concatenate(va), np.concatenate(vb))


ADDSUB_CASES = ["skewed", "rows_32", "all_global", "a_dense_b_empty_staged", "b_dense_a_empty_staged",
                "a_dense_b_empty_global", "b_dense_a_empty_global", "same_pattern", "specials_staged",
                "specials_global"]


def check_addsub_claims(case, what):
    plan = addsub_plan(case.a[0], case.b[0])
    e = case.expect
    assert case.n % plan.rows, f"{what}: the segment count is a multiple of the CTA's rows"
    if "rows" in e:
        assert plan.rows == e["rows"], f"{what}: {plan.rows} rows per CTA"
    if "caps" in e:
        assert (plan.cap_a, plan.cap_b) == e["caps"], f"{what}: caps {(plan.cap_a, plan.cap_b)}"
    else:
        assert plan.cap_a and plan.cap_b, f"{what}: Caps{{0, 0}}"
    glob = np.flatnonzero(~plan.staged).tolist()
    want = list(range(len(plan.staged))) if e["global_ctas"] == "all" else e["global_ctas"]
    assert glob == want, f"{what}: CTAs on the global-memory merge {glob[:8]}, built for {want[:8]}"
    return plan


def cell_keys(ptr, ind, m):
    rows = np.repeat(np.arange(len(ptr) - 1, dtype=np.int64), np.diff(np.asarray(ptr, np.int64)))
    return rows * m + np.asarray(ind, np.int64)


# ------------------------------------------------------------------ CPU: the cases claim their routes
def test_cases_claim_their_routes():
    """Every case at 148 SMs takes the route it was built for, with its stride, probing and plan conditions;
    the value cases' detectors are what they claim to be."""
    for dtype in DTYPES:
        for name, build in MUL_CASES.items():
            check_mul_claims(build(B200_SMS, dtype), B200_SMS, dtype, f"{name} {np.dtype(dtype)}")
        for name in ADDSUB_CASES:
            check_addsub_claims(addsub_case(dtype, name), f"{name} {np.dtype(dtype)}")
        # the fused multiply-add detector: exactly c + a*a != 0, yet 0 with the product rounded first
        from fractions import Fraction
        c, a = fma_pair(dtype)
        exact = Fraction(c) + Fraction(a) ** 2
        assert exact == Fraction(2) ** (-60 if dtype == np.float64 else -26)
        t = np.dtype(dtype).type
        assert t(t(c) * t(1)) + t(t(a) * t(a)) == 0
        # the oracle's side of the value rows (column 0 of each row, in order)
        want = orc.csr_mul(*next(values_case(dtype, "small_hash").forms())[3])
        v = want[2]
        assert v[0] == 0 and not np.signbit(v[0])                       # rounded product, then the add
        assert v[1] == 0                                                 # ascending k
        assert v[2] == 0 and np.signbit(v[2]) and np.signbit(v[5])       # -0.0 copied; underflow to -0.0
        assert 0 < v[6] < np.finfo(dtype).tiny                           # subnormal product
    # the mirrors' rules at their edges
    assert [bits_for(x) for x in (0, 1, 2, 65536, 65537)] == [0, 0, 1, 16, 17]
    assert hs_hash(np.array([0, 1]), 8).tolist() == [0, 2654435761 >> 24]
    assert addsub_plan(np.array([0, 0], np.uint64), np.array([0, 0], np.uint64)).staged.tolist() == [True]


# ------------------------------------------------------------------ GPU
def arrays(m):
    if m._FORMAT == 0:
        return m.rowptr(), m.colind(), m.values()
    return m.colptr(), m.rowind(), m.values()


def bits(v):
    v = np.ascontiguousarray(v)
    return v.view(np.uint32 if v.dtype == np.float32 else np.uint64)


def same_values(got, want, what, arithmetic=None):
    """Pointers and indices equal, values bit for bit, with one exception: where the oracle holds a NaN that an
    add or a multiply produced (`arithmetic`, default every entry), any NaN will do.  The GPU returns the
    canonical NaN where x86 propagates an operand's payload (DESIGN.md, "NaN caveat"); NaNs that are only copied
    or sign-flipped keep their payload and are compared bit for bit."""
    gp, gi, gv = got
    wp, wi, wv = want
    assert gp.dtype == np.uint64 and gi.dtype == np.uint64
    assert np.array_equal(gp, np.asarray(wp, np.uint64)), f"{what}: ptr differs"
    assert np.array_equal(gi, np.asarray(wi, np.uint64)), f"{what}: ind differs"
    wv = np.asarray(wv, gv.dtype)
    free = np.isnan(wv) & (np.ones(len(wv), bool) if arithmetic is None else arithmetic)
    assert np.isnan(gv[free]).all(), f"{what}: a NaN is missing"
    bad = np.flatnonzero(bits(gv)[~free] != bits(wv)[~free])
    assert not len(bad), f"{what}: values differ (bitwise) at {np.flatnonzero(~free)[bad][:5]}: " \
                         f"{gv[~free][bad][:5]} != {wv[~free][bad][:5]}"


@pytest.fixture(scope="module")
def sms():
    torch = pytest.importorskip("torch")
    return torch.cuda.get_device_properties(0).multi_processor_count


def device(M):
    import spalinalg_b200 as sp
    cls = sp.CsrMatrix if M.fmt == "csr" else sp.CscMatrix
    return cls.new(M.nrows, M.ncols, M.ptr, M.ind, M.val)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
@pytest.mark.parametrize("name", list(MUL_CASES))
def test_mul_route(sms, dtype, name):
    case = MUL_CASES[name](sms, dtype)
    check_mul_claims(case, sms, dtype, name)
    for label, A, B, args in case.forms():
        got = device(A) * device(B)
        assert got.shape() == (A.nrows, B.ncols)
        same_values(arrays(got), orc.csr_mul(*args), f"{name} [{label}]")


def addsub_operands(case, fmt):
    """The same arrays as a CSR (rows = segments) or a CSC (columns = segments) pair."""
    shape = (case.n, case.m) if fmt == "csr" else (case.m, case.n)
    return device(Mat(*shape, fmt, *case.a)), device(Mat(*shape, fmt, *case.b))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
@pytest.mark.parametrize("name", ADDSUB_CASES)
def test_addsub_route(dtype, name):
    case = addsub_case(dtype, name)
    check_addsub_claims(case, name)
    ka, kb = cell_keys(case.a[0], case.a[1], case.m), cell_keys(case.b[0], case.b[1], case.m)
    for fmt in ("csr", "csc"):
        A, B = addsub_operands(case, fmt)
        for sub in (0, 1):
            want = orc.addsub(sub, case.n, case.m, case.a, case.b)
            kc = cell_keys(want[0], want[1], case.m)
            both = np.isin(kc, ka) & np.isin(kc, kb)
            same_values(arrays(A - B if sub else A + B), want, f"{name} {fmt} {'-' if sub else '+'}", both)


# representative cases whose launches the profiler records: mul cases by name, add/sub cases by name
PROFILED_MUL = ["grid_stride_small", "grid_stride_large", "router_stride_heavy_last", "boundary_1025_many",
                "key_bits_32", "key_bits_64", "values_n_by_1"]
PROFILED_ADDSUB = ["skewed", "rows_32", "all_global"]
KERNEL = re.compile(r"(\w+)<([^<>]*)>")


def observed_mul(kernels):
    """Route, hash grid / block, router grid of one product from its kernel launches (name, grid, block)."""
    seen = {"router_grid": None, "hash": None}
    route = None
    for name, grid, block, _ in kernels:
        m = KERNEL.search(name)
        fn, targs = (m.group(1), m.group(2)) if m else (name, "")
        if "row_products_kernel" in name:
            seen["router_grid"] = grid
        elif fn == "spgemm_hash_kernel" and ", true," in targs:
            route = {"8": "small_hash", "11": "large_hash"}[targs.split(",")[2].strip()]
            seen["hash"] = (grid, block)
        elif fn == "expand_kernel" and route is None:
            route = "sort64" if "long" in targs else "sort32"
        elif "rs_scatter_kernel" in name:
            seen["sorted"] = True
    if route in ("sort32", "sort64") and not seen.get("sorted"):
        route = "n_by_1" if route == "sort32" else "n_by_1 with 64-bit keys"
    return route, seen


@pytest.mark.gpu
def test_mirrors_agree_with_the_launched_kernels(sms, dtype=np.float64):
    """The kernels each representative case launches, their grids, blocks and shared memory (a torch.profiler
    trace of the library's launches) are those the mirrors predict: the route, the hash and router grids at
    this device's SM count, the add/sub plan's rows per CTA and stage size."""
    torch = pytest.importorskip("torch")
    from torch.profiler import ProfilerActivity, profile
    ops = []
    for name in PROFILED_MUL:
        case = MUL_CASES[name](sms, dtype)
        _, A, B, _ = next(case.forms())
        ops.append(("mul", name, mul_route(A, B, sms, dtype), device(A), device(B)))
    for name in PROFILED_ADDSUB:
        case = addsub_case(dtype, name)
        ops.append(("add", name, addsub_plan(case.a[0], case.b[0]), *addsub_operands(case, "csr")))
    torch.cuda.synchronize()
    results = []
    with tempfile.TemporaryDirectory() as tmp:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for kind, _, _, A, B in ops:
                results.append(A * B if kind == "mul" else A + B)
            torch.cuda.synchronize()
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    kernels = sorted((e["ts"], e["name"], e["args"].get("grid"), e["args"].get("block"), e["args"].get("shared memory"))
                     for e in events if e.get("cat") == "kernel")
    # one segment per operation: a product starts with product_count_kernel, a sum with the symbolic union pass
    starts = [i for i, k in enumerate(kernels)
              if "product_count_kernel" in k[1] or re.search(r"union_block_kernel<\w+, false, false>", k[1])]
    assert len(starts) == len(ops), [k[1][:60] for k in kernels]
    for (kind, name, mirror, _, _), lo, hi in zip(ops, starts, starts[1:] + [len(kernels)]):
        seg = [k[1:] for k in kernels[lo:hi]]
        if kind == "mul":
            route, seen = observed_mul(seg)
            assert route == mirror.route, f"{name}: launched {route}, mirror {mirror.route}"
            assert seen["router_grid"] == [mirror.router_grid, 1, 1], f"{name}: router grid {seen['router_grid']}"
            if seen["hash"]:
                assert seen["hash"] == ([mirror.hash_grid, 1, 1], [32 * mirror.warps, 1, 1]), f"{name}: {seen['hash']}"
        else:
            num = [k for k in seg if re.search(r"union_block_kernel<\w+, false, true>", k[0])]
            assert len(num) == 1, name
            _, grid, block, smem = num[0]
            assert block == [mirror.rows, 1, 1] and grid[0] == len(mirror.staged), f"{name}: {grid} x {block}"
            assert smem == mirror.smem_numeric, f"{name}: {smem} B of shared memory, mirror {mirror.smem_numeric}"
