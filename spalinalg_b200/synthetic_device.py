"""Device-side (torch, plumbing only) generators of BASELINE.json's synthetic matrices
(SURVEY.md 8d) for benchmarks and full-size tests.  Deterministic from their seeds."""
from __future__ import annotations


def stencil_device(torch, offsets_3d, m, diag, off, dtype):
    """Row-major CSR of a stencil on an m^3 (or m^2) grid, built on the device."""
    dev = "cuda"
    dims = len(offsets_3d[0])
    n = m ** dims
    r = torch.arange(n, device=dev, dtype=torch.int64)
    coords = []
    rem = r
    for d in range(dims):
        coords.append(rem // (m ** (dims - 1 - d)))
        rem = rem % (m ** (dims - 1 - d))
    offs = sorted(offsets_3d, key=lambda o: sum(o[d] * m ** (dims - 1 - d) for d in range(dims)))
    cols, masks, vals = [], [], []
    for o in offs:
        ok = torch.ones(n, device=dev, dtype=torch.bool)
        lin = torch.zeros(n, device=dev, dtype=torch.int64)
        for d in range(dims):
            cd = coords[d] + o[d]
            ok &= (cd >= 0) & (cd < m)
            lin += cd * (m ** (dims - 1 - d))
        cols.append(lin)
        masks.append(ok)
        vals.append(torch.full((n,), diag if all(x == 0 for x in o) else off, device=dev, dtype=dtype))
    mask = torch.stack(masks, 1)
    colind = torch.stack(cols, 1)[mask].to(torch.int32)
    values = torch.stack(vals, 1)[mask]
    rowptr = torch.zeros(n + 1, device=dev, dtype=torch.int64)
    rowptr[1:] = torch.cumsum(mask.sum(1), 0)
    return n, rowptr.to(torch.int32), colind, values


def banded_device(torch, n, r0, r1, offsets, dtype, chunk=1 << 24):
    """Rows [r0, r1) of the banded matrix of config 5, global column indices, on the device."""
    dev = "cuda"
    offs = sorted(offsets)
    ptr_parts, col_parts, val_parts = [], [], []
    base = 0
    for s in range(r0, r1, chunk):
        e = min(r1, s + chunk)
        i = torch.arange(s, e, device=dev, dtype=torch.int64)
        cols = torch.stack([i + d for d in offs], 1)
        mask = (cols >= 0) & (cols < n)
        vals = torch.stack([1.0 / (1 + abs(d)) + (i % 7).to(dtype) * 1e-3 for d in offs], 1)
        cnt = torch.cumsum(mask.sum(1), 0)
        ptr_parts.append(cnt + base)
        base = int(ptr_parts[-1][-1].item())
        col_parts.append(cols[mask].to(torch.int32))
        val_parts.append(vals[mask].to(dtype))
        del cols, mask, vals, i
    rowptr = torch.cat([torch.zeros(1, device=dev, dtype=torch.int64)] + ptr_parts).to(torch.int32)
    return rowptr, torch.cat(col_parts), torch.cat(val_parts)


def band_value(torch, i, d):
    """A[i, i + d] of scrambled_band_coo_device, f64 (int64 tensors i, d)."""
    return 1.0 / (1.0 + d.abs().double()) + (i % 7).double() * 1e-3


def scrambled_band_coo_device(torch, n, half, dtype, spare=0, a=1_000_000_007, b=12_345, chunk=1 << 25):
    """Triplets of the n x n band with diagonals -half..half (A[i, i+d] = band_value), one per cell, in an
    order scrambled by the bijection e = (a p + b) mod (2 half + 1) n of the slot index (a coprime to the
    slot count): slot e is cell (e // (2 half + 1), e % (2 half + 1) - half), slots outside the matrix are
    skipped.  Every stretch of the list gathers from the whole matrix.  int32 row, int32 col, values, with
    `spare` unset slots at the end for the caller.  Returns (row, col, val, number of band cells)."""
    import math
    w = 2 * half + 1
    slots = w * n
    assert math.gcd(a, slots) == 1 and a * slots < 2 ** 63
    cells = w * n - half * (half + 1)
    row = torch.empty(cells + spare, device="cuda", dtype=torch.int32)
    col = torch.empty(cells + spare, device="cuda", dtype=torch.int32)
    val = torch.empty(cells + spare, device="cuda", dtype=dtype)
    pos = 0
    for s in range(0, slots, chunk):
        p = torch.arange(s, min(slots, s + chunk), device="cuda", dtype=torch.int64)
        e = (p * a + b) % slots
        i, d = e // w, e % w - half
        j = i + d
        keep = (j >= 0) & (j < n)
        i, d, j = i[keep], d[keep], j[keep]
        k = i.numel()
        row[pos:pos + k] = i.to(torch.int32)
        col[pos:pos + k] = j.to(torch.int32)
        val[pos:pos + k] = band_value(torch, i, d).to(dtype)
        pos += k
        del p, e, i, d, j, keep
    assert pos == cells
    return row, col, val, cells




def device_view(torch, ptr: int, count: int, dtype):
    """torch tensor aliasing `count` elements of raw device memory at `ptr` (no copy)."""
    import numpy as np
    typestr = {torch.int32: "<i4", torch.float32: "<f4", torch.float64: "<f8", torch.int64: "<i8"}[dtype]

    class _Raw:
        __cuda_array_interface__ = {"shape": (int(count),), "typestr": typestr, "data": (int(ptr), False),
                                    "version": 2}
    return torch.as_tensor(_Raw(), device="cuda")


def random_uniform_coo_device(torch, n, per_row, n_extra, dtype, seed=1):
    """Config 3: per row `per_row` iid uniform columns (natural collisions kept), values in [-1,1);
    then n_extra copies of uniformly chosen existing cells with fresh values, of which 1 % are exact
    negations of the chosen entry and 1 % hit cells that were already duplicated (multiplicity >= 3);
    the whole list shuffled.  Returns int32 row, int32 col, values (device)."""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    base = n * per_row
    rows = torch.arange(n, device="cuda", dtype=torch.int32).repeat_interleave(per_row)
    cols = torch.randint(0, n, (base,), device="cuda", dtype=torch.int32, generator=g)
    vals = (torch.rand(base, device="cuda", dtype=dtype, generator=g) * 2 - 1)
    if n_extra:
        idx = torch.randint(0, base, (n_extra,), device="cuda", generator=g)
        k3 = max(1, n_extra // 100)
        idx[-k3:] = idx[:k3]                      # third copies of cells duplicated above
        ev = (torch.rand(n_extra, device="cuda", dtype=dtype, generator=g) * 2 - 1)
        kneg = max(1, n_extra // 100)
        ev[k3:k3 + kneg] = -vals[idx[k3:k3 + kneg]]   # exact cancellations (zero drop)
        rows = torch.cat([rows, rows[idx]])
        cols = torch.cat([cols, cols[idx]])
        vals = torch.cat([vals, ev])
    g.manual_seed(seed + 1)
    perm = torch.randperm(rows.numel(), device="cuda", generator=g)
    return rows[perm].contiguous(), cols[perm].contiguous(), vals[perm].contiguous()


def rmat_coo_device(torch, scale, edge_factor, dtype, seed=3, abcd=(0.57, 0.19, 0.19, 0.05), chunk=1 << 25):
    """Config 4: R-MAT edges (no vertex permutation), values in [-1,1).  int32 row/col (device)."""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    n_edges = edge_factor << scale
    a, b, c, _ = abcd
    rows_p, cols_p = [], []
    for s in range(0, n_edges, chunk):
        m = min(chunk, n_edges - s)
        r = torch.zeros(m, device="cuda", dtype=torch.int32)
        cc = torch.zeros(m, device="cuda", dtype=torch.int32)
        for _level in range(scale):
            u = torch.rand(m, device="cuda", generator=g)
            rbit = (u >= a + b).to(torch.int32)                       # quadrants c, d: lower half
            cbit = (((u >= a) & (u < a + b)) | (u >= a + b + c)).to(torch.int32)   # b, d: right half
            r = (r << 1) | rbit
            cc = (cc << 1) | cbit
        rows_p.append(r)
        cols_p.append(cc)
    rows, cols = torch.cat(rows_p), torch.cat(cols_p)
    vals = torch.rand(n_edges, device="cuda", dtype=dtype, generator=g) * 2 - 1
    return rows, cols, vals
