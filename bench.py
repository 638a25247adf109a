#!/usr/bin/env python
"""bench.py — the hot path of spalinalg on B200, BASELINE.json's metric.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME]
                  [--dump-outputs DIR]

ONE workload at every N: config 5 of BASELINE.json (banded, offsets -4..+4, n = 1e8, 9e8 stored
entries, f64; 12.4 GB algorithmic per product, inputs far larger than L2, so no flush is needed).
N = 1 runs it on one GPU; N > 1 row-shards the SAME matrix over the ranks (fixed total work: strong
scaling).  A step is one SpMV y = A x over the whole matrix.  At N > 1 x stays in its owners'
peer-visible memory; every step runs ONE small kernel that is the device-side barrier (it orders an
iteration's writes of x before the peers' reads) and then copies the few halo values a shard needs
from its neighbours over NVLink next to the own slice, and the SpMV reads one local array.
`value` = algorithmic bytes (nnz*(4+V) + (ncols+nrows)*V, SURVEY.md 8d) of the whole job per second
of the slowest rank, device-timed.  `e2e` = the same metric through the reference-facing call
`&A * &x` with HOST vectors: A is a constructed CsrMatrix (device resident, as the reference's is
host resident), every step moves x from pinned host memory to the device, runs the product and moves
y back (spl_spmv_host at N = 1, spl_spmv_peer_host on every rank at N > 1).
`parity_check`: before anything is timed, a small problem sharded over the same N ranks is compared
with the CPU oracle (assembly and add bit-exact, SpMV within 1e-12, and a 50-step iteration whose x
changes every step with one rank delayed).  The line also carries, as named extras, configs 1-4
(SpMV, assembly, conversions) and the add of config 5 at N = 1, the sharded forms at N > 1,
`roofline`, `cpu_baseline` and `clocks`.

--impl reference times the reference's only SpMV route (`&A * &X`, X n x 1: three counting-sort
transposes + Gustavson) on the host: the oracle's line-by-line port (the reference is Rust; no rustc
in this image: cpu_baseline.kind = "port"), one core because the reference is single-threaded, on a
bounded sample of the same workload (the same banded matrix at n = 1e7).

--dump-outputs DIR writes the product of the last timed step, y, as DIR/y.npy (f64): every row while y
has at most DUMP_ROWS of them, else a fixed sample (the first and last 4096 rows and a seeded uniform
draw), whose row numbers go to DIR/y_rows.npy.  Matrix and x are deterministic, so two builds run with
the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

I_BYTES = 4   # device index width used for the algorithmic byte count (SURVEY.md 8d)

WORKLOADS = {
    # name: (family, size, cpu sample size)
    "banded9_1e8_f64": ("banded", 10 ** 8, 10 ** 7),
    "banded9_1e7_f64": ("banded", 10 ** 7, 10 ** 7),
    "stencil27_128_f64": ("stencil27", 128, 64),
    "laplace2d_1024_f64": ("laplace2d", 1024, 1024),
}
DEFAULT_WORKLOAD = "banded9_1e8_f64"


def spmv_bytes(nnz, nrows, ncols, v):
    return nnz * (I_BYTES + v) + (ncols + nrows) * v


def workload_shape(wl):
    """(nrows, nnz) of a workload without building it."""
    fam, size, _ = WORKLOADS[wl]
    if fam == "banded":
        return size, 9 * size - 20
    if fam == "stencil27":
        return size ** 3, (3 * size - 2) ** 3
    return size * size, 5 * size * size - 4 * size


def config_of(wl):
    """The `config` object, identical in both arms (the reference arm samples it: cpu_baseline.sample)."""
    n, nnz = workload_shape(wl)
    b = spmv_bytes(nnz, n, n, 8)
    return {"workload": wl, "nrows": n, "nnz": nnz, "algorithmic_bytes": b,
            "l2": "inputs larger than L2 (no flush)" if b > 2 * 126e6 else "rotating copies of (A, x, y) larger than L2"}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------- CPU side
def cpu_sample(wl):
    """Bounded sample of the workload for the CPU legs: same family, reference layout (usize indices)."""
    from spalinalg_b200 import synthetic as syn
    fam, _, m = WORKLOADS[wl]
    if fam == "banded":
        n = m
        r, c, v = syn.banded(n, range(-4, 5))
        x = np.sin(np.arange(n) * 1e-3)
        what = f"banded9 n={n}"
    elif fam == "stencil27":
        n = m ** 3
        r, c, v = syn.stencil_27(m)
        x = 1.0 / (1.0 + (np.arange(n) % 97))
        what = f"27-point stencil {m}^3"
    else:
        n = m * m
        r, c, v = syn.laplacian_2d(m)
        order = np.lexsort((c, r))
        r, c, v = r[order], c[order], v[order]
        x = 1.0 / (1.0 + (np.arange(n) % 97))
        what = f"2-D Laplacian {m}^2"
    ptr, ind, val = syn.csr_from_sorted_triplets(n, r, c, v)
    return n, ptr, ind, val, x, f"{what} (n={n}, nnz={len(val)}), f64, X n x 1"


def cpu_reference_step(n, ptr, ind, val, x):
    """The reference's only SpMV route: &A * &X with X n x 1 (src/csr/ops/mul.rs:5-60)."""
    import oracle as orc
    xs = (np.arange(n + 1, dtype=np.uint64), np.zeros(n, np.uint64), x)
    t0 = time.perf_counter()
    orc.csr_mul(n, n, 1, (ptr, ind, val), xs, cap=n)      # n x 1 result: at most n entries
    return time.perf_counter() - t0


def cpu_assembly_baseline():
    """COO->CSR on the CPU: the oracle port of From<&CooMatrix> (src/csr/conv/coo.rs:3-116) on a 512^2
    Laplacian with the triplets shuffled like the device run's.  One core: the reference is
    single-threaded."""
    import oracle as orc
    from spalinalg_b200 import synthetic as syn
    ar, ac, av = syn.laplacian_2d(512)
    perm = np.random.default_rng(42).permutation(len(av))
    trip = orc.make_triplets(ar[perm], ac[perm], av[perm])
    orc.compress_from_coo(512 * 512, 512 * 512, trip, "row")
    t0 = time.perf_counter()
    for _ in range(3):
        orc.compress_from_coo(512 * 512, 512 * 512, trip, "row")
    asm_s = (time.perf_counter() - t0) / 3
    return {"value": len(av) / asm_s / 1e6, "unit": "Mnnz/s", "cores": 1,
            "sample": f"2-D Laplacian 512^2, {len(av)} shuffled triplets, f64, COO->CSR"}


def cpu_mul_baseline():
    """A * A on the CPU: the oracle port of impl Mul for &CsrMatrix (src/csr/ops/mul.rs:5-60: three
    transposes + Gustavson) on a 256^2 Laplacian, one core."""
    import oracle as orc
    from spalinalg_b200 import synthetic as syn
    r, c, v = syn.laplacian_2d(256)
    nn = 256 * 256
    a = orc.compress_from_coo(nn, nn, orc.make_triplets(r, c, v), "row")
    out = orc.csr_mul(nn, nn, nn, a, a)
    t0 = time.perf_counter()
    for _ in range(3):
        out = orc.csr_mul(nn, nn, nn, a, a)
    s_ = (time.perf_counter() - t0) / 3
    return {"value": len(out[1]) / s_ / 1e6, "unit": "Mnnz_out/s", "cores": 1,
            "sample": f"A * A, 2-D Laplacian 256^2, nnz(C)={len(out[1])}, f64"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = workload_name(args)
    n, ptr, ind, val, x, sample = cpu_sample(wl)
    b = spmv_bytes(len(val), n, n, 8)
    for _ in range(args.warmup):
        cpu_reference_step(n, ptr, ind, val, x)
    t = [cpu_reference_step(n, ptr, ind, val, x) for _ in range(args.steps)]
    per = sum(t) / len(t)
    value = b / per / 1e9
    line = {
        "impl": "reference", "metric": "spmv_algorithmic_bandwidth", "value": value, "unit": "GB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": per * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_of(wl),
        "cpu_baseline": {"value": value, "unit": "GB/s", "cores": 1, "kind": "port", "sample": sample,
                         "host_cores": os.cpu_count(),
                         "what": "oracle port of the reference's `&A * &X` route; a rate, so the sample's GB/s stands "
                                 "for the workload's; one core: the reference is single-threaded"},
        "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_name(args):
    return DEFAULT_WORKLOAD if args.workload == "auto" else args.workload


# ------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "50", "-i", str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
                for k, nme in enumerate(names):
                    if r[4 + k].strip().lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                continue
        # "under load": drop samples taken while the GPU was idling (power well below the peak seen)
        if power:
            thr = 0.6 * max(power)
            load = [s for s, p in zip(sm, power) if p >= thr] or sm
        else:
            load = sm
        return {"sm_mhz": statistics.median(load) if load else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "samples_under_load": len(load),
                "power_w_max": max(power) if power else None}


KERNEL_NAMES = {1: "vector", 2: "merge", 3: "split", 4: "sliced", 5: "stream", 6: "scatter"}


# ------------------------------------------------------------------------------- our arm
def build_workload(torch, sp, ctx, wl, rank, world):
    """Rows [r0, r1) of the workload on this rank's device (global column indices)."""
    from spalinalg_b200 import sharding
    from spalinalg_b200.synthetic_device import banded_device, stencil_device
    f64 = torch.float64
    fam, size, _ = WORKLOADS[wl]
    if fam == "banded":
        n = size
        r0, r1 = sharding.row_partition(n, world, rank)
        rowptr, colind, values = banded_device(torch, n, r0, r1, range(-4, 5), f64)
        halo = 4
    else:
        if fam == "stencil27":
            offs = [(a, b, c) for a in (-1, 0, 1) for b in (-1, 0, 1) for c in (-1, 0, 1)]
            n, rowptr, colind, values = stencil_device(torch, offs, size, 26.0, -1.0, f64)
            halo = size * size + size + 1
        else:
            offs = [(0, 0), (-1, 0), (1, 0), (0, -1), (0, 1)]
            n, rowptr, colind, values = stencil_device(torch, offs, size, 4.0, -1.0, f64)
            halo = size
        r0, r1 = sharding.row_partition(n, world, rank)
        if world > 1:                       # keep this rank's rows of the stencil
            lo, hi = int(rowptr[r0].item()), int(rowptr[r1].item())
            rowptr = (rowptr[r0:r1 + 1] - rowptr[r0]).contiguous()
            colind, values = colind[lo:hi].contiguous(), values[lo:hi].contiguous()
    A = sp.CsrMatrix.from_device_arrays(r1 - r0, n, int(colind.numel()), rowptr.data_ptr(), colind.data_ptr(),
                                        values.data_ptr(), np.float64, validate=True, ctx=ctx)
    return A, n, r0, r1, halo


def x_values(torch, wl, lo, hi):
    idx = torch.arange(lo, hi, device="cuda", dtype=torch.int64)
    if wl.startswith("banded"):
        return torch.sin(idx.to(torch.float64) * 1e-3)
    return (1.0 / (1.0 + (idx % 97))).to(torch.float64)


DUMP_ROWS = 1 << 21      # rows of y --dump-outputs writes at most: 16 MB of f64 values, 16 MB of row numbers


def dump_rows(n):
    """Rows of y that --dump-outputs writes, ascending: all n while n <= DUMP_ROWS, else the first and last
    4096 rows and a seeded uniform draw, the same in every build and at every rank count."""
    if n <= DUMP_ROWS:
        return np.arange(n)
    edges = np.concatenate([np.arange(4096), np.arange(n - 4096, n)])
    return np.unique(np.concatenate([edges, np.random.default_rng(0).integers(0, n, DUMP_ROWS - edges.size)]))


def last_step_output(torch, dist, y, n, r0, rank, world):
    """(rows, y[rows]) of the whole product, rows = dump_rows(n), gathered bit for bit from the row blocks
    [r0, r1) of sharding.row_partition that the ranks hold."""
    from spalinalg_b200 import sharding
    rows = dump_rows(n)
    bounds = np.searchsorted(rows, [sharding.row_partition(n, world, g)[0] for g in range(world)] + [n])
    counts = np.diff(bounds)
    mine = torch.zeros(int(counts.max()), dtype=y.dtype, device=y.device)
    mine[:counts[rank]] = y[torch.from_numpy(rows[bounds[rank]:bounds[rank + 1]] - r0).to(y.device)]
    parts = [mine]
    if world > 1:
        parts = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(parts, mine)
    return rows, torch.cat([p[:c] for p, c in zip(parts, counts)]).cpu().numpy()


def write_outputs(path, n, rows, y):
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "y.npy"), y)
    if rows.size < n:
        np.save(os.path.join(path, "y_rows.npy"), rows.astype(np.float64))      # exact below 2^53


def parity_check(torch, dist, sp, spd, ctx, rank, world):
    """A small problem sharded over the SAME ranks, against the CPU oracle (the checker, never the thing
    measured): sharded assembly bit-exact, sharded SpMV within 1e-12, sharded add bit-exact, and the
    changing-x iteration over peer memory (one rank delayed every step) bit-exact."""
    import oracle as orc
    from tests.test_dist import make_coo, shard_of, syn_block
    from tests.test_multi_gpu import iterate_against_oracle
    from spalinalg_b200.synthetic_device import device_view
    out = {"world": world}
    n = 20011
    r, c, v = make_coo(n, n, 400000, 123)
    full = orc.compress_from_coo(n, n, orc.make_triplets(r, c, v), "row")
    a, b = syn_block(len(v), world, rank)
    dev = lambda arr, dt: torch.from_numpy(np.ascontiguousarray(arr).astype(dt)).cuda()
    rd, cd, vd = dev(r[a:b], np.int32), dev(c[a:b], np.int32), dev(v[a:b], np.float64)
    if world > 1:
        ex = spd.PeerExchange(ctx, dist)
        D = spd.DistCsrMatrix.from_device_triplets_peer(dist, torch, n, n, rd, cd, vd, ex)
        ex.check()
        ex.close()
        starts = D.starts
        L = D.local
    else:
        L = sp.CsrMatrix.from_device_triplets(n, n, len(v), rd.data_ptr(), cd.data_ptr(), vd.data_ptr(), np.float64, ctx=ctx)
        starts = [0, n]
        D = spd.DistCsrMatrix(L, starts, 0, n, n)
    want = shard_of(full, starts, rank)
    ok_asm = bool(np.array_equal(L.rowptr(), want[0]) and np.array_equal(L.colind(), want[1])
                  and L.values().tobytes() == want[2].tobytes())
    # SpMV on the shard: x in its owners' memory (peer gather) / one buffer at N = 1
    x = np.random.default_rng(9).standard_normal(n)
    yw = orc.csr_spmv(n, *full, x)
    sc = orc.csr_spmv(n, full[0], full[1], np.abs(full[2]), np.abs(x))
    r0, r1 = starts[rank], starts[rank + 1]
    y = torch.zeros(r1 - r0, dtype=torch.float64, device="cuda")
    if world > 1:
        xv = spd.PeerVector(ctx, dist, n, np.float64, starts)
        device_view(torch, xv.local_ptr, r1 - r0, torch.float64).copy_(torch.from_numpy(x[r0:r1]))
        xv.publish()
        D.spmv_peer(xv, y.data_ptr())
        torch.cuda.synchronize()
        xv.check()
        xv.close(dist)
    else:
        xd = torch.from_numpy(x).cuda()
        torch.cuda.synchronize()
        L.spmv_device(xd.data_ptr(), y.data_ptr())
        torch.cuda.synchronize()
    err = np.abs(y.cpu().numpy() - yw[r0:r1])
    ok_spmv = bool(np.all(err <= 1e-12 * sc[r0:r1] + 1e-300))
    # add on the shared partition
    S = D + D
    w = shard_of(orc.addsub(0, n, n, full, full), starts, rank)
    ok_add = bool(np.array_equal(S.local.rowptr(), w[0]) and np.array_equal(S.local.colind(), w[1])
                  and S.local.values().tobytes() == w[2].tobytes())
    ok_iter = None
    if world > 1:
        ok_iter = iterate_against_oracle(orc, spd, sp, ctx, rank, world, iters=50)
    flags = [ok_asm, ok_spmv, ok_add] + ([ok_iter] if ok_iter is not None else [])
    t = torch.tensor([1 if all(flags) else 0] + [1 if f else 0 for f in flags], device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
    res = [bool(int(q)) for q in t.tolist()]
    out.update({"ok": res[0], "assembly_bit_exact": res[1], "spmv_within_1e-12": res[2], "add_bit_exact": res[3],
                "problem": f"random {n} x {n}, {len(v)} triplets with duplicates and cancellations, f64"})
    if ok_iter is not None:
        out["changing_x_iteration_bit_exact"] = res[4]
        out["iteration"] = "x_{t+1} = A x_t, 50 steps, banded n=300007, y written into the unpublished peer buffer, " \
                           "one rank delayed by a spin kernel every step"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto"] + list(WORKLOADS))
    ap.add_argument("--kernel", default="auto")       # auto | vectorN | stream | merge  (N = 1 only)
    ap.add_argument("--no-extras", action="store_true", help="skip secondary metrics / cpu baseline / parity check")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write y of the last timed step as DIR/y.npy (a fixed sample of its rows when "
                                                          "it is large, their numbers in DIR/y_rows.npy)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the device product (--impl ours)")
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import torch.distributed as dist
    import spalinalg_b200 as sp
    from spalinalg_b200 import _capi as capi
    from spalinalg_b200 import dist as spd
    from spalinalg_b200 import synthetic_device

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node N for --gpus N"
    ngpu = world

    # one explicit stream for everything: our kernels, torch's generators, NCCL and the timing
    # events (torch's default stream has handle 0, which the C ABI reads as "create your own")
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = sp.Context(local, stream.cuda_stream)
    sp.set_default_context(ctx)
    lib = ctx._lib
    wl = workload_name(args)
    f64 = torch.float64
    V = 8

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- parity first: the sharded path against the oracle on this many ranks -----------------
    parity = None
    if not args.no_extras:
        parity = parity_check(torch, dist, sp, spd, ctx, rank, world)
        assert parity["ok"], f"parity check against the oracle failed: {parity}"

    # ---- build the workload on the device -------------------------------------------------
    A, n, r0, r1, halo = build_workload(torch, sp, ctx, wl, rank, world)
    nloc = r1 - r0
    nnz_loc = A.nnz()
    cfg = config_of(wl)
    nnz_t = torch.tensor([nnz_loc], device="cuda", dtype=torch.int64)
    if world > 1:
        dist.all_reduce(nnz_t)
    assert int(nnz_t.item()) == cfg["nnz"] and n == cfg["nrows"]
    bytes_total = cfg["algorithmic_bytes"]
    bytes_local = spmv_bytes(nnz_loc, nloc, n if ngpu == 1 else nloc + 2 * min(halo, nloc), V)

    kern, lanes = capi.SPL_SPMV_AUTO, 0
    if args.kernel.startswith("vector"):
        kern, lanes = capi.SPL_SPMV_VECTOR, int(args.kernel[6:] or 0)
    elif args.kernel == "merge":
        kern = capi.SPL_SPMV_MERGE
    elif args.kernel == "stream":
        kern = capi.SPL_SPMV_STREAM

    # x: at N > 1 every rank keeps only its slice, in peer-visible memory mapped by every rank
    xv = dA = x_full = None
    if world > 1:
        starts = spd.partition_starts(n, world)
        dA = spd.DistCsrMatrix(A, starts, rank, n, n)
        widths = dA.halo_widths(dist, torch)          # how far the shards' columns reach into the neighbours
        xv = spd.PeerVector(ctx, dist, n, np.float64, starts, halo=widths)
        for _ in range(2):                            # both halves of the double buffer hold x: the timed
            synthetic_device.device_view(torch, xv.local_ptr, nloc, f64).copy_(x_values(torch, wl, r0, r1))
            xv.publish(halo=True)                     # steps re-read an unchanged x (barrier + halo, no swap)
    else:
        x_full = x_values(torch, wl, 0, n)
    y = torch.zeros(nloc, device="cuda", dtype=f64)

    def local_spmv():
        if world > 1:
            dA.spmv_halo(xv, y.data_ptr())    # own slice + halo: one local array, the unsharded kernels
        else:
            A.spmv_device(x_full.data_ptr(), y.data_ptr(), kern, lanes)

    def step():
        if world > 1:
            xv.barrier_halo()                 # device-side: peers' slices are final, then the halo comes over NVLink
        local_spmv()

    # ---- sanity before timing: the step's result equals the single-buffer vector kernel's --------
    step()
    torch.cuda.synchronize()
    lo, hi = max(0, r0 - halo), min(n, r1 + halo)
    x_chk = torch.zeros(n, device="cuda", dtype=f64)
    x_chk[lo:hi] = x_values(torch, wl, lo, hi)
    y_chk = torch.empty_like(y)
    A.spmv_device(x_chk.data_ptr(), y_chk.data_ptr(), capi.SPL_SPMV_VECTOR, 0)
    torch.cuda.synchronize()
    if xv is not None:
        xv.check()
    assert torch.equal(y, y_chk), "the step's SpMV differs from the single-buffer vector kernel"
    del x_chk, y_chk

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()

    # ---- device-timed steps ----------------------------------------------------------------
    for _ in range(args.warmup):
        step()
    barrier()
    l0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = ctx.launch_count() - l0
    t = torch.tensor([ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_step = ms_total / args.steps
    value = bytes_total / (ms_step * 1e-3) / 1e9
    if xv is not None:
        xv.check()
    dumped = last_step_output(torch, dist, y, n, r0, rank, world) if args.dump_outputs else None

    # SpMV-kernel-only time on this rank (roofline of the dominant kernel)
    barrier()
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k0.record()
    for _ in range(args.steps):
        local_spmv()
    k1.record()
    torch.cuda.synchronize()
    kern_ms = k0.elapsed_time(k1) / args.steps
    peak, peak_src = peaks()
    achieved = bytes_local / (kern_ms * 1e-3) / 1e9
    choice = A.spmv_choice()
    kname = KERNEL_NAMES.get(kern or choice[0], "?")
    traffic, traffic_src = None, None
    try:     # per-launch DRAM bytes of this kernel on this workload from the committed `ncu --set full` capture
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            t_ = json.load(f)[wl]["spmv_" + kname]
            if ngpu == 1:
                traffic = t_["dram_read_bytes"] + t_["dram_write_bytes"]
                traffic_src = t_.get("source")
    except Exception:
        pass

    # ---- e2e through the reference-facing call with HOST vectors ------------------------------
    # A is a constructed CsrMatrix (device resident; the reference's lives in host memory); a step
    # is `&A * &x`: x from pinned host memory, SpMV, y back to pinned host memory.
    e2e_steps = max(3, min(args.steps, 10))
    h_x = x_values(torch, wl, r0, r1).cpu().pin_memory() if world > 1 else x_full.cpu().pin_memory()
    h_y = torch.empty(nloc, dtype=f64).pin_memory()
    h2d = h_x.numel() * 8
    d2h = h_y.numel() * 8

    def e2e_step():
        if world == 1:
            ctx.check(lib.spl_spmv_host(ctx._h, A._h, C.c_void_p(h_x.data_ptr()), C.c_void_p(h_y.data_ptr())))
        else:
            dA.matvec_host(xv, h_x.data_ptr(), h_y.data_ptr())

    e2e_step()
    assert torch.equal(h_y, y.cpu()), "e2e result differs from the device-resident result"
    e2e_step()
    barrier()
    e2e_l0 = ctx.launch_count()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    e2e_launches = (ctx.launch_count() - e2e_l0) // e2e_steps
    t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    e2e_value = bytes_total / e2e_s / 1e9
    del h_x, h_y

    # keep the device busy long enough for a few clock samples if the timed region was short
    clk = None
    if rank == 0:
        t_end = time.perf_counter() + max(0.0, 0.6 - ms_total * 2e-3)
        while time.perf_counter() < t_end:
            for _ in range(10):
                local_spmv()
            torch.cuda.synchronize()
        clk = clocks.stop()
    barrier()

    # ---- secondary metrics of the path ------------------------------------------------------
    extras = {}
    cpu = None
    if ngpu > 1 and not args.no_extras:
        extras = sharded_extras(torch, dist, sp, spd, ctx, A, n, r0, r1, rank, world)
    if rank == 0 and ngpu == 1 and not args.no_extras:
        x_full = None
        extras = secondary_metrics(torch, sp, ctx, A, wl)
        sn, sptr, sind, sval, sx, sample = cpu_sample(wl)
        sb = spmv_bytes(len(sval), sn, sn, 8)
        cpu_reference_step(sn, sptr, sind, sval, sx)
        ts = [cpu_reference_step(sn, sptr, sind, sval, sx) for _ in range(3)]
        import oracle as orc
        t0 = time.perf_counter()
        for _ in range(3):
            orc.csr_spmv(sn, sptr, sind, sval, sx)
        rowdot = (time.perf_counter() - t0) / 3
        cpu = {"value": sb / statistics.median(ts) / 1e9, "unit": "GB/s", "cores": 1,
               "assembly": cpu_assembly_baseline(), "mul": cpu_mul_baseline(),
               "kind": "port", "host_cores": os.cpu_count(),
               "sample": sample + "; reference route &A * &X (3 transposes + Gustavson), 3 reps median",
               "rowdot_value": sb / rowdot / 1e9}

    if rank == 0:
        line = {
            "metric": "spmv_algorithmic_bandwidth", "value": value, "unit": "GB/s", "n_gpus": ngpu,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": cfg,
            "detail": {"exchange": "peer memory: one kernel per step runs the device-side flag barrier and copies the halo "
                                   "(the columns a shard reaches into its neighbours' slices of x) over NVLink next to "
                                   "the own slice; the product then reads one local array" if ngpu > 1 else "none",
                       "spmv_kernel": kname, "lanes_per_row": choice[1] if lanes == 0 else lanes,
                       "rows_per_rank": nloc, "pct_of_8TBps_nominal_per_gpu": 100.0 * achieved / 8000.0},
            "e2e": {"value": e2e_value, "unit": "GB/s", "h2d_bytes_per_step": h2d * ngpu, "d2h_bytes_per_step": d2h * ngpu,
                    "steps": e2e_steps, "ms_per_step": e2e_s * 1e3, "launches_per_step": e2e_launches,
                    "what": "&A * &x on a constructed (device-resident) CsrMatrix with pinned host x, y: "
                            + ("spl_spmv_host" if ngpu == 1 else "spl_spmv_peer_host on every rank (slice upload, barrier, "
                                                                 "chunked product with the download behind it)")},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src, "kernel": "spmv_" + kname, "kernel_ms": kern_ms,
                         "bytes_per_launch": bytes_local},
            "clocks": clk,
        }
        if parity:
            line["parity_check"] = parity
        if cpu:
            line["cpu_baseline"] = cpu
        line.update(extras)
        if dumped is not None:
            write_outputs(args.dump_outputs, n, *dumped)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------- N > 1 extras
def sharded_extras(torch, dist, sp, spd, ctx, A, n, r0, r1, rank, world):
    """Secondary sharded metrics on FIXED global inputs (the same problem at every N): the add of
    config 5 (A + B, B = offsets {-8,-2,0,2,8}; no exchange), COO->CSR assembly of config 3's triplet
    list block-distributed by entry index (NCCL all-to-all, and routing fused with the exchange over
    peer memory), the general (random-column) SpMV with x all-gathered, and config 4 (R-MAT) with an
    nnz-balanced row partition.  Times are the slowest rank's; rates are whole-job."""
    from spalinalg_b200 import sharding
    from spalinalg_b200.synthetic_device import banded_device, device_view, random_uniform_coo_device, rmat_coo_device
    from tests.test_dist import syn_block
    out = {}

    def timed_all(fn, reps=3, warm=1, batch=1):
        """ms per call, max over ranks, median of `reps`.  batch > 1: that many calls back to back between the events
        (a product of ~0.1 ms timed alone would mostly measure how far apart the ranks' hosts left the barrier)."""
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(reps):
            dist.barrier(); torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(batch):
                fn()
            b.record()
            torch.cuda.synchronize()
            t = torch.tensor([a.elapsed_time(b) / batch], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ts.append(float(t.item()))
        return statistics.median(ts)

    def agree(ok):
        """The same verdict on every rank (a check that failed on one rank only must not leave the others waiting
        in the next collective): True when it held everywhere."""
        t = torch.tensor([1 if ok else 0], device="cuda", dtype=torch.int32)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    def worst(v):
        t = torch.tensor([float(v)], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def total(v, op=None):
        t = torch.tensor([v], device="cuda", dtype=torch.int64)
        dist.all_reduce(t, op=op or dist.ReduceOp.SUM)
        return int(t.item())

    # ---- what the host link gives every rank when all ranks copy at once (explains e2e: the slices of x and y
    # are 2 x (n / N) x 8 bytes of pinned traffic per rank and step)
    probe_h = torch.empty(64 << 20, dtype=torch.uint8).pin_memory()
    probe_d = torch.empty(64 << 20, dtype=torch.uint8, device="cuda")
    side = torch.cuda.Stream()

    def h2d():
        probe_d.copy_(probe_h, non_blocking=True)

    def d2h():
        probe_h.copy_(probe_d, non_blocking=True)

    def both():
        probe_d.copy_(probe_h, non_blocking=True)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            probe_h2.copy_(probe_d2, non_blocking=True)
        torch.cuda.current_stream().wait_stream(side)
    probe_h2 = torch.empty(64 << 20, dtype=torch.uint8).pin_memory()
    probe_d2 = torch.empty(64 << 20, dtype=torch.uint8, device="cuda")
    gb = (64 << 20) / 1e6
    out["host_link_probe"] = {"what": "64 MiB pinned copies on every rank at the same time; GB/s per rank (slowest rank)",
                              "h2d_gbps": gb / timed_all(h2d, reps=5, warm=2), "d2h_gbps": gb / timed_all(d2h, reps=5, warm=2),
                              "both_directions_gbps_each": gb / timed_all(both, reps=5, warm=2)}
    del probe_h, probe_d, probe_h2, probe_d2

    # ---- config 5: A + B, rows sharded, no exchange
    bp, bc, bv = banded_device(torch, n, r0, r1, (-8, -2, 0, 2, 8), torch.float64)
    B = sp.CsrMatrix.from_device_arrays(r1 - r0, n, bc.numel(), bp.data_ptr(), bc.data_ptr(), bv.data_ptr(),
                                        np.float64, validate=False, ctx=ctx)
    del bp, bc, bv
    keep = {}

    def add():
        keep["C"] = A + B
    ms = timed_all(add)
    na, nb, nc = total(A.nnz()), total(B.nnz()), total(keep["C"].nnz())
    b_add = (na + nb + nc) * 12 + 3 * (n + world) * 4
    out["sharded_add"] = {"workload": "banded9 + banded{-8,-2,0,2,8}, n=1e8, f64, rows sharded, no exchange",
                          "ms": ms, "nnz_out": nc, "mnnz_per_s": (na + nb) / ms / 1e3,
                          "gbps_algorithmic": b_add / ms / 1e6}
    del keep["C"], B
    torch.cuda.empty_cache()

    # ---- config 3: the SAME 168 M triplets at every N, rank g holds entries [g*len/N, (g+1)*len/N)
    nr = 10_000_000
    gr, gc, gv = random_uniform_coo_device(torch, nr, 16, 8_000_000, torch.float32, seed=1)
    ln = int(gv.numel())
    a_, b_ = syn_block(ln, world, rank)
    r_, c_, v_ = gr[a_:b_].clone(), gc[a_:b_].clone(), gv[a_:b_].clone()
    del gr, gc, gv
    torch.cuda.empty_cache()

    def asm():
        keep["D"] = spd.DistCsrMatrix.from_device_triplets(dist, torch, nr, nr, r_, c_, v_, ctx=ctx)
    ms = timed_all(asm)
    ex = spd.PeerExchange(ctx, dist)

    def asm_peer():
        keep["P"] = spd.DistCsrMatrix.from_device_triplets_peer(dist, torch, nr, nr, r_, c_, v_, ex)
    ms_p = timed_all(asm_peer)
    ex.check()
    same_nnz = agree(keep["P"].local.nnz() == keep["D"].local.nnz())
    del keep["P"]
    D = keep["D"]
    nnz_d = total(D.local.nnz())
    out["sharded_assembly"] = {"workload": "config 3: random 1e7 x 1e7, 16/row + 5% duplicates, f32, the same 168 M "
                                           "triplets at every N, block-distributed by entry index, one NCCL all-to-all",
                               "len": ln, "nnz_out": nnz_d, "ms": ms, "mnnz_per_s": ln / ms / 1e3}
    out["sharded_assembly_peer"] = {"workload": "same triplets; routing and exchange fused: the partition pass writes "
                                                "into the owners' buffers over NVLink (peer memory), no all-to-all",
                                    "len": ln, "nnz_out": nnz_d, "ms": ms_p if same_nnz else None,
                                    "mnnz_per_s": ln / ms_p / 1e3 if same_nnz else None, "same_nnz_as_nccl_route": same_nnz}
    del r_, c_, v_

    # general (random-column) matrix: x exchanged (NCCL all-gather / pull over peer memory), then the local SpMV
    d0, d1 = D.local_rows()
    xg = torch.rand(nr, device="cuda", dtype=torch.float32) - 0.5
    yg = torch.empty(d1 - d0, device="cuda", dtype=torch.float32)
    even = nr % world == 0

    def spmv_ag():
        sharding.exchange_allgather(dist, xg, d0, d1, world, even)
        D.local.spmv_device(xg.data_ptr(), yg.data_ptr())
    ms = timed_all(spmv_ag, reps=7, warm=3, batch=10)
    b_ag = nnz_d * 8 + 2 * nr * 4
    xs = spd.PeerVector(ctx, dist, nr, np.float32, D.starts)
    device_view(torch, xs.local_ptr, d1 - d0, torch.float32).copy_(xg[d0:d1])
    xs.publish()
    torch.cuda.synchronize()

    def spmv_pull():
        xs.barrier()
        xs.pull(xg.data_ptr())
        D.local.spmv_device(xg.data_ptr(), yg.data_ptr())
    y_ag = yg.clone()
    ms_pull = timed_all(spmv_pull, reps=7, warm=3, batch=10)
    xs.check()
    pull_same = agree(torch.equal(y_ag, yg))                             # same kernel on the same x: bit for bit

    def fused_section():
        # the all-gather fused into the product: one persistent kernel, a copy warp per CTA pulls the slices over NVLink
        # (TMA bulk copies) while the compute warps work through the owner blocks
        D.prepare_gather(torch)

        def spmv_fused():
            D.spmv_gather(xs, xg.data_ptr(), yg.data_ptr(), barrier=True)      # the barrier is part of the kernel
        ms_fused = timed_all(spmv_fused, reps=7, warm=3, batch=10)
        xs.check()
        err = worst(((yg - y_ag).abs().max() / (y_ag.abs().max() + 1e-30)).item())
        fused_ok = err < 1e-5                                                # the same on every rank
        # where the time of one fused product goes: %globaltimer stamps from the kernel (first CTA)
        first = D._gather["first"]
        nb = len(first) - 1
        tl = torch.zeros(2 + 3 * nb, dtype=torch.int64, device="cuda")
        dist.barrier(); torch.cuda.synchronize()
        for _ in range(6):                                                   # stamps of a product in the middle of a run of them:
            spmv_fused()                                                     # a lone launch would mostly show how far apart the
        D.spmv_gather(xs, xg.data_ptr(), yg.data_ptr(), barrier=True, timeline_dev=tl.data_ptr())     # ranks' hosts are
        for _ in range(3):
            spmv_fused()
        torch.cuda.synchronize()
        t = tl.cpu().tolist()
        t0 = t[1]                                                            # the first consumer warp starts
        stamps = [{"block": k, "ring_offsets": [first[k], first[k + 1]], "wait_begins_us": (t[1 + 3 * k] - t0) / 1e3,
                   "slices_landed_us": (t[2 + 3 * k] - t0) / 1e3, "block_done_us": (t[3 + 3 * k] - t0) / 1e3}
                  for k in range(nb)]
        stamps.append({"last_cta_done_us": (t[1 + 3 * nb] - t0) / 1e3, "first_peer_arrived_copy_starts_us": (t[0] - t0) / 1e3})
        # how the shard is blocked (one pass over the rows per block) and how many CTAs stay resident: measured per run,
        # the library's defaults stand in the headline number above
        sweep = {}
        shapes = {"per_rank": list(range(world + 1)), "own|rest": [0, 1, world]}
        if world >= 8:
            shapes["1|1|2|4"] = [0, 1, 2, 4, 8]
            shapes["1|1|1|1|2|2"] = [0, 1, 2, 3, 4, 6, 8]
        for name, bf in shapes.items():
            if bf == first or len(set(bf)) != len(bf):
                continue
            D.prepare_gather(torch, block_first=bf)
            try:
                sweep["blocks " + name] = timed_all(spmv_fused, reps=5, warm=2, batch=10)
                e2 = worst(((yg - y_ag).abs().max() / (y_ag.abs().max() + 1e-30)).item())
                if not e2 < 1e-5:
                    sweep["blocks " + name] = f"MISMATCH against the all-gather product: {e2:.3g}"
            except RuntimeError as e:
                sweep["blocks " + name] = str(e)[:60]
        for knob, value in (("SPL_GATHER_CTAS_PER_SM", "4"), ("SPL_GATHER_CTAS_PER_SM", "2"), ("SPL_GATHER_LANES", "2"),
                            ("SPL_GATHER_STAGES", "3")):
            os.environ[knob] = value
            D.prepare_gather(torch)                                          # fresh counters: the grid size may change
            label = f"{knob[11:].lower()} {value}"
            try:
                sweep[label] = timed_all(spmv_fused, reps=5, warm=2, batch=10)
                e2 = worst(((yg - y_ag).abs().max() / (y_ag.abs().max() + 1e-30)).item())
                if not e2 < 1e-5:
                    sweep[label] = f"MISMATCH against the all-gather product: {e2:.3g}"
            except RuntimeError as e:
                sweep[label] = str(e)[:60]
            os.environ.pop(knob, None)
        xs.check()
        return {"workload": "same matrix; ONE kernel: the device barrier, one copy warp per CTA pulling "
                                                        "the peers' slices of x over NVLink with TMA bulk copies, and the compute "
                                                        "warps multiplying the shard block by block (blocked by column owner, ring "
                                                        "order) as the slices land",
                                            "ms": ms_fused if fused_ok else None,      # no number for a product that is off
                                            "gbps_algorithmic": b_ag / ms_fused / 1e6 if fused_ok else None,
                                            "within_1e-5_of_allgather": fused_ok, "max_rel_diff_vs_allgather": err if err == err else None, "block_first": first, "ms_variants": sweep,
                                            "timeline_rank0_first_cta": stamps}
    try:
        out["sharded_spmv_gather_fused"] = fused_section()
    except RuntimeError as e:                                             # the library refused (same on every rank): say so
        out["sharded_spmv_gather_fused"] = {"error": str(e)[:200]}
        os.environ.pop("SPL_GATHER_CTAS_PER_SM", None); os.environ.pop("SPL_GATHER_LANES", None); os.environ.pop("SPL_GATHER_STAGES", None)
    out["sharded_spmv_allgather"] = {"workload": "config 3 matrix assembled above (random 16/row, f32), x all-gathered "
                                                 "with NCCL every step", "ms": ms, "gbps_algorithmic": b_ag / ms / 1e6,
                                     "x_bytes_received_per_rank": (nr - (d1 - d0)) * 4}
    out["sharded_spmv_peer_pull"] = {"workload": "same matrix; x all-gathered by one pull kernel over peer memory "
                                                 "(device barrier, then a TMA ring per CTA: NVLink reads), then the local SpMV",
                                     "ms": ms_pull if pull_same else None,
                                     "gbps_algorithmic": b_ag / ms_pull / 1e6 if pull_same else None,
                                     "bit_identical_to_allgather": pull_same}
    xs.close(dist)
    del D, keep["D"], xg, yg, y_ag
    torch.cuda.empty_cache()

    # ---- config 4: R-MAT 2^24, the SAME 2^29 edges at every N, nnz-balanced row partition
    scale = 24
    n4 = 1 << scale
    gr, gc, gv = rmat_coo_device(torch, scale, 32, torch.float32, seed=3)
    ln4 = int(gv.numel())
    a_, b_ = syn_block(ln4, world, rank)
    r_, c_, v_ = gr[a_:b_].clone(), gc[a_:b_].clone(), gv[a_:b_].clone()
    del gr, gc, gv
    torch.cuda.empty_cache()
    res4 = {}
    for balance in ("nnz", None):
        def asm4():
            keep["R"] = spd.DistCsrMatrix.from_device_triplets_peer(dist, torch, n4, n4, r_, c_, v_, ex, balance=balance)
        ms_a = timed_all(asm4, reps=2, warm=1)
        R = keep["R"]
        q0, q1 = R.local_rows()
        nnz_max, nnz_sum = total(R.local.nnz(), dist.ReduceOp.MAX), total(R.local.nnz())
        x4 = torch.rand(n4, device="cuda", dtype=torch.float32) - 0.5
        y4 = torch.empty(q1 - q0, device="cuda", dtype=torch.float32)
        xs4 = spd.PeerVector(ctx, dist, n4, np.float32, R.starts)
        device_view(torch, xs4.local_ptr, q1 - q0, torch.float32).copy_(x4[q0:q1])
        xs4.publish()

        def spmv4():
            xs4.barrier()
            xs4.pull(x4.data_ptr())
            R.local.spmv_device(x4.data_ptr(), y4.data_ptr())
        ms_s = timed_all(spmv4, reps=7, warm=3, batch=10)
        xs4.check()
        b4 = nnz_sum * 8 + 2 * n4 * 4
        res4["nnz_balanced" if balance else "equal_rows"] = {
            "assembly_ms": ms_a, "assembly_mnnz_per_s": ln4 / ms_a / 1e3, "nnz": nnz_sum,
            "max_rank_share_of_nnz": nnz_max / nnz_sum, "spmv_ms": ms_s, "spmv_gbps_algorithmic": b4 / ms_s / 1e6,
            "rows_of_rank0": R.starts[1]}
        xs4.close(dist)
        del R, keep["R"], x4, y4
        torch.cuda.empty_cache()
    res4["workload"] = ("config 4: R-MAT scale 24, 2^29 edges (the same list at every N, block-distributed by entry index), "
                        "f32; assembly fused with the exchange over peer memory; SpMV = barrier + pulled all-gather of x "
                        "+ the nnz-split kernel on the shard")
    out["sharded_rmat"] = res4
    ex.close()
    return out if rank == 0 else {}


# ------------------------------------------------------------------------------- N = 1 extras
def secondary_metrics(torch, sp, ctx, A5, wl):
    """Configs 1-4 on one GPU and the add of config 5: SpMV (ms, algorithmic GB/s, fraction of the
    measured HBM peak, kernel chosen), COO->CSR assembly, CSR->CSC / transpose — each with its own
    algorithmic bytes (SURVEY.md 8d) — plus the reference's general Mul on config 1."""
    from spalinalg_b200 import _capi as capi
    from spalinalg_b200.synthetic_device import (banded_device, random_uniform_coo_device, rmat_coo_device,
                                                 stencil_device)
    out = {}
    peak, _ = peaks()

    def timed(fn, reps=5, warm=2):
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record(); fn(); b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return statistics.median(ts)

    def spmv_rate(M, x, y, copies=1, reps=100):
        """Back-to-back launches; `copies` > 1 rotates over independent (A, x, y) sets whose total
        footprint exceeds L2, so every launch reads from HBM."""
        for i in range(5):
            M[i % copies].spmv_device(x[i % copies].data_ptr(), y[i % copies].data_ptr())
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for i in range(reps):
            M[i % copies].spmv_device(x[i % copies].data_ptr(), y[i % copies].data_ptr())
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    def spmv_entry(M, V, tdt, copies=1, reps=100, note=None):
        Ms = M if isinstance(M, list) else [M]
        n_, m_, nnz_ = Ms[0].nrows(), Ms[0].ncols(), Ms[0].nnz()
        xs = [torch.rand(m_, device="cuda", dtype=tdt) - 0.5 for _ in Ms]
        ys = [torch.empty(n_, device="cuda", dtype=tdt) for _ in Ms]
        b = spmv_bytes(nnz_, n_, m_, V)
        ms = spmv_rate(Ms, xs, ys, copies=len(Ms), reps=reps)
        k, l = Ms[0].spmv_choice()
        e = {"ms": ms, "gbps": b / ms / 1e6, "frac_measured_peak": b / ms / 1e6 / peak, "frac_8TBps": b / ms / 1e6 / 8000.0,
             "kernel": KERNEL_NAMES.get(k, "?"), "lanes_per_row": l, "algorithmic_bytes": b, "nrows": n_, "nnz": nnz_}
        if note:
            e["l2"] = note
        return e

    def tr_entry(fn, M, V):
        ms = timed(fn, reps=5, warm=1)
        b = 2 * M.nnz() * (4 + V) + (M.nrows() + 1) * 4 + (M.ncols() + 1) * 4
        return {"ms": ms, "mnnz_per_s": M.nnz() / ms / 1e3, "gbps_algorithmic": b / ms / 1e6,
                "frac_measured_peak": b / ms / 1e6 / peak}

    def asm_entry(nr, nc, r_, c_, v_, npdt, V, reps=5):
        keep = {}
        ln = int(r_.numel())

        def run():
            keep["A"] = sp.CsrMatrix.from_device_triplets(nr, nc, ln, r_.data_ptr(), c_.data_ptr(), v_.data_ptr(), npdt, ctx=ctx)
        ms = timed(run, reps=reps, warm=1)
        M = keep["A"]
        b = ln * (8 + V) + M.nnz() * (4 + V) + (nr + 1) * 4
        return M, {"len": ln, "nnz_out": M.nnz(), "ms": ms, "mnnz_per_s": ln / ms / 1e3,
                   "gbps_algorithmic": b / ms / 1e6, "frac_measured_peak": b / ms / 1e6 / peak}

    # ---- config 5: A + B (the bench matrix is A)
    n5 = A5.nrows()
    if wl.startswith("banded"):
        bp, bc, bv = banded_device(torch, n5, 0, n5, (-8, -2, 0, 2, 8), torch.float64)
        B = sp.CsrMatrix.from_device_arrays(n5, n5, bc.numel(), bp.data_ptr(), bc.data_ptr(), bv.data_ptr(), np.float64,
                                            validate=False, ctx=ctx)
        del bp, bc, bv
        keep = {}

        def add():
            keep["C"] = A5 + B
        ms = timed(add, reps=3, warm=1)
        Cm = keep["C"]
        b = (A5.nnz() + B.nnz() + Cm.nnz()) * 12 + 3 * (n5 + 1) * 4
        out["c5_add"] = {"workload": "banded9 + banded{-8,-2,0,2,8}, n=%d, f64" % n5, "ms": ms, "nnz_out": Cm.nnz(),
                         "mnnz_per_s": (A5.nnz() + B.nnz()) / ms / 1e3, "gbps_algorithmic": b / ms / 1e6,
                         "frac_measured_peak": b / ms / 1e6 / peak}
        del keep, Cm, B
        torch.cuda.empty_cache()

    # ---- config 1: 2-D Laplacian 1024^2, f64
    offs = [(0, 0), (-1, 0), (1, 0), (0, -1), (0, 1)]
    n, rowptr, colind, values = stencil_device(torch, offs, 1024, 4.0, -1.0, torch.float64)
    rows = torch.repeat_interleave(torch.arange(n, device="cuda", dtype=torch.int32),
                                   (rowptr[1:] - rowptr[:-1]).to(torch.int64))
    g = torch.Generator(device="cuda"); g.manual_seed(42)
    perm = torch.randperm(rows.numel(), device="cuda", generator=g)
    shuffled = (rows[perm].contiguous(), colind[perm].contiguous(), values[perm].contiguous())
    _, out["c1_assembly_shuffled"] = asm_entry(n, n, *shuffled, np.float64, 8)
    _, out["c1_assembly_row_ordered"] = asm_entry(n, n, rows, colind, values, np.float64, 8)
    for k_ in ("c1_assembly_shuffled", "c1_assembly_row_ordered"):
        out[k_]["workload"] = "laplace2d_1024_f64 COO->CSR, device-resident SoA triplets in, device CSR out"

    # the same assembly through the reference-facing call: host usize (u64) row/col + f64 values in
    # pinned memory -> spl_mat_from_coo (upload, narrow, sort, sum) -> CsrMatrix
    sr, sc_, sv = shuffled
    coo_h = [t.cpu().pin_memory() for t in (sr.to(torch.int64), sc_.to(torch.int64), sv)]
    lib = ctx._lib

    def asm_host():
        h = C.c_void_p()
        ctx.check(lib.spl_mat_from_coo(ctx._h, capi.SPL_CSR, capi.SPL_F64, n, n, coo_h[2].numel(),
                                       C.c_void_p(coo_h[0].data_ptr()), C.c_void_p(coo_h[1].data_ptr()),
                                       C.c_void_p(coo_h[2].data_ptr()), 1, 1, C.byref(h)))
        ctx.check(lib.spl_mat_free(ctx._h, h))
    asm_host(); asm_host()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(5):
        asm_host()
    torch.cuda.synchronize()
    hs = (time.perf_counter() - t0) / 5
    out["c1_assembly_shuffled_e2e"] = {"workload": "laplace2d_1024_f64 COO->CSR from pinned host usize triplets",
                                       "len": int(coo_h[2].numel()), "ms": hs * 1e3,
                                       "mnnz_per_s": coo_h[2].numel() / hs / 1e6,
                                       "h2d_bytes": int(coo_h[2].numel()) * 24}
    # the same triplets through the streaming CooMatrix storage (spl_coo, SURVEY 8f-4)
    np_trip = [t.numpy() for t in coo_h]
    np_trip = (np_trip[0].view(np.uint64), np_trip[1].view(np.uint64), np_trip[2])
    ln = int(np_trip[2].shape[0])
    fill_s, conv_s = [], []
    for it in range(5):
        pc = sp.PinnedCooMatrix.with_capacity(n, n, ln, np.float64, ctx=ctx)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pc.extend_triplets(*np_trip)
        t1 = time.perf_counter()
        M_ = sp.CsrMatrix.from_coo(pc, ctx=ctx)
        ctx.sync()
        t2 = time.perf_counter()
        if it:
            fill_s.append(t1 - t0); conv_s.append(t2 - t1)
        del M_, pc
    fill_ms, conv_ms = 1e3 * float(np.median(fill_s)), 1e3 * float(np.median(conv_s))
    out["c1_assembly_shuffled_streamed"] = {
        "workload": "laplace2d_1024_f64: PinnedCooMatrix filled from host usize triplets, then CsrMatrix::from(&coo)",
        "len": ln, "fill_ms": fill_ms, "convert_ms": conv_ms, "total_ms": fill_ms + conv_ms,
        "convert_mnnz_per_s": ln / conv_ms / 1e3, "total_mnnz_per_s": ln / (fill_ms + conv_ms) / 1e3}
    del coo_h, np_trip, shuffled, perm, rows

    mk1 = lambda: sp.CsrMatrix.from_device_arrays(n, n, colind.numel(), rowptr.data_ptr(), colind.data_ptr(),
                                                  values.data_ptr(), np.float64, validate=False, ctx=ctx)
    A1 = [mk1() for _ in range(4)]
    out["c1_spmv"] = spmv_entry(A1, 8, torch.float64, reps=400, note="4 rotating copies of (A, x, y), 320 MB > L2")
    out["c1_spmv_l2_resident"] = spmv_entry(A1[0], 8, torch.float64, reps=400, note="one copy, 80 MB: L2-resident")
    out["c1_csr_to_csc"] = tr_entry(lambda: A1[0].to_csc(), A1[0], 8)
    keepm = {}

    def mul():
        keepm["C"] = A1[0] * A1[0]
    ms = timed(mul, reps=5, warm=2)
    out["c1_mul"] = {"workload": "A * A, 2-D Laplacian 1024^2 (impl Mul for &CsrMatrix)", "ms": ms,
                     "nnz_out": keepm["C"].nnz(), "mnnz_out_per_s": keepm["C"].nnz() / ms / 1e3}
    del A1, keepm, rowptr, colind, values
    torch.cuda.empty_cache()

    # ---- config 2: 27-point stencil 128^3, f64
    offs = [(a, b, c) for a in (-1, 0, 1) for b in (-1, 0, 1) for c in (-1, 0, 1)]
    n, rowptr, colind, values = stencil_device(torch, offs, 128, 26.0, -1.0, torch.float64)
    A2 = sp.CsrMatrix.from_device_arrays(n, n, colind.numel(), rowptr.data_ptr(), colind.data_ptr(), values.data_ptr(),
                                         np.float64, validate=False, ctx=ctx)
    del rowptr, colind, values
    out["c2_spmv"] = spmv_entry(A2, 8, torch.float64, reps=100)
    out["c2_csr_to_csc"] = tr_entry(lambda: A2.to_csc(), A2, 8)
    out["c2_transpose"] = tr_entry(lambda: A2.transpose(), A2, 8)
    # the host-vector product on this matrix, pipelined (16.8 MB each way), and with the matrix built from the
    # reference-layout host arrays inside every step
    h_x = torch.rand(n, dtype=torch.float64).pin_memory()
    h_y = torch.empty(n, dtype=torch.float64).pin_memory()
    b2 = spmv_bytes(A2.nnz(), n, n, 8)

    def host_step():
        ctx.check(lib.spl_spmv_host(ctx._h, A2._h, C.c_void_p(h_x.data_ptr()), C.c_void_p(h_y.data_ptr())))
    host_step(); host_step()
    t0 = time.perf_counter()
    for _ in range(10):
        host_step()
    hs = (time.perf_counter() - t0) / 10
    out["c2_spmv_host_vectors"] = {"ms": hs * 1e3, "gbps": b2 / hs / 1e9, "h2d_bytes_per_step": n * 8, "d2h_bytes_per_step": n * 8,
                                   "what": "spl_spmv_host: x up in prefixes, row chunks, y down behind them (3 streams)"}
    del A2, h_x, h_y
    torch.cuda.empty_cache()

    # ---- config 3: random 1e7 x 1e7, 16/row + 5 % duplicates, f32
    n = 10_000_000
    r_, c_, v_ = random_uniform_coo_device(torch, n, 16, 8_000_000, torch.float32, seed=1)
    A3, out["c3_assembly"] = asm_entry(n, n, r_, c_, v_, np.float32, 4, reps=3)
    del r_, c_, v_
    torch.cuda.empty_cache()
    out["c3_spmv"] = spmv_entry(A3, 4, torch.float32, reps=30)
    out["c3_csr_to_csc"] = tr_entry(lambda: A3.to_csc(), A3, 4)
    del A3
    torch.cuda.empty_cache()

    # ---- config 4: R-MAT 2^24, 2^29 edges, f32
    n = 1 << 24
    r_, c_, v_ = rmat_coo_device(torch, 24, 32, torch.float32, seed=3)
    A4, out["c4_assembly"] = asm_entry(n, n, r_, c_, v_, np.float32, 4, reps=3)
    del r_, c_, v_
    torch.cuda.empty_cache()
    out["c4_spmv"] = spmv_entry(A4, 4, torch.float32, reps=20)
    out["c4_transpose"] = tr_entry(lambda: A4.transpose(), A4, 4)
    del A4
    torch.cuda.empty_cache()
    return out


if __name__ == "__main__":
    main()
