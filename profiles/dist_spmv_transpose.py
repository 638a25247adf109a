"""Row-sharded transposed product y = A^T x (DistCsrMatrix.spmv_transpose) against the detour it replaces and
against the forward product of the same shards.

Run with `torchrun --nproc-per-node N profiles/dist_spmv_transpose.py [--samples S]` (one process per GPU; without
torchrun it runs as one rank).  Workloads: config 5 (banded, 9 diagonals, f64, n = 10^8, rows generated per rank)
and config 3's matrix (random 10^7 x 10^7, 16 per row + 5 % duplicates, f32, assembled whole on every rank, each
keeping its row block).  Per workload and sample, ten products back to back on the context's stream, timed with
CUDA events (the detour, which synchronises inside, with a host clock), max over ranks, median over the samples
after one warm-up:
  window   spl_spmv_transpose_window alone (the local partial over the footprint window)
  reduce   spl_peer_reduce_windows alone (flag barrier + the sum of the partials of the own columns)
  new      DistCsrMatrix.spmv_transpose (both launches)
  detour   the CSC view of the same arrays wrapped as a DistCscMatrix, then DistCscMatrix.spmv (full-length
           partial, NCCL reduce-scatter)
  forward  y = A x of the same shards: spmv_halo for the band, spmv_gather (fused all-gather) for the random matrix
The outputs of the new path and of the detour are compared (all-gathered) within rtol * |A|^T |x|."""
import argparse
import ctypes as C
import os
import socket
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import spalinalg_b200 as sp
from spalinalg_b200 import dist as spd
from spalinalg_b200.synthetic_device import banded_device, device_view, random_uniform_coo_device


def card():
    name = torch.cuda.get_device_name()
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    except OSError:
        pl = "unknown"
    return f"{name}, power limit {pl}"


def tmax(x):
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def timed(fn, reps=10):
    """ms per call of `fn` over `reps` calls back to back, CUDA events on the current stream."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def host_timed(fn, reps=10):
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return 1e3 * (time.perf_counter() - t0) / reps


def gather_full(y_local, starts, world):
    """The whole vector from every rank's slice (cut by `starts`)."""
    longest = max(starts[g + 1] - starts[g] for g in range(world))
    buf = torch.zeros(longest, dtype=y_local.dtype, device="cuda")
    buf[:y_local.numel()] = y_local
    allb = torch.empty(longest * world, dtype=y_local.dtype, device="cuda")
    dist.all_gather_into_tensor(allb, buf)
    return torch.cat([allb[g * longest:g * longest + starts[g + 1] - starts[g]] for g in range(world)])


def row_block(ctx, torch, M, n, starts, rank, absval=False):
    p, i, v = M.device_ptrs()
    item = M.dtype.itemsize
    tdt = torch.float32 if M.dtype == np.float32 else torch.float64
    ptr = device_view(torch, p, n + 1, torch.int32).long()
    r0, r1 = starts[rank], starts[rank + 1]
    lo, hi = int(ptr[r0]), int(ptr[r1])
    lp = (ptr[r0:r1 + 1] - lo).to(torch.int32).contiguous()
    vals = device_view(torch, v + item * lo, hi - lo, tdt)
    if absval:
        vals = vals.abs().contiguous()
    torch.cuda.synchronize()
    B = sp.CsrMatrix.from_device_arrays(r1 - r0, n, hi - lo, lp.data_ptr(), i + 4 * lo, vals.data_ptr(), M.dtype,
                                        validate=False, ctx=ctx)
    ctx.sync()
    return B


def workloads(ctx, which, world, rank):
    if "c5" in which:
        n = 100_000_000
        starts = spd.partition_starts(n, world)
        r0, r1 = starts[rank], starts[rank + 1]
        rp, ci, va = banded_device(torch, n, r0, r1, range(-4, 5), torch.float64)
        A = sp.CsrMatrix.from_device_arrays(r1 - r0, n, ci.numel(), rp.data_ptr(), ci.data_ptr(), va.data_ptr(),
                                            np.float64, validate=False, ctx=ctx)
        ctx.sync()
        del rp, ci, va
        # values and x are positive: |A|^T |x| = A^T x
        yield "config 5: banded 9 diagonals, n = 1e8, f64", n, starts, A, None, np.float64
        del A
    if "c3" in which:
        n = 10_000_000
        r_, c_, v_ = random_uniform_coo_device(torch, n, 16, 8_000_000, torch.float32, seed=1)
        torch.cuda.synchronize()
        M = sp.CsrMatrix.from_device_triplets(n, n, r_.numel(), r_.data_ptr(), c_.data_ptr(), v_.data_ptr(), np.float32,
                                              ctx=ctx)
        ctx.sync()
        del r_, c_, v_
        starts = spd.partition_starts(n, world)
        A = row_block(ctx, torch, M, n, starts, rank)
        Aabs = row_block(ctx, torch, M, n, starts, rank, absval=True)
        del M
        yield "config 3: random 1e7 x 1e7, 16/row + 5% duplicates, f32", n, starts, A, Aabs, np.float32


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=5)
    ap.add_argument("--workloads", default="c5,c3")
    args = ap.parse_args()
    if "RANK" not in os.environ:                     # one rank without torchrun
        s = socket.socket()
        s.bind(("127.0.0.1", 0))
        os.environ.update(RANK="0", WORLD_SIZE="1", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(s.getsockname()[1]))
        s.close()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = sp.Context(torch.cuda.current_device(), stream.cuda_stream)
    sp.set_default_context(ctx)
    say = print if rank == 0 else (lambda *a, **k: None)
    say(f"# {card()}; N = {world} GPU(s); ms per product (ten back to back per sample), max over ranks, median of "
        f"{args.samples} samples after one warm-up", flush=True)
    for what, n, starts, A, Aabs, dtype in workloads(ctx, args.workloads.split(","), world, rank):
        tdt = torch.float32 if dtype == np.float32 else torch.float64
        rtol = 1e-5 if dtype == np.float32 else 1e-12
        r0, r1 = starts[rank], starts[rank + 1]
        D = spd.DistCsrMatrix(A, starts, rank, n, n)
        D.prepare_transpose(dist, torch)
        cs = D._transpose["col_starts"]
        c0, c1 = cs[rank], cs[rank + 1]
        idx = torch.arange(r0, r1, device="cuda", dtype=torch.float64)
        x = (1.5 + torch.sin(idx * 1e-3)).to(tdt)
        y = torch.empty(max(c1 - c0, 1), dtype=tdt, device="cuda")
        torch.cuda.synchronize()
        # the two launches of the new path one by one (the reduce without a barrier: flag_ptrs NULL) and together
        T = D._transpose
        part = T["parts"][0]
        cs_arr = (C.c_uint64 * (world + 1))(*cs)
        win = (C.c_uint64 * (2 * world))(*T["windows"])
        pp = (C.c_void_p * world)(*part.ptrs)
        lib, h = ctx._lib, ctx._h
        window = lambda: ctx.check(lib.spl_spmv_transpose_window(h, A._h, C.c_void_p(x.data_ptr()),
                                                                 C.c_void_p(part.local)))
        reduce_ = lambda: ctx.check(lib.spl_peer_reduce_windows(
            h, spd._dtype_code(dtype), world, rank, C.cast(cs_arr, C.c_void_p), C.cast(win, C.c_void_p),
            C.cast(pp, C.c_void_p), None, 0, 2000, C.c_void_p(y.data_ptr())))
        new = lambda: D.spmv_transpose(x.data_ptr(), y.data_ptr())
        # the detour: CSC view of the same arrays (A_local^T, ncols x rows), reduce-scatter of full-length partials
        p_, i_, v_ = A.device_ptrs()
        At = sp.CscMatrix.from_device_arrays(n, max(r1 - r0, 1), A.nnz(), p_, i_, v_, dtype, validate=False, ctx=ctx)
        ctx.sync()
        Dc = spd.DistCscMatrix(At, starts, rank, n, n)
        det_out = {}
        detour = lambda: det_out.update(r=Dc.spmv(dist, torch, x))
        # the forward product of the same shard
        if Aabs is None:
            widths = D.halo_widths(dist, torch)
            xv = spd.PeerVector(ctx, dist, n, dtype, starts, halo=widths)
            device_view(torch, xv.local_ptr, r1 - r0, tdt).copy_(x)
            xv.publish(halo=True)
            yf = torch.empty(max(r1 - r0, 1), dtype=tdt, device="cuda")
            fwd_name = "spmv_halo"
            forward = lambda: (xv.barrier_halo(), D.spmv_halo(xv, yf.data_ptr()))
        else:
            xv = spd.PeerVector(ctx, dist, n, dtype, starts)
            device_view(torch, xv.local_ptr, r1 - r0, tdt).copy_(x)
            xv.publish()
            D.prepare_gather(torch)
            xfull = torch.empty(n, dtype=tdt, device="cuda")
            yf = torch.empty(max(r1 - r0, 1), dtype=tdt, device="cuda")
            fwd_name = "spmv_gather"
            forward = lambda: D.spmv_gather(xv, xfull.data_ptr(), yf.data_ptr(), barrier=True)
        rows = {k: [] for k in ("window", "reduce", "new", "detour", "forward")}
        for s in range(args.samples + 1):
            t = {"window": timed(window), "reduce": timed(reduce_), "new": timed(new),
                 "detour": host_timed(detour), "forward": timed(forward)}
            if s:
                for k, v in t.items():
                    rows[k].append(tmax(v))
        D.check()
        xv.check()
        med = {k: float(np.median(v)) for k, v in rows.items()}
        # agreement of the new path and the detour, and the new path against |A|^T |x|
        new()
        torch.cuda.synchronize()
        y_new = gather_full(y[:c1 - c0], cs, world).double()
        yd, rst = det_out["r"]
        y_det = gather_full(yd, rst, world).double()
        if Aabs is None:
            scale = y_new.abs()
        else:
            Dabs = spd.DistCsrMatrix(Aabs, starts, rank, n, n)
            Dabs.prepare_transpose(dist, torch)
            ya = torch.empty_like(y)
            Dabs.spmv_transpose(x.abs().data_ptr(), ya.data_ptr())
            torch.cuda.synchronize()
            scale = gather_full(ya[:c1 - c0], cs, world).double()
            Dabs.close_transpose(dist)
        worst = float(((y_new - y_det).abs() / (scale + 1e-300)).max().item())
        agree = worst <= 2 * rtol
        say(f"{what}: N={world}  window {med['window']:.3f}  reduce {med['reduce']:.3f}  new (both) {med['new']:.3f}  "
            f"detour (CSC view + reduce-scatter) {med['detour']:.3f}  forward ({fwd_name}) {med['forward']:.3f}  "
            f"[new vs detour: max |diff| / (|A|^T|x|) = {worst:.2e}, {'within' if agree else 'OUTSIDE'} 2 x {rtol:g}]",
            flush=True)
        xv.close(dist)
        D.close_transpose(dist)
        del At, Dc, D, A, Aabs, det_out
        torch.cuda.synchronize()
        ctx.sync()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
