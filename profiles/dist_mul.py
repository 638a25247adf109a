"""Row-sharded sparse product (DistCsrMatrix.mul) against the one-GPU product of the whole problem.

Run with `torchrun --nproc-per-node N profiles/dist_mul.py [--reps R] [--workloads c1,stencil,random]` (one process per GPU).  For each workload
every rank builds the whole matrix on its GPU (also the reference), keeps its row block, and times, device-
synchronised, max over the ranks, median of the timed repetitions after one warm-up product:
  setup    the peer buffers of B (all-gather of the shard sizes, three spl_peer_alloc + opens, the own shard copied in)
  gather   spl_peer_gather_rows between the two flag barriers, with the bytes it read from peers' shards
  product  spl_mat_mul of the row block by the gathered matrix
  total    the three plus closing the buffers
  1-GPU    spl_mat_mul of the whole problem on one GPU
Every rank's block of every timed product is compared bit for bit with the rows of the one-GPU product."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import spalinalg_b200 as sp
from spalinalg_b200 import dist as spd
from spalinalg_b200 import synthetic as syn
from spalinalg_b200.synthetic_device import device_view


def card():
    name = torch.cuda.get_device_name()
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    except OSError:
        pl = "unknown"
    return f"{name}, power limit {pl}"


def workloads(which):
    rng = np.random.default_rng(1)
    if "c1" in which:
        r, c, v = syn.laplacian_2d(1024)
        yield "C1 2-D Laplacian 1024^2 f64, A*A", 1024 * 1024, r, c, v
    if "stencil" in which:
        r, c, v = syn.stencil_27(128)
        yield "27-point stencil 128^3 f64, A*A", 128 ** 3, r, c, v
    if "random" in which:
        n = 1 << 21
        r = np.repeat(np.arange(n, dtype=np.int64), 16)
        yield "random 2^21 rows x 16 per row f32, A*A", n, r, rng.integers(0, n, len(r)), \
            rng.standard_normal(len(r)).astype(np.float32)


def row_block(ctx, M, n, starts, rank):
    p, i, v = M.device_ptrs()
    item = M.dtype.itemsize
    ptr = device_view(torch, p, n + 1, torch.int32).long()
    r0, r1 = starts[rank], starts[rank + 1]
    lo, hi = int(ptr[r0]), int(ptr[r1])
    lp = (ptr[r0:r1 + 1] - lo).to(torch.int32).contiguous()
    B = sp.CsrMatrix.from_device_arrays(r1 - r0, n, hi - lo, lp.data_ptr(), i + 4 * lo, v + item * lo, M.dtype,
                                        validate=False, ctx=ctx)
    ctx.sync()
    return B


def same_rows(W, n, P, r0, r1):
    """P (rows r0..r1 of a product) equals those rows of W bit for bit (compared on the device)."""
    wp, wi, wv = W.device_ptrs()
    pp, pi, pv = P.device_ptrs()
    bits = torch.int32 if W.dtype == np.float32 else torch.int64
    w = device_view(torch, wp, n + 1, torch.int32).long()
    lo, hi = int(w[r0]), int(w[r1])
    if P.nnz() != hi - lo:
        return False
    p = device_view(torch, pp, r1 - r0 + 1, torch.int32).long()
    if not torch.equal(p, w[r0:r1 + 1] - lo):
        return False
    if hi == lo:
        return True
    item = W.dtype.itemsize
    return (torch.equal(device_view(torch, wi + 4 * lo, hi - lo, torch.int32), device_view(torch, pi, hi - lo, torch.int32))
            and torch.equal(device_view(torch, wv + item * lo, hi - lo, bits), device_view(torch, pv, hi - lo, bits)))


def tmax(x):
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", default="c1,stencil,random")
    args = ap.parse_args()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = sp.Context(torch.cuda.current_device(), stream.cuda_stream)
    sp.set_default_context(ctx)
    say = print if rank == 0 else (lambda *a, **k: None)
    say(f"# {card()}; N = {world} GPU(s); times in ms, max over ranks, median of {args.reps} after one warm-up")
    for what, n, r, c, v in workloads(args.workloads.split(",")):
        M = sp.CsrMatrix.from_coo(sp.CooMatrix.with_triplets(n, n, r, c, v), ctx=ctx)
        starts = spd.partition_starts(n, world)
        D = spd.DistCsrMatrix(row_block(ctx, M, n, starts, rank), starts, rank, n, n)
        one = []
        for i in range(args.reps + 1):
            ctx.sync()
            t0 = time.perf_counter()
            W = M * M
            ctx.sync()
            if i:
                one.append(time.perf_counter() - t0)
        rows = {k: [] for k in ("setup", "gather", "product", "total")}
        ok, remote = True, 0
        for i in range(args.reps + 1):
            dist.barrier()
            ctx.sync()
            t0 = time.perf_counter()
            shard = spd._PeerShard(D, dist, torch)
            ctx.sync()
            t1 = time.perf_counter()
            G = shard.gather(D.local)
            ctx.sync()
            t2 = time.perf_counter()
            P = D.local * G
            ctx.sync()
            t3 = time.perf_counter()
            shard.close()
            t4 = time.perf_counter()
            ok &= same_rows(W, n, P, starts[rank], starts[rank + 1])
            gp = device_view(torch, G.device_ptrs()[0], n + 1, torch.int32).long()
            own = int(gp[starts[rank + 1]]) - int(gp[starts[rank]])
            remote = (G.nnz() - own) * (4 + M.dtype.itemsize)
            if i:
                for k, dt in zip(rows, (t1 - t0, t2 - t1, t3 - t2, t4 - t0)):
                    rows[k].append(tmax(dt))
            del G, P
        flag = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        rb = torch.tensor([remote], dtype=torch.float64, device="cuda")
        dist.all_reduce(rb, op=dist.ReduceOp.MAX)
        med = {k: 1e3 * float(np.median(x)) for k, x in rows.items()}
        one_ms = tmax(float(np.median(one))) * 1e3
        rate = rb.item() / (med["gather"] * 1e-3) / 1e9 if rb.item() else 0.0
        say(f"{what}: n={n} nnz(A)={M.nnz()} nnz(A*A)={W.nnz()}  N={world}  setup {med['setup']:.2f}  "
            f"gather {med['gather']:.2f} (remote {rb.item() / 1e6:.1f} MB on the busiest rank, {rate:.0f} GB/s)  "
            f"product {med['product']:.2f}  total {med['total']:.2f}  |  1-GPU spl_mat_mul {one_ms:.2f}  "
            f"bit-exact vs 1-GPU: {'yes' if flag.item() else 'NO'}", flush=True)
        del W, D, M
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
