"""The row-sharded transposed product on real GPUs: one process per GPU over NCCL (skipped on a one-GPU box).
Every rank checks its slice of y = A^T x against the oracle's A^T x of the whole problem (random and banded
matrices, within the SpMV tolerance), then runs 50 steps of v = A x (spmv_halo into a PeerVector) and
x = A^T v (spmv_transpose into the other PeerVector's local_ptr) with one rank delayed at a different point of every
step, and checks the last x bit for bit against a numpy restatement of the same sequence."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, out):
    import oracle as orc
    import spalinalg_b200 as sp
    from spalinalg_b200 import dist as spd
    from spalinalg_b200.synthetic_device import device_view
    from tests.test_spmv_transpose import band9, model_partial, oracle_transpose, random16, shard

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    ok = True
    try:
        stream = torch.cuda.Stream()
        torch.cuda.set_stream(stream)
        ctx = sp.Context(rank, stream.cuda_stream)
        sp.set_default_context(ctx)
        n = 200_003
        starts = spd.partition_starts(n, world)
        r0, r1 = starts[rank], starts[rank + 1]
        for make in (band9, random16):
            full = make(n, np.float64, 21) if make is band9 else make(n, n, np.float64, 22)
            D = spd.DistCsrMatrix(sp.CsrMatrix.new(r1 - r0, n, *shard(full, starts, rank), ctx=ctx), starts, rank, n, n)
            D.prepare_transpose(dist, torch)
            x = np.random.default_rng(23).standard_normal(n)
            xd = torch.from_numpy(x[r0:r1].copy()).cuda()
            yd = torch.full((r1 - r0,), 7.0, dtype=torch.float64, device="cuda")
            for _ in range(3):
                D.spmv_transpose(xd.data_ptr(), yd.data_ptr())
            D.check()
            want, scale = oracle_transpose(full, n, n, x)
            ok &= bool(np.all(np.abs(yd.cpu().numpy() - want[r0:r1]) <= 1e-12 * scale[r0:r1]))
            D.close_transpose(dist)
        assert ok, "sharded A^T x differs from the oracle"

        # x <- A^T (A x), 50 steps; A = the 9-diagonal band scaled so that A^T A stays O(1)
        full = band9(n, np.float64, 24)
        full = (full[0], full[1], full[2] * 0.3)
        D = spd.DistCsrMatrix(sp.CsrMatrix.new(r1 - r0, n, *shard(full, starts, rank), ctx=ctx), starts, rank, n, n)
        D.prepare_transpose(dist, torch)
        widths = D.halo_widths(dist, torch)
        X = spd.PeerVector(ctx, dist, n, np.float64, starts, halo=widths)
        V = spd.PeerVector(ctx, dist, n, np.float64, starts)
        x0 = np.sin(np.arange(n) * 1e-2) + 1.5
        device_view(torch, X.local_ptr, r1 - r0, torch.float64).copy_(torch.from_numpy(x0[r0:r1]))
        X.publish(halo=True)
        delay = 3_000_000
        for t in range(50):
            slow = (t % world) == rank
            if slow and t % 3 == 0:
                torch.cuda._sleep(delay)                # late before v = A x
            D.spmv_halo(X, V.local_ptr)
            V.publish()
            if slow and t % 3 == 1:
                torch.cuda._sleep(delay)                # late between the two products
            D.spmv_transpose(V.published_ptr, X.local_ptr)
            if slow and t % 3 == 2:
                torch.cuda._sleep(delay)                # late after A^T v, before the barrier of x
            X.publish(halo=True)
        torch.cuda.synchronize()
        X.check()
        D.check()
        got = device_view(torch, X.published_ptr, r1 - r0, torch.float64).cpu().numpy()
        ptr, ind, val = full
        windows = D._transpose["windows"]
        ref = x0
        for _ in range(50):
            v = orc.csr_spmv(n, ptr, ind, val, ref)
            v[v == 0] = 0                               # the row kernels' sums start at +0.0
            parts = [model_partial(full, starts, g, n, v) for g in range(world)]
            ref = np.concatenate([spd.reduce_windows_numpy(starts, windows, parts, g, np.float64) for g in range(world)])
        ok &= got.tobytes() == ref[r0:r1].tobytes()
        assert ok, "the A^T A iteration differs from its numpy restatement"
        X.close(dist)
        V.close(dist)
        D.close_transpose(dist)
    finally:
        flag = torch.tensor([1 if ok else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if rank == 0:
            out.put(int(flag.item()))
        dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least two GPUs")
def test_spmv_transpose_on_two_gpus():
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(600)
        assert p.exitcode == 0
    assert out.get(timeout=5) == 1
