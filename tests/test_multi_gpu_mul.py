"""The row-sharded sparse product on real GPUs: DistCsrMatrix.mul / DistCscMatrix.mul with one process per GPU over
NCCL and CUDA IPC peer memory (skipped on a one-GPU box).  Every rank's block of A·B must equal the same rows
(columns) of the oracle's product of the WHOLE problem, bit for bit."""
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
    from spalinalg_b200 import synthetic as syn
    from tests.test_gather_rows import power_law, random_sparse, shard, special_values

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

        def dcsr(full, starts, nrows, ncols):
            p, i, v = shard(full, starts, rank)
            nloc = starts[rank + 1] - starts[rank]
            if nloc == 0:
                p = np.zeros(2, np.uint64)
            return spd.DistCsrMatrix(sp.CsrMatrix.new(max(nloc, 1), ncols, p, i, v, ctx=ctx), starts, rank, nrows, ncols)

        def same(mat, want):
            got = mat._download()
            return bool(np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
                        and got[2].tobytes() == want[2].tobytes())

        m, k, n = 30011, 20011, 25013
        for dtype in (np.float64, np.float32):
            A = random_sparse(m, k, 4, dtype, 21)
            B = power_law(k, n, dtype, 22)
            B = (B[0], B[1], special_values(B[2], dtype))
            whole = orc.csr_mul(m, k, n, A, B)
            rows = torch.from_numpy(np.repeat(np.arange(m), np.diff(A[0].astype(np.int64))).astype(np.int32)).cuda()
            heavy = spd.balanced_starts_from_rows(dist, torch, rows[: len(rows) * 3 // 4] if rank == 0 else rows[:0],
                                                  m, world)                 # rank 0's rows weigh most
            for a_starts, b_starts in ((spd.partition_starts(m, world), spd.partition_starts(k, world)),
                                       (spd.partition_starts(m, world), [0, k // 5, k]),      # B cut elsewhere
                                       (heavy, [0, k - 7, k])):
                P = dcsr(A, a_starts, m, k).mul(dcsr(B, b_starts, k, n), dist, torch)
                ok &= P.starts == a_starts and same(P.local, shard(whole, a_starts, rank))
            assert ok, f"sharded A*B differs from the oracle ({np.dtype(dtype).name})"
        # A*A on the 27-point stencil: the gather moves a halo of whole planes
        r, c, v = syn.stencil_27(24)
        ns = 24 ** 3
        S = orc.compress_from_coo(ns, ns, orc.make_triplets(r, c, v), "row")
        st = spd.partition_starts(ns, world)
        dS = dcsr(S, st, ns, ns)
        ok &= same(dS.mul(dS, dist, torch).local, shard(orc.csr_mul(ns, ns, ns, S, S), st, rank))
        assert ok, "sharded stencil A*A differs from the oracle"
        # the column-sharded CSC twin
        Ac = orc.recompress(m, k, *random_sparse(m, k, 4, np.float64, 23))
        Bc = orc.recompress(k, n, *random_sparse(k, n, 6, np.float64, 24))
        wc = orc.csr_mul(n, k, m, Bc, Ac)
        ka, nb = [0, k // 3, k], spd.partition_starts(n, world)
        pa, pb = shard(Ac, ka, rank), shard(Bc, nb, rank)
        cA = spd.DistCscMatrix(sp.CscMatrix.new(m, ka[rank + 1] - ka[rank], *pa, ctx=ctx), ka, rank, m, k)
        cB = spd.DistCscMatrix(sp.CscMatrix.new(k, nb[rank + 1] - nb[rank], *pb, ctx=ctx), nb, rank, k, n)
        Q = cA.mul(cB, dist, torch)
        ok &= Q.starts == nb and same(Q.local, shard(wc, nb, rank))
        assert ok, "sharded CSC A*B differs from the oracle"
        # a shape mismatch panics on every rank before any collective (nobody waits)
        dB = dcsr(B, spd.partition_starts(k, world), k, n)
        try:
            dB.mul(dB, dist, torch)
            ok = False
        except sp.Panic:
            pass
        assert ok, "a shape mismatch did not panic"
        dist.barrier()
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
def test_sharded_mul_on_real_gpus():
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
