"""The fused all-gather + SpMV kernel for general row shards (spl_spmv_gather_fused) on one GPU.

The ranks are emulated one after the other, without the folded device barrier, so no kernel waits on another
rank: every rank's copy warps pull the peers' slices of x into its own full-length x, and its compute warps wait
only for their own CTAs' copies (all CTAs are resident: cooperative launch).  Without this test the copy warp runs
only in tests/test_multi_gpu.py, which needs two GPUs."""
import ctypes as C

import numpy as np
import pytest
import torch

import oracle as orc
from spalinalg_b200 import dist as spd
from tests.test_dist import _t, make_coo, shard_of


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,world,first", [(np.float64, 2, None), (np.float32, 2, None), (np.float64, 3, None),
                                               (np.float32, 3, None), (np.float64, 3, [0, 1, 3])])
def test_spmv_gather_fused_copies_the_peer_slices(dtype, world, first):
    """spl_spmv_gather_fused with x split over `world` buffers, the ranks run one after the other with no folded
    barrier (flag_ptrs NULL, every rank its own `ready` counters): each rank's copy warps pull the peers' slices into
    its full-length x, which must then hold them bit for bit, and its rows must reproduce the oracle SpMV (random
    columns: every block has entries).  Slices of 3 ranks start at odd columns: some take the element path.  `first`
    groups peers 1 and 2 into one block."""
    import spalinalg_b200 as sp
    from spalinalg_b200 import _capi as capi
    ctx = sp.default_context()
    n = 20000
    rng = np.random.default_rng(4)
    r, c, v = make_coo(n, n, 240000, 23, dtype)
    ptr, ind, val = orc.compress_from_coo(n, n, orc.make_triplets(r, c, v), "row")
    x = rng.standard_normal(n).astype(dtype)
    yw = orc.csr_spmv(n, ptr, ind, val, x)
    scale = orc.csr_spmv(n, ptr, ind, np.abs(val), np.abs(x))
    starts = spd.partition_starts(n, world)
    slices = [_t(x[starts[g]:starts[g + 1]], dtype) for g in range(world)]
    st = (C.c_uint64 * (world + 1))(*starts)
    sl = (C.c_void_p * world)(*[s.data_ptr() for s in slices])
    first = first or list(range(world + 1))
    bf = (C.c_uint32 * len(first))(*first)
    code = capi.SPL_F32 if dtype == np.float32 else capi.SPL_F64
    tol = 1e-12 if dtype == np.float64 else 1e-5
    for g in range(world):
        lp, li, lv = shard_of((ptr, ind, val), starts, g)
        nloc = starts[g + 1] - starts[g]
        lay = spd.gather_block_layout(torch, _t(lp, np.int64), _t(li, np.int32), _t(lv, dtype), starts, g, first)
        x_full = torch.full((n,), float("nan"), dtype=slices[0].dtype, device="cuda")
        y = torch.full((nloc,), 7.0, dtype=slices[0].dtype, device="cuda")
        ready = torch.zeros(capi.SPL_MAX_PEERS, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        ctx.check(ctx._lib.spl_spmv_gather_fused(
            ctx._h, code, nloc, world, g, C.cast(st, C.c_void_p), C.cast(sl, C.c_void_p), len(first) - 1,
            C.cast(bf, C.c_void_p), C.c_void_p(lay["bptr"].data_ptr()), lay["stride"],
            C.cast((C.c_uint32 * 5)(*lay["caps"]), C.c_void_p), C.c_void_p(lay["bind"].data_ptr()),
            C.c_void_p(lay["bval"].data_ptr()), C.c_void_p(x_full.data_ptr()), C.c_void_p(y.data_ptr()),
            C.c_void_p(ready.data_ptr()), 1, len(li), None, 0, 0, None))
        ctx.sync()
        t = C.c_int()
        ctx.check(ctx._lib.spl_peer_barrier_status(ctx._h, C.byref(t)))    # no stage overrun poisoned y
        got_x = x_full.cpu().numpy()
        peers = np.ones(n, dtype=bool)
        peers[starts[g]:starts[g + 1]] = False                            # the own slice is read in place
        assert got_x[peers].tobytes() == x[peers].tobytes()
        got = y.cpu().numpy()
        assert np.all(np.abs(got - yw[starts[g]:starts[g + 1]]) <= tol * scale[starts[g]:starts[g + 1]] + 1e-300)
