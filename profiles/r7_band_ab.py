"""A/B of the band kernel of the stream SpMV (SPL_STREAM_BAND=1 against =0, which runs the stream kernel's row-pattern
path) in one process, on config 5 of bench.py: the band with offsets -4..4, n = 1e8, f64.  Per arm and batch: CUDA
events around LAUNCHES back-to-back products; the arms alternate batch by batch, and each batch starts with one
untimed product (the two arms run different grids, and the partition is cached for one grid at a time); reported:
median, min and max ms per product over the batches, the spread (max - min) / median, the median kernel time of a
torch.profiler run of its own per arm, the algorithmic bytes over the median time, and the SM clock sampled right
after the batches.  y of the two arms is compared bit for bit.  --sweep: the band kernel by SPL_STREAM_STAGES x
SPL_STREAM_CTAS (the CTAs per SM that fit cap the CTAs asked for).
Run: python profiles/r7_band_ab.py [--sweep] [--batches 7] [--launches 200]"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from r3_pattern_ab import card, sm_clock  # noqa: E402


def profiled_kernel_ms(torch, fn, reps=50):
    """median device time of the SpMV kernel over `reps` products, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    d = [e.device_time for e in prof.events() if "spmv_band_kernel" in e.name or "spmv_stream_kernel" in e.name]
    names = sorted({e.name.split("(")[0] for e in prof.events() if "spmv_" in e.name})
    return (statistics.median(d) / 1e3 if d else None), names


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=7)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--sweep", action="store_true", help="band kernel: SPL_STREAM_STAGES x SPL_STREAM_CTAS")
    args = ap.parse_args()
    import numpy as np
    import torch
    import spalinalg_b200 as sp
    from spalinalg_b200.synthetic_device import banded_device
    stream = torch.cuda.Stream()          # products and events on one explicit stream (handle 0 would give the
    torch.cuda.set_stream(stream)         # library a stream of its own, outside the events)
    ctx = sp.Context(0, stream.cuda_stream)
    sp.set_default_context(ctx)
    f64 = torch.float64
    print(json.dumps({"card": card(), "mode": "sweep" if args.sweep else "a/b", "batches": args.batches,
                      "launches_per_batch": args.launches}), flush=True)

    n = 10 ** 8
    rowptr, colind, values = banded_device(torch, n, 0, n, range(-4, 5), f64)
    A = sp.CsrMatrix.from_device_arrays(n, n, colind.numel(), rowptr.data_ptr(), colind.data_ptr(),
                                        values.data_ptr(), np.float64, validate=False, ctx=ctx)
    nbytes = A.nnz() * 8 + 2 * n * 8      # values, x and y: what the band kernel and the row-pattern path move
    x = torch.sin(torch.arange(n, device="cuda", dtype=f64) * 1e-3)
    ys = {1: torch.empty(n, device="cuda", dtype=f64), 0: torch.empty(n, device="cuda", dtype=f64)}

    def batch(arm, reps):
        os.environ["SPL_STREAM_BAND"] = str(arm)
        A.spmv_device(x.data_ptr(), ys[arm].data_ptr())          # untimed: the arm's grid and partition
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(reps):
            A.spmv_device(x.data_ptr(), ys[arm].data_ptr())
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    if args.sweep:
        for stages in (2, 3, 4):
            for ctas in (2, 3):
                os.environ["SPL_STREAM_STAGES"], os.environ["SPL_STREAM_CTAS"] = str(stages), str(ctas)
                batch(1, 10)
                ts = [batch(1, args.launches) for _ in range(args.batches)]
                med = statistics.median(ts)
                print(json.dumps({"sweep": "C5 band kernel", "stages": stages, "ctas_asked": ctas, "ms_median": med,
                                  "spread": (max(ts) - min(ts)) / med, "algorithmic_tbps": nbytes / med / 1e9,
                                  "sm_clock_after": sm_clock(), "ms_batches": ts}), flush=True)
        return

    for arm in (1, 0):                                           # plan and warm-up of both arms
        batch(arm, 10)
    ts = {1: [], 0: []}
    for _ in range(args.batches):
        for arm in (1, 0):
            ts[arm].append(batch(arm, args.launches))
    clock = sm_clock()
    same = torch.equal(ys[1], ys[0])
    out = {"matrix": "C5 banded9 n=1e8 f64", "kernel": A.spmv_choice(), "algorithmic_bytes": nbytes,
           "same_bits": same, "sm_clock_after_batches": clock}
    for arm in (1, 0):
        med = statistics.median(ts[arm])
        os.environ["SPL_STREAM_BAND"] = str(arm)
        A.spmv_device(x.data_ptr(), ys[arm].data_ptr())
        prof, names = profiled_kernel_ms(torch, lambda: A.spmv_device(x.data_ptr(), ys[arm].data_ptr()))
        out["band_%d" % arm] = {"ms_median": med, "ms_min": min(ts[arm]), "ms_max": max(ts[arm]),
                                "spread": (max(ts[arm]) - min(ts[arm])) / med, "algorithmic_tbps": nbytes / med / 1e9,
                                "kernel_ms_profiler": prof, "kernels": names, "ms_batches": ts[arm]}
    out["speedup"] = out["band_0"]["ms_median"] / out["band_1"]["ms_median"]
    # what a plain stream reaches on this card now: torch.sum over the 7.2 GB of values (one read)
    values.sum()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(50):
        values.sum()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 50
    out["read_reference"] = {"what": "torch.sum over the values (f64)", "bytes": values.numel() * 8, "ms": ms,
                             "tbps": values.numel() * 8 / ms / 1e9, "sm_clock_after": sm_clock()}
    print(json.dumps(out), flush=True)
    assert same, "the two arms differ"


if __name__ == "__main__":
    main()
