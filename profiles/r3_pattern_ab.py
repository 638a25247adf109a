"""A/B of the stream SpMV's row-pattern path (SPL_STREAM_PATTERN=1 against =0) in one process, on the
matrices of bench.py: C5 (band, offsets -4..4, n = 1e8, f64), C1 (2-D Laplacian 1024^2, f64; four rotating
copies so every launch reads HBM, and one copy, L2-resident) and C2 (27-point stencil 128^3, f64).  Per arm and
batch: CUDA events around LAUNCHES back-to-back products; the arms alternate batch by batch; reported: median,
min and max ms per product over the batches, the spread (max - min) / median, the median kernel time of a
torch.profiler run of its own per arm, and the SM clock sampled right after the batches.  y of the two arms is
compared bit for bit.  --sweep: C5 with the path on, by SPL_STREAM_STAGES x SPL_STREAM_CTAS.
Run: python profiles/r3_pattern_ab.py [--sweep] [--batches 7] [--launches 200]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else None
    except (OSError, subprocess.SubprocessError):
        return None


def sm_clock():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,clocks_event_reasons.sw_power_cap", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else None
    except (OSError, subprocess.SubprocessError):
        return None


def profiled_kernel_ms(torch, fn, reps=50):
    """median device time of the stream kernel over `reps` products, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(reps):
            fn(i)
        torch.cuda.synchronize()
    d = [e.device_time for e in prof.events() if "spmv_stream_kernel" in e.name]
    return statistics.median(d) / 1e3 if d else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=7)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--sweep", action="store_true", help="C5 only, pattern on: SPL_STREAM_STAGES x SPL_STREAM_CTAS")
    args = ap.parse_args()
    import numpy as np
    import torch
    import spalinalg_b200 as sp
    from spalinalg_b200.synthetic_device import banded_device, stencil_device
    stream = torch.cuda.Stream()          # products and events on one explicit stream (handle 0 would give the
    torch.cuda.set_stream(stream)         # library a stream of its own, outside the events)
    ctx = sp.Context(0, stream.cuda_stream)
    sp.set_default_context(ctx)
    f64 = torch.float64
    print(json.dumps({"card": card(), "mode": "sweep" if args.sweep else "a/b", "batches": args.batches,
                      "launches_per_batch": args.launches}), flush=True)

    def from_arrays(n, rowptr, colind, values):
        return sp.CsrMatrix.from_device_arrays(n, n, colind.numel(), rowptr.data_ptr(), colind.data_ptr(),
                                               values.data_ptr(), np.float64, validate=False, ctx=ctx)

    def ab(name, mats, nbytes):
        n = mats[0].nrows()
        xs = [torch.sin(torch.arange(n, device="cuda", dtype=f64) * 1e-3 + i) for i in range(len(mats))]
        ys = {arm: [torch.empty(n, device="cuda", dtype=f64) for _ in mats] for arm in (1, 0)}

        def batch(arm, reps):
            os.environ["SPL_STREAM_PATTERN"] = str(arm)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            for i in range(reps):
                k = i % len(mats)
                mats[k].spmv_device(xs[k].data_ptr(), ys[arm][k].data_ptr())
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / reps

        for arm in (1, 0):                                       # plan, partition, warm-up of both arms
            batch(arm, 10)
        ts = {1: [], 0: []}
        for _ in range(args.batches):
            for arm in (1, 0):
                ts[arm].append(batch(arm, args.launches))
        clock = sm_clock()
        same = all(torch.equal(p, q) for p, q in zip(ys[1], ys[0]))
        out = {"matrix": name, "kernel": mats[0].spmv_choice(), "algorithmic_bytes": nbytes, "same_bits": same,
               "sm_clock_after_batches": clock}
        for arm in (1, 0):
            med = statistics.median(ts[arm])
            os.environ["SPL_STREAM_PATTERN"] = str(arm)
            prof = profiled_kernel_ms(torch, lambda i: mats[i % len(mats)].spmv_device(
                xs[i % len(mats)].data_ptr(), ys[arm][i % len(mats)].data_ptr()))
            out["pattern_%d" % arm] = {"ms_median": med, "ms_min": min(ts[arm]), "ms_max": max(ts[arm]),
                                       "spread": (max(ts[arm]) - min(ts[arm])) / med,
                                       "algorithmic_gbps": nbytes / med / 1e6, "kernel_ms_profiler": prof,
                                       "ms_batches": ts[arm]}
        out["speedup"] = out["pattern_0"]["ms_median"] / out["pattern_1"]["ms_median"]
        print(json.dumps(out), flush=True)
        assert same, name + ": the two arms differ"

    def spmv_bytes(nnz, n):
        return nnz * 12 + 2 * n * 8                           # as bench.py: values, indices, x and y

    # C5
    n = 10 ** 8
    rowptr, colind, values = banded_device(torch, n, 0, n, range(-4, 5), f64)
    A = from_arrays(n, rowptr, colind, values)
    if args.sweep:
        x, y = torch.sin(torch.arange(n, device="cuda", dtype=f64) * 1e-3), torch.empty(n, device="cuda", dtype=f64)
        os.environ["SPL_STREAM_PATTERN"] = "1"
        for stages in (2, 3, 4):
            for ctas in (1, 2, 3):
                os.environ["SPL_STREAM_STAGES"], os.environ["SPL_STREAM_CTAS"] = str(stages), str(ctas)
                ts = []
                for rep in range(args.batches + 1):
                    reps = 10 if rep == 0 else args.launches
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    torch.cuda.synchronize()
                    a.record()
                    for _ in range(reps):
                        A.spmv_device(x.data_ptr(), y.data_ptr())
                    b.record()
                    torch.cuda.synchronize()
                    if rep:
                        ts.append(a.elapsed_time(b) / reps)
                print(json.dumps({"sweep": "C5 pattern on", "stages": stages, "ctas_asked": ctas,
                                  "ms_median": statistics.median(ts), "spread": (max(ts) - min(ts)) / statistics.median(ts),
                                  "sm_clock_after": sm_clock(), "ms_batches": ts}), flush=True)
        return
    ab("C5 banded9 n=1e8 f64", [A], spmv_bytes(A.nnz(), n))
    del A, rowptr, colind, values
    torch.cuda.empty_cache()
    # C1, four rotating copies (320 MB > L2)
    n, rowptr, colind, values = stencil_device(torch, [(0, 0), (-1, 0), (1, 0), (0, -1), (0, 1)], 1024, 4.0, -1.0, f64)
    A1 = [from_arrays(n, rowptr, colind, values) for _ in range(4)]
    ab("C1 laplace2d 1024^2 f64 (4 rotating copies)", A1, spmv_bytes(A1[0].nnz(), n))
    ab("C1 laplace2d 1024^2 f64 (one copy, L2-resident)", A1[:1], spmv_bytes(A1[0].nnz(), n))
    del A1, rowptr, colind, values
    torch.cuda.empty_cache()
    # C2
    offs = [(a, b, c) for a in (-1, 0, 1) for b in (-1, 0, 1) for c in (-1, 0, 1)]
    n, rowptr, colind, values = stencil_device(torch, offs, 128, 26.0, -1.0, f64)
    A2 = from_arrays(n, rowptr, colind, values)
    ab("C2 stencil27 128^3 f64", [A2], spmv_bytes(A2.nnz(), n))


if __name__ == "__main__":
    main()
