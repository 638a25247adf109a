"""A/B of the one-byte value codes of the band kernel (SPL_STREAM_BAND_CODES=1 against =0, which streams the values)
in one process, on config 5 of bench.py (the band with offsets -4..4, n = 1e8, f64: 35 distinct values) and on the
same band with all-distinct values (no codes: both arms run the value kernel, the code route only costs its one-time
check).  Per matrix, arm and batch: CUDA events around LAUNCHES back-to-back products; the arms alternate batch by
batch, each batch after one untimed product.  Reported per arm: median, min and max ms per product, the spread
(max - min) / median, the median kernel time from a torch.profiler run of its own, and the SM clock sampled after the
batches; y of the two arms is compared bit for bit.  The one-time plan cost of the codes (value set, dictionary,
encode) is the host time of the first product with codes on, minus that of a planned one; a torch.profiler run on a
fresh handle of the same matrix splits its device time by kernel.  Bounds: the bytes the
code kernel moves (codes, x windows, y: computed from the format) over the time torch.sum takes to read as many bytes
on the same card, and the shared-memory wavefronts per tile the consumers issue (computed) at the sampled clock.
--sweep: the code kernel on config 5 by SPL_STREAM_STAGES x SPL_STREAM_CTAS.
Run: python profiles/r8_band_codes_ab.py [--sweep] [--batches 7] [--launches 200]"""
import argparse
import json
import os
import re
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from r3_pattern_ab import card, sm_clock  # noqa: E402


def profiled_kernel_ms(torch, fn, reps=50):
    """median device time of the band kernels over `reps` products, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    d = [e.device_time for e in prof.events() if "spmv_band" in e.name]
    names = sorted({re.search(r"spmv_\w+<[^>]*>", e.name).group(0) for e in prof.events()
                    if re.search(r"spmv_\w+<[^>]*>", e.name)})
    return (statistics.median(d) / 1e3 if d else None), names


def read_ms(torch, nbytes, reps=50):
    """ms of torch.sum over nbytes of f64: a plain read of as many bytes"""
    t = torch.ones(nbytes // 8, device="cuda", dtype=torch.float64)
    t.sum()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        t.sum()
    b.record()
    torch.cuda.synchronize()
    del t
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=7)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--sweep", action="store_true", help="code kernel: SPL_STREAM_STAGES x SPL_STREAM_CTAS")
    args = ap.parse_args()
    import numpy as np
    import torch
    import spalinalg_b200 as sp
    from spalinalg_b200.synthetic_device import banded_device
    stream = torch.cuda.Stream()          # products and events on one explicit stream
    torch.cuda.set_stream(stream)
    ctx = sp.Context(0, stream.cuda_stream)
    sp.set_default_context(ctx)
    f64 = torch.float64
    print(json.dumps({"card": card(), "mode": "sweep" if args.sweep else "a/b", "batches": args.batches,
                      "launches_per_batch": args.launches}), flush=True)

    n = 10 ** 8
    rowptr, colind, values = banded_device(torch, n, 0, n, range(-4, 5), f64)
    nnz = colind.numel()
    x = torch.sin(torch.arange(n, device="cuda", dtype=f64) * 1e-3)
    ys = {1: torch.empty(n, device="cuda", dtype=f64), 0: torch.empty(n, device="cuda", dtype=f64)}

    def matrix(vals):
        return sp.CsrMatrix.from_device_arrays(n, n, nnz, rowptr.data_ptr(), colind.data_ptr(), vals.data_ptr(),
                                               np.float64, validate=False, ctx=ctx)

    def product(A, arm):
        os.environ["SPL_STREAM_BAND_CODES"] = str(arm)
        A.spmv_device(x.data_ptr(), ys[arm].data_ptr())

    def batch(A, arm, reps):
        product(A, arm)                                          # untimed: the arm's grid and partition
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(reps):
            product(A, arm)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    def first_then_steady(A):
        os.environ["SPL_STREAM_BAND_CODES"] = "0"
        product(A, 0)
        torch.cuda.synchronize()
        t = time.perf_counter()
        product(A, 1)                                            # plans the codes
        torch.cuda.synchronize()
        first = (time.perf_counter() - t) * 1e3
        steady = []
        for _ in range(5):
            t = time.perf_counter()
            product(A, 1)
            torch.cuda.synchronize()
            steady.append((time.perf_counter() - t) * 1e3)
        return {"first_product_ms": first, "planned_product_ms": statistics.median(steady),
                "plan_cost_ms": first - statistics.median(steady)}

    def plan_kernels(vals):
        """device ms of every kernel the first coded product of a fresh handle launches, from torch.profiler (a run
        of its own: the host-timed plan cost above is taken without the profiler)"""
        from torch.profiler import ProfilerActivity, profile
        B = matrix(vals)
        product(B, 0)                                            # plans the matrix and the value kernel's grid
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            product(B, 1)
            torch.cuda.synchronize()
        ms = {}
        for e in prof.events():
            if e.device_time > 0:
                m = re.search(r"(\w+_kernel|Memset|Memcpy\w*)", e.name)
                k = m.group(1) if m else e.name[:40]
                ms[k] = ms.get(k, 0.0) + e.device_time / 1e3
        del B
        torch.cuda.synchronize()
        return ms

    A = matrix(values)
    c5_plan = first_then_steady(A)
    if not args.sweep:
        c5_plan["device_ms_by_kernel"] = plan_kernels(values)
    # bytes per product, computed from the format: codes (1 B per entry) or values (8 B), x windows (264 elements per
    # 256-row tile), y
    tiles = (n + 255) // 256
    x_bytes, y_bytes = tiles * 264 * 8, n * 8
    bytes_codes, bytes_values = nnz + x_bytes + y_bytes, nnz * 8 + x_bytes + y_bytes

    if args.sweep:
        for stages in (4, 6, 8, 12, 16):
            for ctas in (2, 3, 4):
                os.environ["SPL_STREAM_STAGES"], os.environ["SPL_STREAM_CTAS"] = str(stages), str(ctas)
                batch(A, 1, 10)
                ts = [batch(A, 1, args.launches) for _ in range(args.batches)]
                med = statistics.median(ts)
                print(json.dumps({"sweep": "C5 code kernel", "stages": stages, "ctas_asked": ctas, "ms_median": med,
                                  "spread": (max(ts) - min(ts)) / med, "tbps_of_code_bytes": bytes_codes / med / 1e9,
                                  "sm_clock_after": sm_clock(), "ms_batches": ts}), flush=True)
        return

    def ab(A, what, nbytes):
        for arm in (1, 0):
            batch(A, arm, 10)
        ts = {1: [], 0: []}
        for _ in range(args.batches):
            for arm in (1, 0):
                ts[arm].append(batch(A, arm, args.launches))
        out = {"matrix": what, "same_bits": torch.equal(ys[1], ys[0]), "sm_clock_after_batches": sm_clock()}
        for arm in (1, 0):
            med = statistics.median(ts[arm])
            product(A, arm)
            prof, names = profiled_kernel_ms(torch, lambda: product(A, arm))
            out["codes_%d" % arm] = {"ms_median": med, "ms_min": min(ts[arm]), "ms_max": max(ts[arm]),
                                     "spread": (max(ts[arm]) - min(ts[arm])) / med, "bytes": nbytes[arm],
                                     "tbps": nbytes[arm] / med / 1e9, "kernel_ms_profiler": prof, "kernels": names,
                                     "ms_batches": ts[arm]}
        out["speedup"] = out["codes_0"]["ms_median"] / out["codes_1"]["ms_median"]
        return out

    out = ab(A, "C5 banded9 n=1e8 f64, 35 distinct values", {1: bytes_codes, 0: bytes_values})
    out["plan"] = c5_plan
    print(json.dumps(out), flush=True)
    ok = out["same_bits"]

    # the bounds of the code kernel on C5
    clock = sm_clock()
    rd = read_ms(torch, bytes_codes)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    # shared-memory wavefronts per 256-row tile (f64, K = 9) of the consumers' loop, computed: per entry and warp one
    # for the pattern offset (a broadcast), one for the 32 code bytes, one for the dictionary (7 neighbouring values
    # per warp here), two for 32 x values; the bulk copies write (2592 + 2144) / 128 more
    wf_tile = 8 * 9 * (1 + 1 + 1 + 2) + (2592 + 2144) / 128
    mhz = None
    try:
        mhz = float(clock.split(",")[0].split()[0])
    except (AttributeError, ValueError, IndexError):
        pass
    print(json.dumps({"bounds": "C5 code kernel", "code_route_bytes": bytes_codes,
                      "hbm_read_ms_same_bytes": rd, "hbm_read_tbps": bytes_codes / rd / 1e9,
                      "smem_wavefronts_per_tile": wf_tile, "tiles_per_sm": tiles / sms,
                      "smem_bound_ms": (wf_tile * tiles / sms / (mhz * 1e3)) if mhz else None,
                      "code_kernel_ms_profiler": out["codes_1"]["kernel_ms_profiler"], "sm_clock": clock}), flush=True)
    del A

    # all-distinct values: no codes; both arms run the value kernel
    distinct = 1.0 + torch.arange(nnz, device="cuda", dtype=f64) * 2.0 ** -30        # exact, all different
    B = matrix(distinct)
    b_plan = first_then_steady(B)
    b_plan["device_ms_by_kernel"] = plan_kernels(distinct)
    out = ab(B, "banded9 n=1e8 f64, all values distinct", {1: bytes_values, 0: bytes_values})
    out["plan"] = b_plan
    print(json.dumps(out), flush=True)
    ok = ok and out["same_bits"]
    assert ok, "the two arms differ"


if __name__ == "__main__":
    main()
