"""C1 (2-D Laplacian 1024^2, f64) products back to back, run from the root of a build tree: one L2-resident copy
(us_1) and four rotating copies (us_4), CUDA events, 7 batches of 400 launches, median and spread; the host time
per call; the median kernel time from torch.profiler (with programmatic dependent launch it includes the overlap
with the product before).  One line per arm (environment settings).
Run: python profiles/r3_c1_pdl.py LABEL '[{"SPL_STREAM_PATTERN": "1"}, {"SPL_STREAM_PATTERN": "0"}]'"""
import json, os, statistics, sys, time
label = sys.argv[1]; arms = json.loads(sys.argv[2])      # build label, list of environment settings (one arm each)
sys.path.insert(0, os.getcwd())
import numpy as np, torch
import spalinalg_b200 as sp
from spalinalg_b200.synthetic_device import stencil_device
stream = torch.cuda.Stream(); torch.cuda.set_stream(stream)
ctx = sp.Context(0, stream.cuda_stream); sp.set_default_context(ctx)
f64 = torch.float64
n, rp, ci, va = stencil_device(torch, [(0, 0), (-1, 0), (1, 0), (0, -1), (0, 1)], 1024, 4.0, -1.0, f64)
mk = lambda: sp.CsrMatrix.from_device_arrays(n, n, ci.numel(), rp.data_ptr(), ci.data_ptr(), va.data_ptr(), np.float64, validate=False, ctx=ctx)
mats = [mk() for _ in range(4)]
xs = [torch.rand(n, device="cuda", dtype=f64) - 0.5 for _ in mats]
ys = [torch.empty(n, device="cuda", dtype=f64) for _ in mats]
def run(copies, reps):
    for i in range(reps):
        k = i % copies
        mats[k].spmv_device(xs[k].data_ptr(), ys[k].data_ptr())
def events(copies, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); a.record(); run(copies, reps); b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / reps * 1e3
for arm in arms:
    for k in ("SPL_STREAM_PATTERN", "SPL_NO_PDL"):
        os.environ.pop(k, None)
    os.environ.update(arm)
    run(4, 20); torch.cuda.synchronize()
    res = {}
    for copies in (1, 4):
        ts = [events(copies, 400) for _ in range(7)]
        res["us_%d" % copies] = round(statistics.median(ts), 3)
        res["spread_%d" % copies] = round((max(ts) - min(ts)) / statistics.median(ts), 4)
    torch.cuda.synchronize(); t0 = time.perf_counter(); run(1, 400); t1 = time.perf_counter(); torch.cuda.synchronize()
    res["host_us_per_call"] = round((t1 - t0) / 400 * 1e6, 3)
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run(1, 200); torch.cuda.synchronize()
    ev = [e for e in prof.events() if "spmv_stream" in e.name]
    if ev:
        d = [e.device_time for e in ev] if hasattr(ev[0], "device_time") else [e.cuda_time for e in ev]
        res["kernel_us_median_prof"] = round(statistics.median(d), 3); res["kernel_count"] = len(d)
        res["kernel_name"] = ev[0].name[:120]
    print(json.dumps({"build": label, "arm": arm, **res}), flush=True)
