"""COO -> CSR assembly in buckets of whole majors (wide_assemble.cu), on one GPU, run from the root of a build tree.

1. Config 3 (168 M f32 triplets): the direct 32-bit route, and the bucketed route forced to 2 and 4 buckets with
   SPL_ASSEMBLE_BUCKET_MAX; CUDA events after a warm-up, arms alternating, median of 5; the three outputs compared
   with torch.equal.
2. The scrambled f32 band of n = 2^26, 65 diagonals (4.36 G triplets, one per cell, wide output): assembly time
   by CUDA events (two runs after the config-3 warm-up), Gnnz/s as input triplets per second, then one run under
   torch.profiler for the number of buckets and the device time in the histogram, the compaction, the per-bucket
   assemblies and the stitch.
Card name and power limit are read in the same run.  Run: python profiles/r5_wide_assembly.py"""
import gc, json, os, statistics, subprocess, sys
sys.path.insert(0, os.getcwd())
import numpy as np, torch
import spalinalg_b200 as sp
from spalinalg_b200 import synthetic_device as sd

stream = torch.cuda.Stream(); torch.cuda.set_stream(stream)
ctx = sp.Context(0, stream.cuda_stream); sp.set_default_context(ctx)
KNOB = "SPL_ASSEMBLE_BUCKET_MAX"


def out(**kw):
    print(json.dumps(kw), flush=True)


q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True).stdout.strip().splitlines()
out(card=q[0] if q else "unknown")


def assemble(n, r, c, v):
    return sp.CsrMatrix.from_device_triplets(n, n, r.numel(), r.data_ptr(), c.data_ptr(), v.data_ptr(), np.float32)


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); a.record(stream)
    res = fn()
    b.record(stream); torch.cuda.synchronize()
    return a.elapsed_time(b), res


def arm(knob):
    if knob:
        os.environ[KNOB] = str(knob)
    else:
        os.environ.pop(KNOB, None)


def device_arrays(A):
    p, i, v = A.device_ptrs()
    view = sd.device_view
    return (view(torch, p, A.nrows() + 1, torch.int32), view(torch, i, A.nnz(), torch.int32),
            view(torch, v, A.nnz(), torch.int32))


CATS = (("histogram", ("wide_coo_scan", "wide_max")),
        ("compaction", ("wide_bucket_count", "wide_bucket_scatter", "wide_scan_")),
        ("stitch", ("wide_stitch_ptr", "Memcpy DtoD")),)


def profiled(fn):
    """Device time (ms) per category of one call; per-bucket assembly = every other kernel, memset and copy."""
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn(); torch.cuda.synchronize()
    sums = {k: 0.0 for k, _ in CATS}
    sums["bucket_assembly"] = 0.0
    buckets = 0
    for e in prof.events():
        t = getattr(e, "device_time", None)
        if t is None:
            t = getattr(e, "cuda_time", 0.0)
        if not t or str(getattr(e, "device_type", "")).endswith("CPU"):
            continue
        buckets += "wide_bucket_scatter" in e.name
        for k, keys in CATS:
            if any(s in e.name for s in keys):
                sums[k] += t / 1e3
                break
        else:
            sums["bucket_assembly"] += t / 1e3
    return {k: round(v, 2) for k, v in sums.items()}, buckets, res


# ---- config 3: direct route against 2 and 4 buckets
n3 = 10_000_000
r, c, v = sd.random_uniform_coo_device(torch, n3, 16, 8_000_000, torch.float32, seed=1)
L = r.numel()
arms = [("direct", 0), ("2 buckets", L // 2 + 1000), ("4 buckets", L // 4 + 1000)]
outs = {}
for name, knob in arms:                                    # warm-up of every arm; outputs kept for the comparison
    arm(knob)
    _, A = timed(lambda: assemble(n3, r, c, v))
    outs[name] = A
ref = device_arrays(outs["direct"])
for name, _ in arms[1:]:
    got = device_arrays(outs[name])
    out(config=3, arm=name, nnz=outs[name].nnz(), equal_to_direct=all(torch.equal(a, b) for a, b in zip(got, ref)))
del outs, ref, got, A
gc.collect()
times = {name: [] for name, _ in arms}
for rep in range(5):
    for name, knob in arms:
        arm(knob)
        ms, A = timed(lambda: assemble(n3, r, c, v))
        times[name].append(ms)
        del A
for name, knob in arms:
    arm(knob)
    split, nb, A = profiled(lambda: assemble(n3, r, c, v))
    del A
    ms = statistics.median(times[name])
    out(config=3, arm=name, triplets=L, ms_median=round(ms, 2), ms_all=[round(t, 2) for t in times[name]],
        gnnz_per_s=round(L / ms / 1e6, 2), buckets=nb, profile_ms=split)
arm(0)
del r, c, v
gc.collect(); torch.cuda.empty_cache(); ctx.trim()

# ---- full size: scrambled band, 4.36 G triplets
n, half = 1 << 26, 32
r, c, v, cells = sd.scrambled_band_coo_device(torch, n, half, torch.float32)
torch.cuda.synchronize()
free, _ = torch.cuda.mem_get_info()
out(full_size="band", n=n, diagonals=2 * half + 1, triplets=cells, free_gb_after_input=round(free / 2 ** 30, 1))
for rep in range(2):
    ms, A = timed(lambda: assemble(n, r, c, v))
    out(full_size="band", run=rep, ms=round(ms, 1), gnnz_per_s=round(cells / ms / 1e6, 2), nnz=A.nnz(),
        wide=A.device_ptr64() is not None)
    del A
split, nb, A = profiled(lambda: assemble(n, r, c, v))
out(full_size="band", profiled=True, buckets=nb, profile_ms=split, nnz=A.nnz())
del A
