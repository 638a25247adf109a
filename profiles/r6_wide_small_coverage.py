"""Which wide.cu / wide_assemble.cu kernels tests/test_wide_small.py runs.

Runs the module once under torch.profiler with CUDA activities, lists every launched kernel whose name starts
with `wide_` with its template arguments and launch count, and checks the list against the instantiations the
module is meant to reach: the SpMV vector kernel at all six lane counts in f32 and f64, the four lane counts
of the transpose scatter, the five segment-repair shapes with 32- and 64-bit values, and the stitch of
bucketed assembly writing 64-bit pointers.  Exit code 1 if one is missing or a test fails.

    python profiles/r6_wide_small_coverage.py OUT.txt
"""
import collections
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import pytest  # noqa: E402
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

REQUIRED = ([f"wide_spmv_vector_kernel<{t}, {l}>" for t in ("float", "double") for l in (1, 2, 4, 8, 16, 32)]
            + [f"wide_minor_scatter_kernel<{v}, {l}>" for v in ("unsigned int", "unsigned long") for l in (1, 4, 8, 32)]
            + [f"wide_segment_repair_kernel<{v}, {s}>" for v in ("unsigned int", "unsigned long")
               for s in ("8, 2", "16, 2", "32, 2", "32, 4", "32, 8")]
            + ["wide_stitch_ptr_kernel<unsigned long>"])


def main(out_path):
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        rc = pytest.main([os.path.join(ROOT, "tests", "test_wide_small.py"), "-q", "-m", "gpu", "-p", "no:cacheprovider",
                          "--rootdir", ROOT])
    launches = collections.Counter()
    for e in prof.events():
        name = re.sub(r"\((?:unsigned )?(?:int|long)\)", "", e.name)         # <double, (int)16> -> <double, 16>
        m = re.search(r"\b(wide_\w+)(<[^()]*>)?\(", name)
        if m and e.device_type == torch.autograd.DeviceType.CUDA:
            launches[m.group(1) + (m.group(2) or "")] += 1
    missing = [k for k in REQUIRED if k not in launches]
    lines = [f"tests/test_wide_small.py under torch.profiler (CUDA activities) on {torch.cuda.get_device_name(0)}",
             f"pytest exit code: {int(rc)}", "", "wide kernels launched (name<template arguments>: launches):"]
    lines += [f"  {k}: {launches[k]}" for k in sorted(launches)]
    lines += ["", f"required instantiations: {len(REQUIRED)}, missing: {len(missing)}"]
    lines += [f"  MISSING {k}" for k in missing]
    text = "\n".join(lines) + "\n"
    sys.stdout.write(text)
    with open(out_path, "w") as f:
        f.write(text)
    return 0 if rc == 0 and not missing else 1


if __name__ == "__main__":
    sys.exit(main(sys.argv[1]))
