"""bench.py --dump-outputs: the rows it writes are fixed and bounded (CPU), and what it writes is the product of
the timed steps, checked against the oracle (GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
import oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_rows_are_fixed_and_bounded():
    n = 10 ** 8
    rows = bench.dump_rows(n)
    assert np.array_equal(rows, bench.dump_rows(n))                    # the same sample in every run
    assert np.all(np.diff(rows) > 0) and rows[0] == 0 and rows[-1] == n - 1
    assert np.array_equal(rows[:4096], np.arange(4096)) and np.array_equal(rows[-4096:], np.arange(n - 4096, n))
    assert 2 * 8 * rows.size <= 64 << 20                              # y and its row numbers, f64
    assert np.array_equal(bench.dump_rows(bench.DUMP_ROWS), np.arange(bench.DUMP_ROWS))


@pytest.mark.gpu
def test_dump_outputs_is_the_product_of_the_timed_steps(tmp_path):
    """banded9_1e7_f64: 10^7 rows, more than DUMP_ROWS, so y is sampled.  A[i, i+d] = 1/(1+|d|) + (i mod 7) 1e-3
    for |d| <= 4, x_j = sin(j 1e-3): the sampled rows' product is restated on the CPU by the oracle."""
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1",
                        "--workload", "banded9_1e7_f64", "--no-extras", "--dump-outputs", str(out)],
                       cwd=tmp_path, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["config"]["workload"] == "banded9_1e7_f64"
    n = 10 ** 7
    y, rows = np.load(out / "y.npy"), np.load(out / "y_rows.npy")
    assert sorted(os.listdir(out)) == ["y.npy", "y_rows.npy"]
    assert y.dtype == np.float64 and rows.dtype == np.float64 and y.shape == rows.shape
    assert np.array_equal(rows, bench.dump_rows(n).astype(np.float64))
    # the sampled rows as a CSR matrix of their own (global columns), multiplied by the oracle
    i = rows.astype(np.int64)
    cols = i[:, None] + np.arange(-4, 5)[None, :]
    keep = (cols >= 0) & (cols < n)
    vals = 1.0 / (1 + np.abs(np.arange(-4, 5)))[None, :] + (i % 7)[:, None] * 1e-3
    ptr = np.concatenate([[0], np.cumsum(keep.sum(1))]).astype(np.uint64)
    ind, val = cols[keep].astype(np.uint64), vals[keep]
    x = np.sin(np.arange(n) * 1e-3)
    want = orc.csr_spmv(len(i), ptr, ind, val, x)
    scale = orc.csr_spmv(len(i), ptr, ind, np.abs(val), np.abs(x))
    assert np.all(np.abs(y - want) <= 1e-12 * scale + 1e-300)
