"""bench.py --dump-outputs: the outputs of the last timed pass as .npy files, identical from run to run with the same
arguments, so that two builds of the project can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROW_BYTES = (16 + 26 + 576) * 8  # stats, x, P of one filter


def test_dump_rows_is_a_fixed_sample_within_the_budget():
    import bench

    assert bench.dump_rows(4096, ROW_BYTES, 64 << 20) is None  # the default batch is written whole
    n = 1 << 20
    rows = bench.dump_rows(n, ROW_BYTES, 64 << 20)
    assert len(rows) * ROW_BYTES <= 64 << 20 and len(rows) == (64 << 20) // ROW_BYTES
    assert np.all(np.diff(rows) > 0) and rows[0] >= 0 and rows[-1] < n
    assert np.array_equal(rows, bench.dump_rows(n, ROW_BYTES, 64 << 20))


@pytest.mark.gpu
def test_bench_dump_outputs_are_reproducible(tmp_path):
    n, steps = 96, 2

    def run(d):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--filters",
                            str(n), "--no-cpu-baseline", "--no-configs", "--dump-outputs", str(d)],
                           cwd=tmp_path, capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-2000:]
        line = json.loads(p.stdout)  # stdout is the one JSON line
        assert line["steps"] == steps
        return {k: np.load(d / f"{k}.npy") for k in ("stats", "stats_sum", "x", "P")}

    a, b = run(tmp_path / "a"), run(tmp_path / "b")
    assert a["stats"].shape == (n, 16) and a["stats_sum"].shape == (16,)
    assert a["x"].shape == (n, 26) and a["P"].shape == (n, 24, 24)
    for k in a:
        assert a[k].dtype == np.float64
        assert np.array_equal(a[k], b[k], equal_nan=True), k
    assert np.all(np.isfinite(a["x"])) and np.all(np.isfinite(a["P"]))
