"""bench.py --dump-outputs on the CUDA path: the same arguments give the same seeded inputs and therefore the same
outputs, bit for bit, which is what makes the dumps of two builds comparable."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = ["--gpus", "1", "--steps", "2", "--warmup", "1", "--samples-per-gpu", "6", "--points", "2048", "--inits", "4",
        "--no-configs", "--no-cpu-baseline"]


def run_bench(out_dir):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *ARGS, "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-3000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    return {n[:-4]: np.load(os.path.join(out_dir, n)) for n in sorted(os.listdir(out_dir))}


def test_dump_outputs_are_reproducible(cuda, tmp_path):
    a = run_bench(tmp_path / "a")
    b = run_bench(tmp_path / "b")
    assert sorted(a) == ["P", "best", "cost", "costs", "degenerate", "init", "init_y_angle", "n_pts", "params", "stats"]
    for name in a:
        assert a[name].dtype in (np.float32, np.float64) and a[name].shape[0] == 6, name
        np.testing.assert_array_equal(a[name], b[name], err_msg=name)
    live = a["degenerate"] == 0                          # a degenerate cloud reports cost 1e4, not one of its solves
    best = a["best"].astype(np.int64)
    np.testing.assert_array_equal(a["cost"][live], a["costs"][np.arange(6), best][live])
