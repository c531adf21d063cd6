"""bench.py contract pieces that need no GPU: the reference (CPU) arm prints exactly ONE JSON line on stdout with the
keys the driver reads, and anything a library writes to file descriptor 1 ends up on stderr instead."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--points", "2048", "--inits", "4"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, p.stdout[:500]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] and d["unit"] and d["higher_is_better"] is True
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["gpu_launches"] == 0


def test_dump_outputs_writes_float_arrays_within_the_size_cap(tmp_path, monkeypatch):
    import bench
    rng = np.random.default_rng(0)
    arrays = {"P": rng.standard_normal((1000, 4, 4)), "best": rng.integers(0, 60, 1000, dtype=np.int32),
              "xyz": rng.standard_normal((1000, 3)).astype(np.float32)}
    bench.dump_outputs(str(tmp_path / "whole"), arrays)                  # under the cap: everything, integers exact
    assert sorted(os.listdir(tmp_path / "whole")) == ["P.npy", "best.npy", "xyz.npy"]
    for name, a in arrays.items():
        got = np.load(tmp_path / "whole" / (name + ".npy"))
        assert got.dtype in (np.float32, np.float64) and np.array_equal(got, a)
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 1 << 16)              # over the cap: the same seeded sample every time
    bench.dump_outputs(str(tmp_path / "a"), arrays)
    bench.dump_outputs(str(tmp_path / "b"), arrays)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["P.npy", "best.npy", "sample_rows.npy", "xyz.npy"]
    total = 0
    for name in names:
        a, b = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b)
        total += a.nbytes
    assert total <= bench.DUMP_MAX_BYTES
    rows = np.load(tmp_path / "a" / "sample_rows.npy").astype(np.int64)
    assert 0 < len(rows) < 1000
    for name, a in arrays.items():
        np.testing.assert_array_equal(np.load(tmp_path / "a" / (name + ".npy")), a[rows])


def test_dump_outputs_is_refused_where_nothing_is_registered_on_the_gpu():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", "x"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert p.returncode == 2 and "--dump-outputs" in p.stderr
