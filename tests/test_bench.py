"""CPU checks of bench.py's host logic: the --dump-outputs sample and the argument checks."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def _load(path):
    return {n[:-4]: np.load(os.path.join(path, n)) for n in sorted(os.listdir(path))}


def test_dump_is_a_fixed_bounded_sample_of_the_outputs(tmp_path):
    rng = np.random.default_rng(1)
    n = (1 << 20) + 3
    out = rng.integers(0, 256, (n, 32), np.uint8); st = rng.integers(0, 6, n, np.uint8)
    bench.dump_outputs(str(tmp_path / "a"), out, st)
    d = _load(str(tmp_path / "a"))
    assert sorted(d) == ["out", "rows", "status"]
    assert (d["out"].dtype, d["status"].dtype, d["rows"].dtype) == (np.float32, np.float32, np.float64)
    assert sum(os.path.getsize(str(tmp_path / "a" / f)) for f in os.listdir(str(tmp_path / "a"))) <= 64 << 20
    idx = d["rows"].astype(np.int64)
    assert len(idx) == bench.DUMP_ROWS and (np.diff(idx) > 0).all() and idx[0] >= 0 and idx[-1] < n
    assert (d["out"] == out[idx]).all() and (d["status"] == st[idx]).all()
    # the same rows are sampled whatever the outputs are
    bench.dump_outputs(str(tmp_path / "b"), np.zeros_like(out), np.zeros_like(st))
    assert (_load(str(tmp_path / "b"))["rows"] == d["rows"]).all()


def test_dump_of_a_small_batch_keeps_every_row(tmp_path):
    out = np.arange(1000 * 32).astype(np.uint8).reshape(1000, 32); st = (np.arange(1000) % 6).astype(np.uint8)
    bench.dump_outputs(str(tmp_path), out, st)
    d = _load(str(tmp_path))
    assert (d["rows"] == np.arange(1000)).all() and (d["out"] == out).all() and (d["status"] == st).all()


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bad_arguments_are_refused_before_any_work(argv):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "error" in r.stderr and r.stdout == ""
