"""bench.py --dump-outputs: the timed path's results, identical from run to run, for comparing two builds."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c2", "--steps", str(steps), "--warmup", "3",
                          "--no-e2e", "--no-cpu", "--no-refgpu", "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    return json.loads(res.stdout.strip().splitlines()[-1])


def test_bench_dump_outputs_are_the_timed_steps_and_reproducible(tmp_path):
    steps = 7
    line = _bench(tmp_path / "a", steps)
    _bench(tmp_path / "b", steps)
    assert line["steps"] == steps
    files = sorted(os.listdir(tmp_path / "a"))
    # c2 runs with lambda_g1 = lambda_d = 1 and no vg / entropy terms
    assert files == ["kl_reg.npy", "main_loss.npy", "mapping.npy", "mapping_rows.npy", "total_loss.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64e6
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype in (np.float32, np.float64) and np.all(np.isfinite(a)), f
        assert np.array_equal(a, b), f
    for f in ("total_loss.npy", "main_loss.npy", "kl_reg.npy"):
        assert np.load(tmp_path / "a" / f).shape == (steps,)
    assert np.load(tmp_path / "a" / "total_loss.npy")[-1] == np.float32(line["parity"]["loss_last"])
    P, rows = np.load(tmp_path / "a" / "mapping.npy"), np.load(tmp_path / "a" / "mapping_rows.npy")
    assert P.shape == (10_000, 1_000) and np.array_equal(rows, np.arange(10_000))    # c2's mapping fits whole
    assert np.allclose(P.sum(axis=1), 1.0, atol=1e-4)
