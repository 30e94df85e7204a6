"""bench.py's reference arm runs on the host cores, so its JSON line can be checked without a
GPU: the keys the driver reads, the bounded sample, and that exactly the requested number of
steps is timed.  --dump-outputs is checked against the oracle in both arms."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_py as O
from ceres_b200 import problems as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line():
    out = subprocess.run(
        [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
         "--warmup", "1", "--scale", "0.005"],
        capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["steps"] == 2 and d["warmup"] == 1
    for key in ("metric", "value", "unit", "n_gpus", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["unit"] == "residual blocks/s" and d["value"] > 0 and d["dtype"] == "f64"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def _check_dump(path):
    """--dump-outputs of the L workload at scale 0.005: every array is the oracle's output for
    the same problem at the written positions, float64, 64 MB at most in all."""
    op = O.OracleProblem(P.bal_shape("L", scale=0.005))
    ok, c_o, r_o, g_o, j_o = op.evaluate(op.initial_state())
    assert ok
    c = np.load(path / "cost.npy")
    assert c.dtype == np.float64 and c.shape == (1,) and abs(c[0] - c_o) <= 1e-10 * c_o
    for name, want, rtol in (("residuals", r_o, 1e-12), ("gradient", g_o, 1e-10),
                             ("jacobian", j_o[:op.num_jacobian_values], 1e-12)):
        got, idx = np.load(path / f"{name}.npy"), np.load(path / f"{name}_index.npy")
        assert got.dtype == np.float64 and got.shape == idx.shape
        idx = idx.astype(np.int64)
        assert np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < want.size
        assert np.max(np.abs(got - want[idx])) <= rtol * np.max(np.abs(want)), name
    # 290 k residuals are written whole; of the 3.5 M Jacobian values, a sample
    assert np.load(path / "residuals.npy").size == r_o.size
    assert np.load(path / "jacobian.npy").size < op.num_jacobian_values
    assert sum(f.stat().st_size for f in path.iterdir()) <= 64 << 20
    return float(c[0])


def test_reference_arm_dumps_its_last_step(tmp_path):
    out = subprocess.run(
        [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
         "--warmup", "1", "--scale", "0.005", "--dump-outputs", str(tmp_path)],
        capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    _check_dump(tmp_path)


@pytest.mark.gpu
def test_gpu_arm_dumps_its_last_step(tmp_path):
    out = subprocess.run(
        [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2",
         "--warmup", "1", "--scale", "0.005", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
        capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["steps"] == 2 and d["cost"] == _check_dump(tmp_path)


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run(
        [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
         "--steps", "1", "--warmup", "1", "--scale", "0.005"],
        capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
