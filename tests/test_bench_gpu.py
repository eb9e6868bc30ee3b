"""bench.py on the device: `--dump-outputs DIR` writes what the last timed step returned, and the same arguments give the same
inputs, so runs with different step counts store the same outputs (up to the kernels' run-to-run rounding)."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "tiny", "--steps", str(steps), "--warmup", "0",
                        "--no-cpu-baseline", "--no-eager-baseline", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    return line, {f.stem: np.load(f) for f in out_dir.glob("*.npy")}


def test_dump_outputs_hold_the_last_timed_step_and_repeat_across_runs(tmp_path):
    line1, a = _bench(tmp_path / "a", 1)
    line3, b = _bench(tmp_path / "b", 3)
    assert line1["steps"] == 1 and line3["steps"] == 3
    assert set(a) == set(b) == {"velocity", "moe_loss", "expert_counts"}
    v = a["velocity"]
    assert v.dtype == np.float32 and v.shape == (1, 256, 64) and np.isfinite(v).all() and np.abs(v).max() > 0
    assert a["expert_counts"].dtype == np.float64 and a["expert_counts"].sum() > 0
    assert np.linalg.norm(v - b["velocity"]) <= 1e-3 * np.linalg.norm(b["velocity"])
    assert abs(float(a["moe_loss"]) - float(b["moe_loss"])) <= 1e-3 * abs(float(b["moe_loss"])) + 1e-6
