"""CPU: the driver-facing contract of bench.py that can be checked without a GPU — the reference arm (`--impl reference`)
prints ONE JSON line with the required keys, and under a multi-rank launch only rank 0 prints."""
import json
import os
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
REQUIRED = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"}


def _run(env_extra=None):
    env = dict(os.environ, **(env_extra or {}))
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--workload", "tiny", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, env=env, cwd=str(ROOT))
    assert r.returncode == 0, r.stderr[-2000:]
    return [ln for ln in r.stdout.splitlines() if ln.startswith("{")]


def test_reference_arm_prints_one_contract_line():
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert REQUIRED <= set(d)
    assert d["impl"] == "reference" and d["unit"] == "steps/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and "workload" in d["config"]


def test_reference_arm_other_ranks_stay_silent():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == []


def test_dump_outputs_writes_float_arrays_and_samples_past_the_budget(tmp_path):
    """`--dump-outputs`: float32 for floating outputs, exact float64 for integer ones; past the byte budget a fixed, seeded
    sample of each array's elements (the same positions in every run)."""
    import numpy as np
    import torch
    import bench
    vel = torch.randn(2, 64, 8, generator=torch.Generator().manual_seed(0)).to(torch.bfloat16)
    arrays = {"velocity": vel, "moe_loss": torch.tensor(0.25), "expert_counts": torch.tensor([3, 0, 5], dtype=torch.int32)}

    def dump(name, **kw):
        bench.dump_outputs(str(tmp_path / name), arrays, **kw)
        return {f.stem: np.load(f) for f in (tmp_path / name).glob("*.npy")}

    full = dump("full")
    assert set(full) == set(arrays)
    assert full["velocity"].dtype == np.float32 and np.array_equal(full["velocity"], vel.float().numpy())
    assert full["moe_loss"].dtype == np.float32 and full["moe_loss"] == 0.25
    assert full["expert_counts"].dtype == np.float64 and full["expert_counts"].tolist() == [3.0, 0.0, 5.0]
    a, b = dump("a", budget=1024), dump("b", budget=1024)
    assert sum(v.nbytes for v in a.values()) <= 1024
    assert 0 < a["velocity"].size < vel.numel() and np.isin(a["velocity"], full["velocity"]).all()
    assert all(np.array_equal(a[k], b[k]) for k in a)


def test_steps_below_one_and_dump_outputs_of_the_reference_arm_are_refused():
    for extra in (["--steps", "0"], ["--dump-outputs", "unused"]):
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--workload", "tiny", *extra],
                           capture_output=True, text=True, timeout=600, cwd=str(ROOT))
        assert r.returncode == 2 and "error" in r.stderr, (extra, r.stderr[-2000:])
