"""GPU: `bench.py --dump-outputs DIR` writes what the last timed step returned, the same bits from run to run, and
`--steps` sets how many steps were timed (one more step gives different outputs)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INFO = ("reward", "revenue", "der_cost", "ess_cost", "discomfort_penalty", "voltage_penalty", "cumulative_reward", "solver_failed")


def run_bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "3",
           "--envs-per-gpu", "2048", "--rows", "3000", "--dump-outputs", str(out_dir), "--no-cpu-baseline", "--no-config2",
           "--no-config3", "--no-config4", "--no-obs", "--no-strong", "--no-rollout"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    return {f[:-4]: np.load(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}


def test_bench_dump_outputs(cuda, tmp_path):
    a = run_bench(tmp_path / "a", 4)
    assert set(a) == {"reward", "terminated"} | {f"info_{k}" for k in INFO}
    for name, v in a.items():
        assert v.shape == (2048,) and v.dtype == (np.float32 if name == "terminated" else np.float64), name
    assert np.array_equal(a["reward"], a["info_reward"]) and np.isfinite(a["reward"]).all()
    b = run_bench(tmp_path / "b", 4)
    for name in a:
        assert np.array_equal(a[name], b[name]), name
    c = run_bench(tmp_path / "c", 5)
    assert not np.array_equal(a["info_cumulative_reward"], c["info_cumulative_reward"])
