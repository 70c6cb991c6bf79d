"""GPU: bench.py end to end on one device at a few steps - --steps sets the number of timed steps, and --dump-outputs
writes the last timed step's loss-kernel outputs and the updated parameters."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dump_outputs(tmp_path):
    T, B, A = 20, 8, 6
    out_dir = tmp_path / "outputs"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "2", "--T", str(T),
           "--B", str(B), "--no_cpu_baseline", "--no_profile", "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == 3 and line["warmup"] == 2
    got = {f[:-4]: np.load(str(out_dir / f)) for f in os.listdir(str(out_dir))}
    assert sorted(got) == sorted(["vs", "pg_advantages", "log_rhos", "behavior_action_log_probs", "target_action_log_probs",
                                  "losses", "grad_logits", "grad_values", "params"])
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in got.values())
    assert got["vs"].shape == (T, B) and got["grad_logits"].shape == (T + 1, B, A) and got["losses"].shape == (4,)
    assert float(got["losses"][3]) == line["final_total_loss"]
    np.testing.assert_allclose(got["losses"][3], got["losses"][:3].sum(), rtol=1e-5, atol=1e-5 * np.abs(got["losses"][:3]).sum())
    assert sum(os.path.getsize(str(out_dir / f)) for f in os.listdir(str(out_dir))) <= 64 << 20
