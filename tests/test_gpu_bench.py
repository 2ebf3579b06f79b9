"""bench.py --dump-outputs on the GPU: the arrays of the headline's last timed step, the same from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg1", "--steps", str(steps), "--warmup", "3", "--idle", "0",
           "--no-extra", "--no-cpu-baseline", "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-4000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == steps
    return {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


@pytest.mark.gpu
def test_dump_outputs_repeat_with_the_arguments(tmp_path):
    a, b, c = _run(tmp_path / "a", 2), _run(tmp_path / "b", 2), _run(tmp_path / "c", 3)
    K, H, nx, nu = 1000, 20, 3, 1  # config 1: pendulum; every sample is dumped below DUMP_SAMPLES
    shapes = {"action": (nu,), "U": (H, nu), "cost_total": (K,), "omega": (K,), "states": (K, H, nx), "perturbed_action": (K, H, nu),
              "noise": (K, H, nu)}
    assert {k: v.shape for k, v in a.items()} == shapes
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
    assert abs(float(a["omega"].sum()) - 1.0) < 1e-4
    assert np.array_equal(a["noise"], b["noise"])  # the on-device sampler: keyed on the seed and the step count only
    for k in shapes:
        assert np.abs(a[k] - b[k]).max() <= 1e-4 * max(np.abs(a[k]).max(), 1e-30), k
    assert not np.array_equal(a["noise"], c["noise"])  # --steps sets how many steps ran: another step, other noise
