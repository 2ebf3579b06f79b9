"""bench.py contract pieces that need no GPU: the peaks file, and the CPU arm's JSON line (``--impl reference``)."""
import importlib.util
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_load_peaks_falls_back_key_by_key(tmp_path, monkeypatch):
    b = _bench()
    monkeypatch.setattr(b, "ROOT", str(tmp_path))
    assert b.load_peaks()["source"] == "fallback"
    (tmp_path / "MEASURED_PEAKS.json").write_text(json.dumps({"hbm_gbs": 6700.0, "bf16_tflops": 1600.0}))
    p = b.load_peaks()
    assert p["source"] == "measured" and p["hbm_gbs"] == 6700.0 and p["bf16_tflops_sustained"] == 1600.0
    (tmp_path / "MEASURED_PEAKS.json").write_text(json.dumps({"hbm_gbs": 6700.0, "bf16_tflops": 1600.0, "bf16_tflops_sustained": 1410.0}))
    assert b.load_peaks()["bf16_tflops_sustained"] == 1410.0
    (tmp_path / "MEASURED_PEAKS.json").write_text("{not json")
    assert b.load_peaks() == {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def test_reference_arm_prints_one_contract_line():
    """The CPU arm (oracle port of the reference path) on a tiny bounded sample: one JSON line with the keys the
    driver reads, no GPU launches."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-samples", "64", "--workload", "cfg1"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "mppi_rollout_steps_per_sec" and d["unit"] == "rollout-steps/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0 and d["config"]["workload"].startswith("oderl Pendulum")


def test_rejects_zero_steps_and_dump_outputs_of_the_cpu_arm(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "out")]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120,
                             cwd=ROOT)
        assert out.returncode == 2 and out.stdout == "", (extra, out.stderr[-2000:])
    assert not (tmp_path / "out").exists()


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
