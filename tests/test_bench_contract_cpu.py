"""The reference arm of bench.py (`--impl reference`: the oracle port of CrossAttention.forward timed on the host
cores) runs without a GPU; check the one JSON line it prints against the driver's contract."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "1", "--cpu-seconds", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "cross_attn_core_tflops" and d["unit"] == "TFLOP/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["gpu_launches"] == 0
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None
    assert d["config"]["M"] == 65536 and d["config"]["N"] == 512 and d["config"]["B"] == 8
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=300, cwd=ROOT)
    assert r.returncode == 2 and "--steps must be >= 1" in r.stderr


def test_our_arm_refuses_to_run_without_a_gpu():
    import torch

    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--skip-cpu"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)
