"""-m gpu: bench.py --dump-outputs writes what the headline leg's last timed step returned, from inputs that are the
same in every run with the same arguments (a small shape; the legs that do not feed the dump are skipped)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                        "--warmup", "3", "--B", "2", "--M", "4096", "--skip-cpu", "--skip-module", "--skip-training",
                        "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    line = json.loads(lines[0])
    assert line["steps"] == steps and line["e2e"]["steps"] == steps
    out = np.load(os.path.join(out_dir, "attention_out.npy"))
    assert sorted(os.listdir(out_dir)) == ["attention_out.npy"]
    assert out.dtype == np.float32 and out.shape == (2, line["config"]["N"], line["config"]["d"])
    assert np.isfinite(out).all() and np.abs(out).max() > 0
    return out


def test_dump_outputs_are_reproducible(tmp_path):
    a = _bench(tmp_path / "a", 2)
    b = _bench(tmp_path / "b", 5)
    # same seeded q/k/v in both runs: equal up to bf16 rounding of differently ordered sums (independent draws would
    # differ by the size of the outputs themselves)
    assert np.abs(a - b).max() <= 1e-2 * np.abs(a).max()
