"""bench.py contract.  On the CPU: the reference arm (the reference's own modules when staged under baseline/_ref, else the oracle CPU
port) prints exactly one JSON line on stdout with the agreed keys.  On the GPU: --dump-outputs writes the same arrays every run."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, OMP_NUM_THREADS="4")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "utt/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "utt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


@pytest.mark.gpu
def test_dump_outputs_repeat_run_to_run(tmp_path):
    """--dump-outputs: with the same arguments two runs write the same arrays up to the rounding of one step's atomic reductions"""
    import numpy as np
    runs = []
    for i in range(2):
        d = tmp_path / str(i)
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--batch", "2", "--steps", "2", "--warmup", "0", "--no-extras",
                              "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        runs.append({f[:-4]: np.load(d / f) for f in sorted(os.listdir(d))})
    assert set(runs[0]) == {"generator_loss", "discriminator_loss", "est_audio", "generator_grads", "discriminator_grads"}
    for name, a in runs[0].items():
        b = runs[1][name]
        assert a.dtype == np.float32 and a.shape == b.shape and np.isfinite(a).all() and np.abs(a).max() > 0, name
        err = np.abs(a.astype(np.float64) - b).max() / np.abs(b).max()
        print(f"[dump] {name} {a.shape}: run 1 vs run 2 max-abs / max {err:.3e}")
        assert err <= 1e-4, name


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ""
