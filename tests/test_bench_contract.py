"""bench.py's command line: the reference arm (`--impl reference`) runs the CPU oracle on a small sample and prints
one JSON line of a fixed shape, `--steps` sets the number of timed steps, and (on a GPU) `--dump-outputs` writes the
outputs of the last timed step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_contract():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1",
                          "--steps", "1", "--warmup", "1", "--ref-cells", "20000"], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "cells/s/iter" and d["higher_is_better"] is True
    assert d["metric"].startswith("cells/sec/Harmony-iteration")
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["n_gpus"] == 1
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and abs(cb["value"] - d["value"]) < 1e-6 * d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "cells/s/iter", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_steps_sets_the_number_of_timed_steps():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1",
                          "--steps", "4", "--ref-cells", "20000"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][0])
    assert d["steps"] == 4
    for bad in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + bad, capture_output=True, text=True,
                             timeout=120, cwd=ROOT)
        assert out.returncode == 2 and out.stdout == "", bad


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    """--dump-outputs: the caller-visible state after the timed steps, float32/float64 .npy files, under 64 MB."""
    n, d, K = 40_000, 50, 100
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1",
                          "--cells-per-gpu", str(n), "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][0])
    assert line["steps"] == 3
    files = sorted(os.listdir(tmp_path))
    assert files == ["R.npy", "Y.npy", "Z_corr.npy", "objective_harmony.npy"]
    assert sum(os.path.getsize(tmp_path / f) for f in files) <= 64 << 20
    a = {f[:-4]: np.load(tmp_path / f) for f in files}
    assert all(v.dtype in (np.float32, np.float64) and np.all(np.isfinite(v)) for v in a.values())
    cells = min(n, 32_768)
    assert a["Z_corr"].shape == (d, cells) and a["R"].shape == (K, cells) and a["Y"].shape == (d, K)
    assert a["objective_harmony"].shape == (1,)
    np.testing.assert_allclose(a["R"].sum(axis=0), 1.0, atol=1e-4)
