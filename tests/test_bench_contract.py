"""bench.py contract: the reference arm (the restated CPU path on the host cores) runs within its time budget and prints ONE
JSON line with the keys the benchmark reports; the GPU arm refuses to run without a CUDA device, and on one times exactly
--steps steps and dumps the state they leave with --dump-outputs."""
import json
import os
import subprocess
import sys

import pytest

from tests.helpers import ROOT


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ)
    env.pop("RANK", None)
    env.pop("WORLD_SIZE", None)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "leapfrog_steps_per_sec" and d["unit"] == "steps/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("cfg2") and d["config"]["ny"] == 200 and d["config"]["nfreq"] == 30


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=120, env=env, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_gpu_arm_refuses_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and "no CUDA device" in (out.stderr + out.stdout)


@pytest.mark.gpu
def test_gpu_arm_dumps_the_state_of_its_last_timed_step(tmp_path):
    """Two runs with the same arguments time --steps steps each and dump the same chain state; one more step moves it."""
    import numpy as np
    from hmcmt2d_b200.synthetic import AIR

    def run(steps, d):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                              "--no-strong-scaling", "--no-cpu-baseline", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
        assert line["steps"] == steps and line["validated"] is True
        files = sorted(os.listdir(d))
        assert files == ["model.npy", "momentum.npy"]
        assert sum(os.path.getsize(d / f) for f in files) <= 64 << 20
        arrays = {f: np.load(d / f) for f in files}
        for a in arrays.values():
            assert a.dtype == np.float64 and a.shape == (1, line["config"]["ny"] * (line["config"]["nz"] - len(AIR))) and np.isfinite(a).all()
        return arrays

    a, b, c = run(2, tmp_path / "a"), run(2, tmp_path / "b"), run(3, tmp_path / "c")
    for f in a:
        assert np.array_equal(a[f], b[f]), f
        assert not np.array_equal(a[f], c[f]), f
