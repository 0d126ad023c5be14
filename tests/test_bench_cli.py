"""bench.py's CLI contract: the reference arm and the loud failure without a GPU on CPU, --dump-outputs on the GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "env_steps_per_sec" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_under_torchrun_env_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=120, env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_gpu_arm_fails_loudly_without_a_gpu():
    import importlib
    sys.path.insert(0, ROOT)
    q = importlib.import_module("q-learning_b200")
    if q.device_count() > 0:
        return
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=300)
    assert res.returncode != 0 and "no CPU fallback" in (res.stderr + res.stdout)


@pytest.mark.gpu
def test_dump_outputs_are_reproducible(tmp_path):
    """--dump-outputs: two runs with the same arguments write the same f32 / f64 arrays of the last timed launch; --steps is the
    number of timed launches."""
    n, k, steps = 256, 16, 7
    args = ["--envs", str(n), "--steps-per-launch", str(k), "--replay-capacity", str(n * 32), "--steps", str(steps), "--warmup", "2",
            "--no-extra", "--no-cpu-baseline"]
    runs = []
    for i in range(2):
        out = tmp_path / str(i)
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args + ["--dump-outputs", str(out)],
                             capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-2000:]
        line = json.loads(res.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps and line["gpu_launches"] == steps
        runs.append({f.name: np.load(f) for f in out.iterdir()})
    a, b = runs
    assert sorted(a) == sorted(b) and {"reward.npy", "done.npy", "obs.npy", "state_ball_cx.npy", "state_bricks_hi.npy"} <= set(a)
    assert sum(x.nbytes for x in a.values()) < 64 << 20
    for name in a:
        assert a[name].dtype in (np.float32, np.float64), name
        assert np.array_equal(a[name], b[name], equal_nan=True), name
    assert a["reward.npy"].shape == a["done.npy"].shape == (k, n) and a["obs.npy"].shape == (n, 4, 84, 84)
    assert set(np.unique(a["done.npy"]).tolist()) <= {0.0, 1.0} and set(np.unique(a["obs.npy"]).tolist()) <= {0.0, 96.0, 236.0, 255.0}
    assert a["obs.npy"].any() and a["state_episode_step.npy"].max() > 0
