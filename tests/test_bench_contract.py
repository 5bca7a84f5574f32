"""bench.py contract (CPU part): the reference arm runs here and prints one well-formed JSON line."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "3", "--ref-envs", "4"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, "exactly one JSON line on stdout"
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "agent_steps_per_sec" and d["unit"] == "agent-slot-steps/s"
    assert d["higher_is_better"] is True and d["steps"] == 3 and d["warmup"] == 3 and d["value"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    e = d["e2e"]
    assert e["value"] == d["value"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    import os
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "3", "--warmup", "3"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_only_for_the_native_step_benchmark(tmp_path):
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode != 0 and "--dump-outputs" in out.stderr and not any(tmp_path.iterdir())


@pytest.mark.gpu
def test_dump_outputs_same_arguments_same_arrays(tmp_path):
    """--dump-outputs: the outputs of the last timed tick as finite float32 / float64 .npy files, at most 64 MB,
    identical from run to run, and those of a later tick when --steps is one more."""
    cmd = [sys.executable, str(ROOT / "bench.py"), "--envs", "64", "--warmup", "2", "--steady-steps", "0", "--no-cpu"]
    dumps = []
    for k, steps in (("a", 5), ("b", 5), ("c", 6)):
        out = subprocess.run(cmd + ["--steps", str(steps), "--dump-outputs", str(tmp_path / k)], capture_output=True, text=True,
                             timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout)["steps"] == steps
        dumps.append({p.stem: np.load(p) for p in sorted((tmp_path / k).glob("*.npy"))})
    a, b, c = dumps
    assert not (np.array_equal(a["obs"], c["obs"]) and np.array_equal(a["actions"], c["actions"])), "--steps 6 dumps tick 6"
    assert {"rewards", "terminated", "truncated", "mask", "info", "info_valid", "episode_done", "actions", "obs"} <= set(a)
    assert sum(p.stat().st_size for p in (tmp_path / "a").glob("*.npy")) <= 64 << 20
    assert a["obs"].shape == (256, a["obs"].shape[1]) and a["mask"].sum() > 0
    for name, x in a.items():
        assert x.dtype in (np.float32, np.float64) and np.isfinite(x).all(), name
        assert np.array_equal(x, b[name]), name


def test_native_arm_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "3", "--warmup", "3"], capture_output=True, text=True,
                         timeout=300, cwd=ROOT)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)
