"""`bench.py --dump-outputs`: the outputs of the last timed step, identical from run to run with the same arguments, and the
same whether the timed steps ran as fused launches or one launch per step."""

import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ROOT = Path(__file__).resolve().parents[1]
NAMES = ("obs", "reward", "agent_flags", "env_flags", "actions")


def run_bench(out_dir, *extra):
    cmd = [sys.executable, str(ROOT / "bench.py"), "--envs", "3000", "--steps", "7", "--warmup", "2", "--reps", "2", "--no-extras",
           "--e2e-steps", "1", "--cpu-seconds", "0.2", "--dump-outputs", str(out_dir), *extra]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 7
    return line, {n: np.load(out_dir / f"{n}.npy") for n in NAMES}


def test_dumped_outputs_repeat_and_do_not_depend_on_the_launch_shape(tmp_path):
    line, a = run_bench(tmp_path / "a")
    assert line["roofline"]["steps_per_launch"] == 7 and line["gpu_launches"] == 1     # the 7 timed steps: one fused launch
    _, b = run_bench(tmp_path / "b")
    # one launch per step; the 7 more warm-up steps stand for the fused launch that warms the fused path above
    single, c = run_bench(tmp_path / "c", "--steps-per-launch", "1", "--warmup", "9")
    assert single["gpu_launches"] == 7
    assert a["obs"].shape == (3000, 8, 38) and a["reward"].shape == (3000, 8) and a["env_flags"].shape == (3000,)
    for n in NAMES:
        assert a[n].dtype == np.float32, n
        assert np.array_equal(a[n], b[n]) and np.array_equal(a[n], c[n]), n
    assert (a["agent_flags"] != 0).any() and (a["actions"] != 0).any()


def test_large_outputs_are_dumped_as_a_sample(tmp_path):
    _, a = run_bench(tmp_path / "a", "--envs", "100000", "--steps-per-launch", "1")
    _, b = run_bench(tmp_path / "b", "--envs", "100000", "--steps-per-launch", "1")
    total = sum(v.nbytes for v in a.values())
    assert total <= 64 * 10**6 and a["obs"].shape[0] == a["reward"].shape[0] == a["env_flags"].shape[0] < 100000
    for n in NAMES:
        assert np.array_equal(a[n], b[n]), n
