"""The reference arm of bench.py runs without a GPU: one JSON line with the keys the contract names."""

import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "agent_steps_per_sec" and d["unit"] == "agent-steps/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    # the unmodified reference where it is mounted or staged (oracle/_ref/reference.zip), else the oracle's Python port
    from oracle import refload

    assert d["cpu_baseline"]["kind"] == ("reference" if refload.available() else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_other_ranks_of_the_reference_arm_exit_silently():
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=60, cwd=ROOT, env={**__import__("os").environ, "RANK": "1", "WORLD_SIZE": "2"})
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.parametrize("args", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_refuses_arguments_it_cannot_honour(args):
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=60, cwd=ROOT)
    assert out.returncode == 2 and out.stdout == "" and "error:" in out.stderr


DUMP_TWICE = """
import sys
from pathlib import Path
import torch
import bench
n, out = 200_000, Path(sys.argv[1])
env = torch.arange(n, dtype=torch.float32)
outputs = {"obs": env[:, None, None].expand(n, 8, 38).contiguous(), "reward": env[:, None].expand(n, 8).contiguous(),
           "env_flags": env.clone(), "agent_info": None}
for run in ("a", "b"):
    bench.dump_outputs(out / run, outputs, torch)
"""


def test_dump_sample_keeps_the_same_envs_in_every_output(tmp_path):
    """Outputs above the size limit are cut to one seeded sample of envs, the same for every array and every run.  (In a
    subprocess: torch's worker threads would otherwise be running when later tests fork.)"""
    import numpy as np

    out = subprocess.run([sys.executable, "-c", DUMP_TWICE, str(tmp_path)], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    got = {run: {k: np.load(tmp_path / run / f"{k}.npy") for k in ("obs", "reward", "env_flags")} for run in ("a", "b")}
    assert not (tmp_path / "a" / "agent_info.npy").exists()
    ids = got["a"]["env_flags"]
    assert sum(v.nbytes for v in got["a"].values()) <= 48 * 10**6 and 0 < len(ids) < 200_000
    assert np.all(np.diff(ids) > 0) and ids[-1] > len(ids)       # sorted, distinct, not a prefix
    assert (got["a"]["obs"] == ids[:, None, None]).all() and (got["a"]["reward"] == ids[:, None]).all()
    for k in got["a"]:
        assert np.array_equal(got["a"][k], got["b"][k]), k


def test_committed_bench_record_carries_the_contract():
    """profiles/r2_bench_1gpu.json is a line `python bench.py` printed on a B200: every key of the measurement contract is there and
    the numbers agree with each other (value = units / time, frac = achieved / peak, e2e measured with copies)."""
    import json
    from pathlib import Path

    line = json.loads((Path(__file__).resolve().parents[1] / "profiles" / "r2_bench_1gpu.json").read_text())
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"):
        assert key in line, key
    assert line["metric"] == "agent_steps_per_sec" and line["unit"] == "agent-steps/s" and line["higher_is_better"] is True
    assert line["n_gpus"] == 1 and line["warmup"] >= 3 and line["vs_baseline"] is None and line["scaling"] == "weak"
    assert "workload" in line["config"] and "model" not in line["config"]
    cfg = line["config"]
    units = cfg["envs_total"] * cfg["agents_per_env"]
    assert abs(line["value"] - units / (line["ms_per_step"] * 1e-3)) / line["value"] < 1e-6
    r = line["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["traffic"]
    assert abs(r["achieved"] - r["algorithmic_bytes_per_env_step"] * cfg["envs_total"] / (line["ms_per_step"] * 1e-3) / 1e9) / r["achieved"] < 1e-6
    assert 0.5 < r["traffic"] / r["algorithmic_bytes_per_launch"] < 1.1          # ncu's DRAM bytes against the algorithmic bytes of one launch
    e = line["e2e"]
    assert e["unit"] == line["unit"] and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] < line["value"]
    c = line["cpu_baseline"]
    assert c["kind"] in ("reference", "port") and c["cores"] >= 1 and c["value"] > 0 and c["sample"]
    assert line["gpu_launches"] > 0 and not set(line["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    assert len(line["repetitions"]["ms_per_region"]) >= 5
