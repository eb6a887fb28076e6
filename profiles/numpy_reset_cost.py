"""Cost of numpy-mode placements (``reset_rng="numpy"``) against the default Philox placements on one GPU.

Two envs with identical seeded starts, one per mode, are timed in the same process, alternating region by region
(CUDA events around each region; median of the regions).  Workloads:

* ``headline``: README config, 1,048,576 envs, greedy, float32 rows, fused launches of 20 steps (``bench.py``'s
  headline), after a warm-up long enough that the episodes are spread over all phases (resets every step);
* ``none_waiting``: the same envs without observations, one launch per step with the waiting policy — the
  instruction-bound mode in which resets were already about a quarter of the time (DESIGN.md §3.3).

Prints one JSON line per workload (with the GPU's name and power limit) and, with ``--out``, appends them there.
Usage: python profiles/numpy_reset_cost.py [--envs N] [--regions 5] [--out FILE]
"""

from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]

import torch  # noqa: E402
from cases import readme_config  # noqa: E402

from collectivecrossing_b200 import BatchedCollectiveCrossing  # noqa: E402


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["?, ?"])[0].split(", ")
    return {"gpu": name, "power_limit": power}


def timed(fn, reps: int) -> float:
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end)


def measure(name, obs, run, steps_per_call, calls, warm_calls, n, regions):
    envs = {}
    for mode in ("philox", "numpy"):
        env = BatchedCollectiveCrossing(readme_config(), n, "cuda:0", seed=7, obs_dtype=obs, reset_rng=mode)
        env.reset_seeded(torch.arange(n, dtype=torch.int64, device="cuda:0"))
        for _ in range(warm_calls):
            run(env)
        envs[mode] = env
    ms = {m: [] for m in envs}
    for _ in range(regions):
        for mode, env in envs.items():
            ms[mode].append(timed(lambda: run(env), calls) / (calls * steps_per_call))
    for env in envs.values():
        env.check_error()
    med = {m: statistics.median(v) for m, v in ms.items()}
    return {"workload": name, "envs": n, "ms_per_step": med, "regions_ms_per_step": ms,
            "numpy_over_philox": med["numpy"] / med["philox"], "kernel": {m: e.last_kernel_name for m, e in envs.items()}}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--regions", type=int, default=5)
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    info = gpu_info()
    rows = [
        measure("headline", "float32", lambda e: e.rollout_trajectory(20, policy="greedy"), 20, 10, 15, a.envs, a.regions),
        measure("none_waiting", "none", lambda e: e.step(policy="waiting"), 1, 200, 300, a.envs, a.regions),
    ]
    for r in rows:
        line = json.dumps({**r, **info})
        print(line)
        if a.out:
            with open(a.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
