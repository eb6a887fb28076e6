"""Writes real float32 observation rows for compressible_write_probe.cu: N README envs stepped by the C oracle
(greedy policy, auto-reset) and observed after STEPS steps, as raw [N, 8, 38] float32.
    python profiles/probes/oracle_rows.py OUT [N=32768] [STEPS=37]"""
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[2]
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]

import numpy as np  # noqa: E402

import oracle  # noqa: E402
from cases import readme_config  # noqa: E402
from collectivecrossing_b200 import _abi  # noqa: E402
from collectivecrossing_b200.lowering import lower_config  # noqa: E402

out = sys.argv[1]
n = int(sys.argv[2]) if len(sys.argv) > 2 else 32768
steps = int(sys.argv[3]) if len(sys.argv) > 3 else 37
envs = oracle.OracleEnvs(lower_config(readme_config()), n, seed=2026)
envs.reset(obs_dtype=_abi.OBS_FP32)
for _ in range(steps):
    r = envs.step(policy="greedy", auto_reset=True, obs_dtype=_abi.OBS_FP32)
rows = np.ascontiguousarray(r["obs"], np.float32)
words = rows.view(np.uint32)
print(f"{n} envs x {rows.shape[1]} agents x {rows.shape[2]} floats after {steps} greedy steps: "
      f"{len(np.unique(words))} distinct words, low 20 bits zero in all: {bool(np.all(words & 0xFFFFF == 0))}, "
      f"zero bytes {np.mean(rows.view(np.uint8) == 0):.3f}, all-zero 32 B sectors {np.mean(np.all(rows.view(np.uint8).reshape(-1, 32) == 0, axis=1)):.4f}")
rows.tofile(out)
