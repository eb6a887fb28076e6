"""Generate tests/golden/*.npz by running the UNMODIFIED reference (build container only).

    python tests/golden/make_golden.py

Each file holds, for a handful of envs, the state after ``reset(seed)``, the action stream and
everything ``CollectiveCrossingEnv.step`` returned at every step, in the batched encoding of
``include/ccb200.h`` (see ``oracle/refrun.py:record``).  ``cassette_basic.npz`` /
``cassette_regression.npz`` are the reference's own golden cassettes
(tests/fixtures/trajectories/golden/*.json) converted to the same encoding; the two JSON files are stored
next to them as they are.
The reference cannot travel to the GPU box, these files do.
"""

from __future__ import annotations

import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from cases import GOLDEN_CASES, cassette_config  # noqa: E402

from collectivecrossing_b200 import _abi  # noqa: E402
from oracle import refload, refrun  # noqa: E402

OUT = Path(__file__).resolve().parent


def convert_cassette(path: Path) -> dict:
    """Reference VCR cassette (test_trajectory_vcr.py:40-121 schema; env.step got `active_actions`) -> batched arrays, N = 1."""
    cas = json.loads(path.read_text())
    cfg = cassette_config()
    ids = refrun.agent_ids(cfg)
    A, L, T = len(ids), 6 + 4 * len(ids), len(cas["steps"])
    init = np.array([cas["initial_observations"][i] for i in ids])
    rec = dict(
        init_x=init[None, :, 0].astype(np.int8), init_y=init[None, :, 1].astype(np.int8),
        init_flags=np.full((1, A), _abi.F_ACTIVE, np.uint8), init_step=np.zeros(1, np.int32),
        init_obs=init[None].astype(np.int8),
        actions=np.full((T, 1, A), refrun.WAIT, np.int8), order=np.full((T, 1, A), -1, np.int8),
        reward=np.zeros((T, 1, A), np.float64), agent_flags=np.zeros((T, 1, A), np.uint8),
        agent_info=np.zeros((T, 1, A), np.uint8), env_flags=np.zeros((T, 1), np.uint8), obs=np.zeros((T, 1, A, L), np.int8),
    )
    for t, st in enumerate(cas["steps"]):
        for pos, (i, a) in enumerate(st["active_actions"].items()):
            rec["actions"][t, 0, ids.index(i)] = a
            rec["order"][t, 0, pos] = ids.index(i)
        for k, i in enumerate(ids):
            bits = 0
            if i in st["next_rewards"]:
                bits |= _abi.O_ALIVE_PREV
                rec["reward"][t, 0, k] = st["next_rewards"][i]
            bits |= _abi.O_TERM_VALUE if st["next_terminated"][i] else 0
            bits |= _abi.O_TRUNC_VALUE if st["next_truncated"].get(i, False) else 0
            if i in st["next_observations"]:
                bits |= _abi.O_OBS_PRESENT
                rec["obs"][t, 0, k] = np.array(st["next_observations"][i]).astype(np.int8)
                inf = st["next_infos"][i]
                rec["agent_info"][t, 0, k] = (
                    (_abi.I_IN_TRAM_AREA if inf["in_tram_area"] else 0) | (_abi.I_AT_DOOR if inf["at_door"] else 0)
                    | (_abi.I_ACTIVE if inf["active"] else 0) | (_abi.I_AT_DESTINATION if inf["at_destination"] else 0)
                )
                bits |= _abi.O_ACTIVE if inf["active"] else 0
            rec["agent_flags"][t, 0, k] = bits
        rec["env_flags"][t, 0] = (_abi.E_TERMINATED_ALL if st["next_terminated"]["__all__"] else 0) | (
            _abi.E_TRUNCATED_ALL if st["next_truncated"]["__all__"] else 0
        )
    return rec


def main() -> None:
    if not refload.available():
        raise SystemExit("the reference is not mounted at /root/reference")
    for name, (make_cfg, kw) in GOLDEN_CASES.items():
        cfg = make_cfg()
        kw = dict(kw)
        kw["seeds"] = list(kw["seeds"])
        rec = refrun.record(cfg, **kw)
        got = refrun.replay_with_oracle(cfg, rec)
        refrun.compare(rec, got, what=f"{name}: oracle")
        np.savez_compressed(OUT / f"{name}.npz", seeds=np.array(kw["seeds"], np.int64), **rec)
        print(f"{name}: {rec['actions'].shape} -> {(OUT / (name + '.npz')).stat().st_size / 1024:.0f} KiB")
    gold = refload.REFERENCE_TESTS / "fixtures" / "trajectories" / "golden"
    for src, dst in (("golden_basic_trajectory.json", "cassette_basic"), ("regression_test.json", "cassette_regression")):
        rec = convert_cassette(gold / src)
        np.savez_compressed(OUT / f"{dst}.npz", seeds=np.array([42], np.int64), **rec)
        (OUT / src).write_bytes((gold / src).read_bytes())   # the cassette itself, for tests/test_cassette_cpu.py
        print(f"{dst}: {rec['actions'].shape}")


if __name__ == "__main__":
    main()
