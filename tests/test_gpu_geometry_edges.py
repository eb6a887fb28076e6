"""GPU: every step kernel against the oracle on the lattices of tests/geometry_edges.py, at and just past each size
limit the kernels dispatch on (small-lattice kernel, the three occupancy paths of the thread-per-env kernel, the
largest lattice).  Seeded random starts with spread phases, ragged env counts, auto-reset, a global env offset above
2**32; state, episode return, reward, both flag bytes, infos, applied actions and rows at every step, then the
statistics.  Every case also asserts which instantiation ran (``expected_kernel``), so a case cannot pass on the wrong
kernel."""

import os
import subprocess
import sys
import zlib
from pathlib import Path

import numpy as np
import pytest
from geometry_edges import LATTICES, OBS_CODE, TPE2_LATTICES, TPE_LATTICES, Case, device_cases, tpe2_off_cases
from helpers import random_states

from collectivecrossing_b200 import _abi
from collectivecrossing_b200.lowering import lower_config

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
ROOT = Path(__file__).resolve().parents[1]
OFFSET = 2**32 + 4093   # both words of the counter-based RNG's env index matter


def make_env(cfg, n, **kw):
    from collectivecrossing_b200 import BatchedCollectiveCrossing

    return BatchedCollectiveCrossing(cfg, n, "cuda:0", **kw)


def _setup(case: Case, **env_kw):
    """Env and oracle of one case from the same seeded start states (phases spread over the episode)."""
    import oracle

    cfg = case.config()
    low = lower_config(cfg)
    key = zlib.crc32(case.id.encode())
    n = 32 * (2 if low.num_agents > 8 else 5) + 1 + key % 31
    rng = np.random.default_rng(key)
    seed = key % 1000
    env = make_env(cfg, n, seed=seed, global_env_offset=OFFSET, obs_dtype=case.obs, auto_reset=True, with_info=True,
                   kernel=case.kernel, **env_kw)
    orc = oracle.OracleEnvs(low, n, seed=seed, global_env_offset=OFFSET)
    x, y, f, s = random_states(cfg, n, rng, step_hi=low.max_steps)
    env.set_state(*(torch.from_numpy(v).cuda() for v in (x, y, f, s)))
    orc.set_state(x, y, f, s)
    return env, orc, rng


def _same_state(env, orc, tag):
    for k, u, v in (("x", env.x, orc.x), ("y", env.y, orc.y), ("flags", env.flags, orc.flags), ("step", env.step_count, orc.step_count),
                    ("episode_return", env.episode_return, orc.episode_return)):
        assert np.array_equal(u.cpu().numpy(), v), f"{tag}: state {k}"


def _same_outputs(out, res, obs, tag):
    for k, u in (("reward", out["reward"]), ("agent_flags", out["agent_flags"]), ("agent_info", out["agent_info"]),
                 ("env_flags", out["env_flags"]), ("actions_out", out["actions"])):
        assert np.array_equal(u.cpu().numpy(), res[k]), f"{tag}: {k}"
    if obs != "none":
        assert np.array_equal(out["obs"].cpu().numpy(), res["obs"]), f"{tag}: rows"


def _same_stats(env, orc):
    st, want = env.stats(), orc.stats.as_dict()
    for k in ("env_steps", "episodes", "terminated_all", "truncated_all", "arrivals", "episode_length_sum"):
        assert st[k] == want[k], (k, st[k], want[k])
    for k in ("episode_return_sum", "reward_sum"):
        assert st[k] == pytest.approx(want[k], rel=1e-9, abs=1e-9), k
    return st


def _step_outputs(out):
    return dict(reward=out.reward, agent_flags=out.agent_flags, agent_info=out.agent_info, env_flags=out.env_flags,
                actions=out.actions, obs=out.obs)


def run_steps(case: Case, steps: int, tpe2_enabled: bool = True):
    env, orc, rng = _setup(case)
    A, code = env.num_agents, OBS_CODE[case.obs]
    for t in range(steps):
        acts = rng.integers(0, 5, size=(env.num_envs, A)).astype(np.int8) if case.policy == "external" else None
        out = env.step(None if acts is None else torch.from_numpy(acts).cuda(), policy=case.policy)
        res = orc.step(acts, policy=case.policy, auto_reset=True, obs_dtype=code)
        tag = f"{case.id} t={t}"
        _same_state(env, orc, tag)
        _same_outputs(_step_outputs(out), res, case.obs, tag)
    env.check_error()
    assert env.last_kernel_name == case.expected(tpe2_enabled=tpe2_enabled)[0]
    st = _same_stats(env, orc)
    assert st["episodes"] > 0
    env.close()


CASES = device_cases()


@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_edge_lattice_matches_oracle(case):
    run_steps(case, 40 if LATTICES[case.lattice].max_steps < 20 else 50)


# ---- fused rollouts: state in registers across resets ------------------------------------------------------------
def _fused_cases():
    out = []
    for i, name in enumerate(TPE2_LATTICES + TPE_LATTICES):
        lat = LATTICES[name]
        even = next((b, e) for b, e in lat.crews if (b + e) % 2 == 0)
        pols = ("greedy", "waiting", "random", "external")
        out.append((Case(name, *even, "float32", pols[i % 4]), 20 if i == 0 else 7))
        out.append((Case(name, *lat.crews[-1], ("table", "none")[i % 2], pols[(i + 1) % 4]), 7))
    return out


FUSED = _fused_cases()


@pytest.mark.parametrize("case,T", FUSED, ids=[f"{c.id}-T{T}" for c, T in FUSED])
def test_edge_lattice_fused_rollout_matches_oracle(case, T):
    env, orc, rng = _setup(case)
    A, code = env.num_agents, OBS_CODE[case.obs]
    for _ in range(3):       # spread the phases before the fused launch
        env.step(policy="waiting")
        orc.step(policy="waiting", auto_reset=True, obs_dtype=code)
    acts = rng.integers(0, 5, size=(T, env.num_envs, A)).astype(np.int8) if case.policy == "external" else None
    launches = env.launch_count
    traj = env.rollout_trajectory(T, policy=case.policy, actions=None if acts is None else torch.from_numpy(acts).cuda())
    assert env.launch_count == launches + 1 and env.last_kernel_name == case.expected()[0]
    resets = 0
    for t in range(T):
        res = orc.step(None if acts is None else acts[t], policy=case.policy, auto_reset=True, obs_dtype=code)
        _same_outputs({k: v[t] if v is not None else None for k, v in traj.items()}, res, case.obs, f"{case.id} fused t={t}")
        resets += int((res["env_flags"] & _abi.E_WAS_RESET).astype(bool).sum())
    _same_state(env, orc, f"{case.id} after the fused launch")
    _same_stats(env, orc)
    env.check_error()
    assert resets > 0
    env.close()


# ---- numpy-mode placements: np_place_agent in all three kernel families at lattice edges ------------------------
NUMPY_CASES = [Case("t2_256_square", 3, 3, "table", "greedy"), Case("t2_256_square", 4, 2, "float32", "random"),
               Case("tpe_cols33", 4, 2, "float32", "waiting"), Case("tpe_cols33", 2, 2, "none", "greedy", "lanes"),
               Case("max_120", 4, 4, "float32", "greedy"), Case("max_120", 5, 4, "table", "random")]


@pytest.mark.parametrize("case", NUMPY_CASES, ids=[c.id for c in NUMPY_CASES])
def test_edge_lattice_numpy_placements_match_oracle(case):
    from np_oracle import NumpyOracleEnvs

    cfg = case.config()
    low = lower_config(cfg)
    n = 32 * 3 + 7
    seed = 11
    env = make_env(cfg, n, seed=seed, global_env_offset=OFFSET, obs_dtype=case.obs, auto_reset=True, with_info=True,
                   kernel=case.kernel, reset_rng="numpy")
    seeds = np.arange(n, dtype=np.int64) * 7919 + 3
    env.reset_seeded(torch.from_numpy(seeds).cuda())
    orc = NumpyOracleEnvs(low, n, seed=seed, global_env_offset=OFFSET)
    orc.reset_seeded(seeds)
    _same_state(env, orc, f"{case.id} seeded reset")
    code = OBS_CODE[case.obs]
    for t in range(2 * low.max_steps + 5):
        out = env.step(policy=case.policy)
        res = orc.step(policy=case.policy, auto_reset=True, obs_dtype=code)
        _same_state(env, orc, f"{case.id} t={t}")
        _same_outputs(_step_outputs(out), res, case.obs, f"{case.id} t={t}")
    traj = env.rollout_trajectory(7, policy=case.policy)
    for t in range(7):
        res = orc.step(policy=case.policy, auto_reset=True, obs_dtype=code)
        _same_outputs({k: v[t] if v is not None else None for k, v in traj.items()}, res, case.obs, f"{case.id} trajectory t={t}")
    env.check_error()
    assert env.last_kernel_name == case.expected(np_reset=True)[0]
    _same_state(env, orc, f"{case.id} end")
    assert np.array_equal(env.get_state()["rng"].cpu().numpy().view(np.uint64), orc.gen)
    assert _same_stats(env, orc)["episodes"] > 0
    env.close()


# ---- the thread-per-env kernel on the small lattices (CCB200_TPE2=0 is read once per process) ----------------------
TPE2_OFF = tpe2_off_cases()


@pytest.mark.parametrize("case", TPE2_OFF, ids=[c.id for c in TPE2_OFF])
def test_tpe_on_small_lattice_matches_oracle(case):
    """Runs in the subprocess of test_tpe_serves_small_lattices_with_tpe2_off."""
    if os.environ.get("CCB200_TPE2") != "0":
        pytest.skip("needs CCB200_TPE2=0 at process start (test_tpe_serves_small_lattices_with_tpe2_off sets it)")
    run_steps(case, 40, tpe2_enabled=False)


def test_tpe_serves_small_lattices_with_tpe2_off():
    """cc_step_tpe_kernel on lattices cc_step_tpe2_kernel normally takes: float32 rows of 2, 4 and 6/8 agents (bitmap
    capacities 2, 8 and 16 in the TMA image ring) and the compact output modes."""
    env = dict(os.environ, CCB200_TPE2="0")
    sel = f"tests/{Path(__file__).name}::test_tpe_on_small_lattice_matches_oracle"
    proc = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", "-p", "no:cacheprovider", sel], cwd=ROOT, env=env,
                          capture_output=True, text=True, timeout=900)
    tail = (proc.stdout + proc.stderr)[-3000:]
    assert proc.returncode == 0, tail
    assert f"{len(TPE2_OFF)} passed" in tail and "skipped" not in tail, tail
