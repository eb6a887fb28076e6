"""Numpy-mode auto-reset (``reset_rng="numpy"``) of the C oracle against the reference's own loop: N envs, each
``reset(seed=s_n)`` once, then ``step`` with ``reset()`` (no seed) whenever ``__all__`` is done.  Every field of every
step over several episodes per env, and the generators at the end.  The loop runs through ``oracle/pyport.py`` on any
checkout and through the unmodified reference where its sources are staged."""

from __future__ import annotations

import numpy as np
import pytest
from cases import crew_config, readme_config, readme_crew

from np_oracle import NumpyOracleEnvs
from collectivecrossing_b200 import _abi
from collectivecrossing_b200.lowering import lower_config
from oracle import refload
from oracle.pyport import PyEnv

CASES = {
    # (config, steps): at least 3 episodes per env; max_steps small enough that episodes also end by truncation
    "readme": (lambda: readme_config(max_steps=30), 130),
    "crew_1": (lambda: readme_crew(1, 0, max_steps=12), 60),
    "crew_7_5": (lambda: crew_config(7, 5, width=16, height=10, max_steps=14), 80),
}
# (case, policy) runs in which some episodes also end with every agent at its destination (the others deadlock or wander)
TERMINATES = {("readme", "waiting"), ("readme", "greedy"), ("crew_1", "greedy"), ("crew_1", "waiting")}
N_ENVS = 6


def _gen_row(rng) -> list[int]:
    st = rng.bit_generator.state
    s, inc = st["state"]["state"], st["state"]["inc"]
    m = (1 << 64) - 1
    return [s >> 64, s & m, inc >> 64, inc & m, st["uinteger"], st["has_uint32"]]


def run_against(make_env, gen_of, cfg_py, steps, policy, seeds):
    """Step the oracle in numpy mode next to N single envs from ``make_env``; returns (episodes, term_all, trunc_all)."""
    cfg = lower_config(cfg_py)
    n, a = len(seeds), cfg.num_agents
    orc = NumpyOracleEnvs(cfg, n, seed=7)
    orc.reset_seeded(np.asarray(seeds, np.int64), obs_dtype=_abi.OBS_FP32)
    envs = [make_env() for _ in range(n)]
    first = [e.reset(seed=int(s)) for e, s in zip(envs, seeds)]
    rows0 = orc.observe(_abi.OBS_FP32)
    ids = [f"boarding_{i}" for i in range(cfg.num_boarding)] + [f"exiting_{i}" for i in range(cfg.num_exiting)]
    for k in range(n):
        for j, i in enumerate(ids):
            assert np.array_equal(rows0[k, j], np.asarray(first[k][0][i], np.float32))
    counts = np.zeros(3, np.int64)
    for t in range(steps):
        res = orc.step(policy=policy, auto_reset=True, obs_dtype=_abi.OBS_FP32, reward_dtype=_abi.REWARD_F64, check=False)
        assert res["status"] == _abi.OK
        for k, env in enumerate(envs):
            acts = res["actions_out"][k]
            live = list(env.agents)
            if policy != "random":
                want = env.policy_actions(policy) if isinstance(env, PyEnv) else None
                if want is not None:
                    assert all(int(acts[ids.index(i)]) == v for i, v in want.items()), (t, k)
            obs, rew, term, trunc, infos = env.step({i: int(acts[ids.index(i)]) for i in live})
            af, ef = res["agent_flags"][k], int(res["env_flags"][k])
            for j, i in enumerate(ids):
                bits = int(af[j])
                assert bool(bits & _abi.O_ALIVE_PREV) == (i in rew), (t, k, i)
                if i in rew:
                    assert res["reward"][k, j] == rew[i], (t, k, i)
                    assert bool(bits & _abi.O_TRUNC_VALUE) == trunc[i], (t, k, i)
                assert bool(bits & _abi.O_TERM_VALUE) == term[i], (t, k, i)
                assert bool(bits & _abi.O_OBS_PRESENT) == (i in obs), (t, k, i)
                if i in infos:
                    info = int(res["agent_info"][k, j])
                    assert (bool(info & _abi.I_IN_TRAM_AREA), bool(info & _abi.I_AT_DOOR), bool(info & _abi.I_ACTIVE),
                            bool(info & _abi.I_AT_DESTINATION)) == (infos[i]["in_tram_area"], infos[i]["at_door"],
                                                                    infos[i]["active"], infos[i]["at_destination"]), (t, k, i)
            assert bool(ef & _abi.E_TERMINATED_ALL) == term["__all__"] and bool(ef & _abi.E_TRUNCATED_ALL) == trunc["__all__"], (t, k)
            done = term["__all__"] or trunc["__all__"]
            assert bool(ef & _abi.E_WAS_RESET) == done, (t, k)
            if done:
                counts += (1, term["__all__"], trunc["__all__"] and not term["__all__"])
                obs, _ = env.reset()                                  # reset() without a seed: the env's generator continues
            # the oracle's rows show the post-step (post-reset) state
            for j, i in enumerate(ids):
                if i in obs:
                    assert np.array_equal(res["obs"][k, j], np.asarray(obs[i], np.float32)), (t, k, i)
            if isinstance(env, PyEnv):
                assert [tuple(env.pos[i]) for i in ids] == list(zip(orc.x[k].tolist(), orc.y[k].tolist())), (t, k)
                assert [env.active[i] for i in ids] == [bool(f & _abi.F_ACTIVE) for f in orc.flags[k]], (t, k)
    for k, env in enumerate(envs):
        assert [int(v) for v in orc.gen[k]] == _gen_row(gen_of(env)), k
    return counts


@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("policy", ["greedy", "waiting", "random"])
def test_oracle_numpy_auto_reset_equals_pyport_loop(case, policy):
    make_cfg, steps = CASES[case]
    cfg_py = make_cfg()
    seeds = [1000 * k + 17 for k in range(N_ENVS)]
    episodes, term_all, trunc_all = run_against(lambda: PyEnv(cfg_py), lambda e: e.rng, cfg_py, steps, policy, seeds)
    assert episodes >= 3 * N_ENVS
    assert trunc_all > 0
    if (case, policy) in TERMINATES:
        assert term_all > 0


@pytest.mark.skipif(not refload.available(), reason="reference sources not mounted")
@pytest.mark.parametrize("case", list(CASES))
@pytest.mark.parametrize("policy", ["greedy", "random"])
def test_oracle_numpy_auto_reset_equals_live_reference_loop(case, policy):
    ref = refload.load()
    make_cfg, steps = CASES[case]
    cfg_py = make_cfg()
    rcfg = refload.to_reference_config(cfg_py, validate=case != "crew_7_5")
    seeds = [1000 * k + 17 for k in range(N_ENVS)]
    episodes, _, _ = run_against(lambda: ref.CollectiveCrossingEnv(rcfg), lambda e: e.np_random, cfg_py, steps, policy, seeds)
    assert episodes >= 3 * N_ENVS


def test_oracle_masked_reset_continues_only_the_masked_generators():
    cfg = lower_config(readme_config())
    orc = NumpyOracleEnvs(cfg, 4)
    with pytest.raises(ValueError):
        orc.reset(obs_dtype=_abi.OBS_FP32)
    orc.reset_seeded(np.arange(4, dtype=np.int64) + 5, obs_dtype=_abi.OBS_FP32)
    rows = orc.observe(_abi.OBS_FP32)
    gen0, x0 = orc.gen.copy(), orc.x.copy()
    buf = orc.reset(mask=np.array([0, 1, 0, 1], np.uint8), obs_dtype=_abi.OBS_FP32)
    ports = [PyEnv(readme_config()) for _ in range(4)]
    for k, p in enumerate(ports):
        p.reset(seed=5 + k)
    for k in (1, 3):
        obs, _ = ports[k].reset()
        assert [int(v) for v in orc.gen[k]] == _gen_row(ports[k].rng)
        assert np.array_equal(buf[k], np.stack([obs[i] for i in ports[k].ids]))
    for k in (0, 2):
        assert np.array_equal(orc.gen[k], gen0[k]) and np.array_equal(orc.x[k], x0[k])
        assert np.array_equal(orc.observe(_abi.OBS_FP32)[k], rows[k])
