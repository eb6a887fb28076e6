"""Cassette I/O and the rasteriser on the CPU: the schema round-trips through the pure-Python
port, and the reference's own golden cassettes replay through it with our replayer."""

import json
from pathlib import Path

import numpy as np
import pytest
from cases import cassette_config, readme_config

from collectivecrossing_b200 import cassette, rendering
from collectivecrossing_b200.utils.geometry import calculate_tram_boundaries
from oracle import refload
from oracle.pyport import PyEnv

# the reference's own golden cassettes, stored next to their converted arrays by tests/golden/make_golden.py
GOLDEN = Path(__file__).resolve().parent / "golden"
CASSETTES = {"golden_basic_trajectory": "cassette_basic", "regression_test": "cassette_regression"}
STEP_KEYS = {"step", "actions", "active_actions", "observations", "next_observations", "next_rewards", "next_terminated",
             "next_truncated", "next_infos"}


def random_action_dicts(env, n, seed):
    rng = np.random.default_rng(seed)
    return [{a: int(rng.integers(0, 5)) for a in env.ids} for _ in range(n)]


def test_record_then_replay_round_trip(tmp_path):
    cfg = readme_config(max_steps=30)
    env = PyEnv(cfg)
    path = tmp_path / "c.json"
    traj = cassette.record_trajectory(env, random_action_dicts(env, 40, 1), path)
    assert set(traj) == {"config", "initial_observations", "initial_infos", "steps"}
    assert all(set(s) == STEP_KEYS for s in traj["steps"])
    assert traj["config"]["width"] == 12 and traj["config"]["truncated_config"]["max_steps"] == 30
    assert traj["steps"][-1]["next_truncated"]["__all__"] or traj["steps"][-1]["next_terminated"]["__all__"]
    assert json.loads(path.read_text()) == traj               # plain JSON types only
    cassette.replay_trajectory(PyEnv(cfg), path)              # what the reference's replay asserts
    cassette.replay_trajectory(PyEnv(cfg), traj, strict=True)  # and everything else in the cassette


def test_replay_detects_a_changed_trajectory():
    cfg = readme_config(max_steps=30)
    env = PyEnv(cfg)
    traj = cassette.record_trajectory(env, random_action_dicts(env, 10, 2))
    a = next(iter(traj["steps"][3]["next_observations"]))
    traj["steps"][3]["next_observations"][a][0] += 1.0
    with pytest.raises(AssertionError, match="Step 3 next observation mismatch"):
        cassette.replay_trajectory(PyEnv(cfg), traj)


@pytest.mark.parametrize("name", list(CASSETTES))
def test_reference_golden_cassettes_replay(name):
    """The reference's own cassettes (test_trajectory_vcr.py:494-593) through our replayer."""
    if not (GOLDEN / f"{name}.json").exists():
        pytest.skip("the reference's JSON cassettes are not stored yet (tests/golden/make_golden.py stores them)")
    traj = cassette.load_cassette(GOLDEN / f"{name}.json")
    cassette.replay_trajectory(PyEnv(cassette_config()), traj)
    cassette.replay_trajectory(PyEnv(cassette_config()), traj, strict=True)
    # and our recorder reproduces the file from the same actions
    again = cassette.record_trajectory(PyEnv(cassette_config()), [s["actions"] for s in traj["steps"]])
    assert again["steps"] == traj["steps"] and again["initial_observations"] == traj["initial_observations"]
    assert again["initial_infos"] == traj["initial_infos"]


@pytest.mark.parametrize("name", list(CASSETTES.values()))
def test_port_reproduces_the_stored_reference_cassettes(name):
    """The reference's golden cassettes as stored (converted by make_golden.py): the Python port, reset with the cassettes'
    seed and driven by their actions in their order, returns the same observations, float64 rewards, flags and infos."""
    from collectivecrossing_b200 import _abi
    from helpers import load_golden

    rec = load_golden(name)
    env = PyEnv(cassette_config())
    env.reset(seed=int(rec["seeds"][0]))
    assert [env.pos[i][0] for i in env.ids] == rec["init_x"][0].tolist() and [env.pos[i][1] for i in env.ids] == rec["init_y"][0].tolist()
    info_bits = {"in_tram_area": _abi.I_IN_TRAM_AREA, "at_door": _abi.I_AT_DOOR, "active": _abi.I_ACTIVE, "at_destination": _abi.I_AT_DESTINATION}
    for t in range(rec["actions"].shape[0]):
        order = [int(k) for k in rec["order"][t, 0] if k >= 0]
        obs, rew, term, trunc, infos = env.step({env.ids[k]: int(rec["actions"][t, 0, k]) for k in order})
        for k, i in enumerate(env.ids):
            bits = int(rec["agent_flags"][t, 0, k])
            assert (i in rew) == bool(bits & _abi.O_ALIVE_PREV) and rew.get(i, 0.0) == rec["reward"][t, 0, k], (t, i)
            assert term[i] == bool(bits & _abi.O_TERM_VALUE) and trunc.get(i, False) == bool(bits & _abi.O_TRUNC_VALUE), (t, i)
            assert (i in obs) == bool(bits & _abi.O_OBS_PRESENT), (t, i)
            if i in obs:
                assert np.array_equal(obs[i], rec["obs"][t, 0, k].astype(np.float32)), (t, i)
                want = int(rec["agent_info"][t, 0, k])
                assert {f: bool(want & b) for f, b in info_bits.items()} == {f: infos[i][f] for f in info_bits}, (t, i)
        env_bits = (_abi.E_TERMINATED_ALL if term["__all__"] else 0) | (_abi.E_TRUNCATED_ALL if trunc["__all__"] else 0)
        assert env_bits == rec["env_flags"][t, 0], t


@pytest.mark.skipif(not refload.available(), reason="reference sources not mounted")
def test_cassette_recorded_here_replays_on_the_unmodified_reference():
    ref = refload.load()
    cfg = readme_config(max_steps=25)
    env = PyEnv(cfg)
    traj = cassette.record_trajectory(env, random_action_dicts(env, 30, 3))
    cassette.replay_trajectory(ref.CollectiveCrossingEnv(refload.to_reference_config(cfg)), traj, strict=True)


def test_rasteriser_draws_regions_and_agents():
    cfg = readme_config()
    tb = calculate_tram_boundaries(cfg)
    cell = 8
    img = rendering.render_state(cfg, tb, [1, 8, 3], [3, 7, 0], [True, True, False], num_boarding=1, cell=cell)
    rows, cols = cfg.height + 2, cfg.width + 2
    assert img.shape == (rows * cell, cols * cell, 3) and img.dtype == np.uint8

    def centre(x, y):
        return tuple(int(v) for v in img[(rows - 1 - y) * cell + cell // 2, x * cell + cell // 2])

    assert centre(1, 3) == rendering.COLORS["boarding_agent"]      # agent 0 is a boarding agent
    assert centre(8, 7) == rendering.COLORS["exiting_agent"]
    assert centre(3, 0) == rendering.COLORS["inactive_agent"]
    assert centre(13, 9) == rendering.COLORS["background"]         # margin cell, nothing drawn
    assert centre(5, 5) != rendering.COLORS["background"]          # inside the tram area
    assert centre(5, 5) != centre(5, 2)                            # tram area and waiting area differ
