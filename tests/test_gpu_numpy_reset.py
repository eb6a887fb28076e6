"""GPU: numpy-mode placements (``reset_rng="numpy"``, ``cc_set_reset_rng(CC_RESET_RNG_NUMPY)``) against the C oracle's
numpy mode, which tests/test_numpy_reset_cpu.py pins to the reference's own reset-on-done loop.  Every output field of
every step, the state and the per-env generators (``cc_get_rng_state``) after the run, through all three kernels."""

import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch
from cases import crew_config, readme_config

from np_oracle import NumpyOracleEnvs
from collectivecrossing_b200 import BatchedCollectiveCrossing, VectorCollectiveCrossing, _abi
from collectivecrossing_b200.lowering import lower_config

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
OBS_CODE = {"none": _abi.OBS_NONE, "table": _abi.OBS_TABLE, "int8": _abi.OBS_INT8, "float32": _abi.OBS_FP32}


def make_pair(cfg_py, n, obs="float32", kernel="auto", reward="float32", seed0=17, offset=0):
    env = BatchedCollectiveCrossing(cfg_py, n, "cuda:0", seed=7, obs_dtype=obs, reward_dtype=reward, auto_reset=True,
                                    with_info=True, kernel=kernel, reset_rng="numpy")
    assert env.reset_rng == "numpy"
    seeds = torch.arange(n, dtype=torch.int64, device="cuda:0") * 1000 + seed0
    env.reset_seeded(seeds)
    orc = NumpyOracleEnvs(lower_config(cfg_py), n, seed=7, global_env_offset=offset)
    orc.reset_seeded(seeds.cpu().numpy())
    return env, orc


def gen_of(env):
    return env.get_state()["rng"].cpu().numpy().view(np.uint64)


def same_outputs(dev, res, obs, t=None):
    sl = (lambda v: v) if t is None else (lambda v: v[t])
    for name, key in (("reward", "reward"), ("agent_flags", "agent_flags"), ("agent_info", "agent_info"), ("env_flags", "env_flags")):
        assert np.array_equal(sl(dev[name]).cpu().numpy(), res[key]), (name, t)
    if "actions" in dev:
        assert np.array_equal(sl(dev["actions"]).cpu().numpy(), res["actions_out"]), ("actions", t)
    if obs != "none":
        assert np.array_equal(sl(dev["obs"]).cpu().numpy(), res["obs"]), ("obs", t)


def same_state(env, orc):
    torch.cuda.synchronize()
    env.check_error()
    assert np.array_equal(env.x.cpu().numpy(), orc.x) and np.array_equal(env.y.cpu().numpy(), orc.y)
    assert np.array_equal(env.flags.cpu().numpy(), orc.flags) and np.array_equal(env.step_count.cpu().numpy(), orc.step_count)
    assert np.array_equal(env.episode_return.cpu().numpy(), orc.episode_return)
    assert np.array_equal(gen_of(env), orc.gen)


def step_dict(env):
    return dict(reward=env.reward, agent_flags=env.agent_flags, agent_info=env.agent_info, env_flags=env.env_flags,
                actions=env.actions_out, obs=env.obs)


def run_all_paths(env, orc, obs, policy="greedy", steps=30):
    """single steps, cc_rollout (last step's outputs) and one fused rollout_trajectory(T=20)"""
    code = OBS_CODE[obs]
    resets = 0
    for _ in range(steps):
        env.step(policy=policy)
        res = orc.step(policy=policy, auto_reset=True, obs_dtype=code)
        same_outputs(step_dict(env), res, obs)
        resets += int((res["env_flags"] & _abi.E_WAS_RESET).astype(bool).sum())
    env.rollout(5, policy=policy)
    for _ in range(5):
        res = orc.step(policy=policy, auto_reset=True, obs_dtype=code)
    same_outputs(step_dict(env), res, obs)
    traj = env.rollout_trajectory(20, policy=policy)
    for t in range(20):
        res = orc.step(policy=policy, auto_reset=True, obs_dtype=code)
        same_outputs(traj, res, obs, t)
        resets += int((res["env_flags"] & _abi.E_WAS_RESET).astype(bool).sum())
    same_state(env, orc)
    assert resets > 0
    return resets


@pytest.mark.parametrize("obs", ["none", "table", "int8", "float32"])
@pytest.mark.parametrize("kernel", ["threads", "lanes"])
def test_readme_config_matches_oracle(kernel, obs):
    env, orc = make_pair(readme_config(max_steps=12), 1000, obs, kernel)
    run_all_paths(env, orc, obs)
    want = "cc_step_tpe2_kernel" if kernel == "threads" else "cc_kernel"
    assert want in env.last_kernel_name and env.last_kernel == kernel


@pytest.mark.parametrize("obs", ["none", "table", "float32"])
def test_large_lattice_runs_the_general_thread_per_env_kernel(obs):
    env, orc = make_pair(crew_config(5, 3, max_steps=20), 700, obs, "threads")   # (40+3) x (24+3) padded cells > 256
    run_all_paths(env, orc, obs, policy="waiting")
    assert "cc_step_tpe_kernel<" in env.last_kernel_name


@pytest.mark.parametrize("boarding,exiting", [(7, 5), (30, 20)])
def test_big_crews_float64_rewards_and_dict_order(boarding, exiting):
    cfg_py = crew_config(boarding, exiting, width=16, height=10, max_steps=10)
    env, orc = make_pair(cfg_py, 96, "int8", "auto", reward="float64")
    a = env.num_agents
    rng = np.random.default_rng(3)
    for _ in range(25):
        acts = rng.integers(0, 5, (96, a)).astype(np.int8)
        order = np.stack([rng.permutation(a) for _ in range(96)]).astype(np.int8)
        order[rng.random((96, a)) < 0.1] = -1
        env.step(torch.from_numpy(acts).cuda(), order=torch.from_numpy(order).cuda())
        res = orc.step(acts, order=order, auto_reset=True, obs_dtype=_abi.OBS_INT8, reward_dtype=_abi.REWARD_F64)
        same_outputs(step_dict(env), res, "int8")
    assert env.last_kernel == "lanes"
    same_state(env, orc)


def test_host_path_chunks_equal_the_device_path():
    cfg_py = readme_config(max_steps=12)
    dev, _ = make_pair(cfg_py, 1000, "float32", "auto")
    host, _ = make_pair(cfg_py, 1000, "float32", "auto")
    host.set_host_chunk(256)
    hb = host.make_host_buffers()
    for _ in range(15):
        dev.step(policy="greedy")
        host.step_host(hb, policy="greedy")
        assert host.last_host_call()["chunks"] == 4
        same_outputs({k: v for k, v in hb.items() if k != "actions"} | {"actions": hb["actions_out"]},
                     {k: v.cpu().numpy() for k, v in step_dict(dev).items() if k != "actions"} | {"actions_out": dev.actions_out.cpu().numpy()},
                     "float32")
    traj = dev.rollout_trajectory(20, policy="greedy")
    hb20 = host.make_host_buffers(n_steps=20)
    host.rollout_host(hb20, 20, policy="greedy")
    for name in ("obs", "reward", "agent_flags", "agent_info", "env_flags"):
        assert np.array_equal(hb20[name].numpy(), traj[name].cpu().numpy()), name
    torch.cuda.synchronize()
    assert np.array_equal(gen_of(dev), gen_of(host)) and torch.equal(dev.x, host.x)


@pytest.mark.parametrize("kernel", ["auto", "lanes"])
def test_manual_reset_on_done_loop_matches_oracle(kernel):
    cfg_py = readme_config(max_steps=10)
    env, orc = make_pair(cfg_py, 500, "float32", kernel)
    env.auto_reset = False
    masked = 0
    for _ in range(40):
        out = env.step(policy="greedy")
        res = orc.step(policy="greedy", auto_reset=False, obs_dtype=_abi.OBS_FP32)
        same_outputs(step_dict(env), res, "float32")            # terminal observations included
        done = (res["env_flags"] & (_abi.E_TERMINATED_ALL | _abi.E_TRUNCATED_ALL)) != 0
        if done.any():
            before = out.obs.cpu().numpy()
            env.reset(mask=torch.from_numpy(done.astype(np.uint8)).cuda())
            rows = orc.reset(mask=done.astype(np.uint8), obs_dtype=_abi.OBS_FP32)
            after = env.obs.cpu().numpy()
            assert np.array_equal(after[done], rows[done]) and np.array_equal(after[~done], before[~done])
            masked += int(done.sum())
    assert masked > 0
    same_state(env, orc)


def test_checkpoint_resume_continues_exactly():
    cfg_py = readme_config(max_steps=12)
    a, _ = make_pair(cfg_py, 600, "table", "auto")
    for _ in range(17):
        a.step(policy="waiting")
    state = a.get_state()
    b = BatchedCollectiveCrossing(cfg_py, 600, "cuda:0", seed=7, obs_dtype="table", with_info=True, reset_rng="numpy")
    b.load_state(state)
    ta = {k: v.clone() for k, v in a.rollout_trajectory(20, policy="waiting").items() if v is not None}
    tb = b.rollout_trajectory(20, policy="waiting")
    for k, v in ta.items():
        assert torch.equal(v, tb[k]), k
    assert (ta["env_flags"] & _abi.E_WAS_RESET).any()
    torch.cuda.synchronize()
    assert np.array_equal(gen_of(a), gen_of(b)) and torch.equal(a.x, b.x) and torch.equal(a.flags, b.flags)


def test_unseeded_numpy_mode_fails_before_enqueueing():
    env = BatchedCollectiveCrossing(readme_config(), 64, "cuda:0", obs_dtype="float32", reset_rng="numpy")
    env.step(policy="random", auto_reset=False)   # nothing is placed: allowed
    torch.cuda.synchronize()
    x, obs, t, launches = env.x.clone(), env.obs.clone(), env.step_counter, env.launch_count
    for call in (lambda: env.step(policy="greedy"), lambda: env.rollout(3), lambda: env.rollout_trajectory(4),
                 lambda: env.reset(), lambda: env.step_host(env.make_host_buffers(), policy="greedy")):
        with pytest.raises(ValueError, match="seed them first"):
            call()
    torch.cuda.synchronize()
    assert torch.equal(env.x, x) and torch.equal(env.obs, obs) and env.step_counter == t and env.launch_count == launches
    with pytest.raises(ValueError):
        BatchedCollectiveCrossing(readme_config(), 64, "cuda:0", reset_rng="pcg")


def test_random_actions_are_those_of_philox_mode():
    cfg_py = readme_config(max_steps=15)
    envs = [BatchedCollectiveCrossing(cfg_py, 512, "cuda:0", seed=9, obs_dtype="float32", reset_rng=r) for r in ("philox", "numpy")]
    for e in envs:
        e.reset_seeded(torch.arange(512, dtype=torch.int64, device="cuda:0"))
    before_reset = True
    for _ in range(40):
        outs = [e.step(policy="random") for e in envs]
        assert torch.equal(outs[0].actions, outs[1].actions)
        if before_reset:
            # on the step of the first reset the outputs of the finished step still agree; the rows show the new episodes
            before_reset = not bool(outs[0].was_reset.any())
            for name in ("obs", "reward", "agent_flags", "env_flags")[0 if before_reset else 1:]:
                assert torch.equal(getattr(outs[0], name), getattr(outs[1], name)), name
    assert not before_reset


def test_vector_env_reproduces_seeded_reference_envs():
    cfg_py = readme_config(max_steps=12)
    venv = VectorCollectiveCrossing(cfg_py, 256, "cuda:0", reset_rng="numpy")
    venv.reset(seed=100)
    orc = NumpyOracleEnvs(lower_config(cfg_py), 256)
    orc.reset_seeded(np.arange(256, dtype=np.int64) + 100, obs_dtype=_abi.OBS_FP32)
    for _ in range(30):
        st = venv.step(policy="greedy")
        res = orc.step(policy="greedy", auto_reset=True, obs_dtype=_abi.OBS_FP32)
        assert np.array_equal(st.obs.cpu().numpy(), res["obs"]) and np.array_equal(st.rewards.cpu().numpy(), res["reward"])


def test_one_million_envs_fused_launches_on_strided_blocks():
    n, block = 1 << 20, 256
    cfg_py = readme_config()
    env = BatchedCollectiveCrossing(cfg_py, n, "cuda:0", seed=7, obs_dtype="float32", reset_rng="numpy")
    env.reset_seeded(torch.arange(n, dtype=torch.int64, device="cuda:0") * 3 + 1)
    starts = list(range(0, n, n // 8)) + [n - block]
    orcs = []
    for s in starts:
        o = NumpyOracleEnvs(lower_config(cfg_py), block, seed=7, global_env_offset=s)
        o.reset_seeded(np.arange(s, s + block, dtype=np.int64) * 3 + 1)
        orcs.append(o)
    resets = 0
    for _ in range(10):
        traj = env.rollout_trajectory(20, policy="greedy")
        cut = {k: torch.cat([v[:, s:s + block] for s in starts], 1).cpu().numpy() for k, v in traj.items() if v is not None}
        for t in range(20):
            for b, o in enumerate(orcs):
                res = o.step(policy="greedy", auto_reset=True, obs_dtype=_abi.OBS_FP32)
                sl = slice(b * block, (b + 1) * block)
                for name, key in (("obs", "obs"), ("reward", "reward"), ("agent_flags", "agent_flags"), ("env_flags", "env_flags"), ("actions", "actions_out")):
                    assert np.array_equal(cut[name][t, sl], res[key]), (name, t, starts[b])
                resets += int((res["env_flags"] & _abi.E_WAS_RESET).astype(bool).sum())
    assert resets > 0
    assert "tpe2" in env.last_kernel_name
    gen = gen_of(env)
    for s, o in zip(starts, orcs):
        assert np.array_equal(gen[s:s + block], o.gen)
    env.check_error()


def test_numpy_cases_pass_in_the_checked_build():
    checked = ROOT / "collectivecrossing_b200" / "csrc" / "libccb200_checked.so"
    if not checked.exists():
        pytest.skip("checked library not built (make -C collectivecrossing_b200/csrc libccb200_checked.so)")
    sel = [f"{__file__}::test_readme_config_matches_oracle", f"{__file__}::test_large_lattice_runs_the_general_thread_per_env_kernel",
           f"{__file__}::test_manual_reset_on_done_loop_matches_oracle", f"{__file__}::test_host_path_chunks_equal_the_device_path"]
    proc = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", "-p", "no:cacheprovider", *sel], cwd=ROOT,
                          env=dict(os.environ, CCB200_LIB=str(checked)), capture_output=True, text=True, timeout=1500)
    tail = (proc.stdout + proc.stderr)[-3000:]
    assert proc.returncode == 0 and " passed" in tail and "failed" not in tail, tail
