"""GPU: the step outputs live in memory from the library's allocator (cc_device_alloc: compressible where the device grants
it).  Rollouts written there equal the same seeded rollouts written through the raw C ABI into plain torch.zeros buffers;
`outputs_compressed` says what the driver granted; an output tensor outlives its env and its memory returns afterwards."""

import ctypes as C
import gc

import pytest
from cases import readme_config

from collectivecrossing_b200 import _abi, _native

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

FIELDS = ("obs", "reward", "agent_flags", "agent_info", "env_flags", "actions")


def make_env(n, obs):
    from collectivecrossing_b200 import BatchedCollectiveCrossing

    env = BatchedCollectiveCrossing(readme_config(), n, "cuda:0", seed=11, obs_dtype=obs, with_info=True)
    env.reset()
    return env


def raw_outputs(env, lead):
    """Plain torch.zeros output buffers (the allocation before cc_device_alloc) and the CCStepIO that points at them."""
    n, a, dev = env.num_envs, env.num_agents, env.device
    out = dict(obs=None if env.obs is None else torch.zeros(lead + (n, a, env.obs_width), dtype=env.obs_torch_dtype, device=dev),
               reward=torch.zeros(lead + (n, a), dtype=env.reward_torch_dtype, device=dev),
               agent_flags=torch.zeros(lead + (n, a), dtype=torch.uint8, device=dev),
               agent_info=torch.zeros(lead + (n, a), dtype=torch.uint8, device=dev),
               env_flags=torch.zeros(lead + (n,), dtype=torch.uint8, device=dev),
               actions=torch.zeros(lead + (n, a), dtype=torch.int8, device=dev))
    io = _abi.CCStepIO()
    io.actions, io.order = None, None
    io.actions_out = out["actions"].data_ptr()
    io.obs = None if out["obs"] is None else out["obs"].data_ptr()
    io.reward, io.agent_flags = out["reward"].data_ptr(), out["agent_flags"].data_ptr()
    io.agent_info, io.env_flags = out["agent_info"].data_ptr(), out["env_flags"].data_ptr()
    io.obs_dtype, io.reward_dtype, io.policy, io.auto_reset = env.obs_code, env.reward_code, _abi.POLICIES["greedy"], 1
    return out, io


@pytest.mark.parametrize("n", [65536, 1048576])
@pytest.mark.parametrize("T", [1, 20])
@pytest.mark.parametrize("obs", ["float32", "int8", "table", "none"])
def test_library_buffers_equal_plain_buffers(obs, T, n):
    lib_env, raw_env = make_env(n, obs), make_env(n, obs)
    raw, io = raw_outputs(raw_env, (T,) if T > 1 else ())
    stream = torch.cuda.current_stream().cuda_stream
    for _ in range(2):   # the second launch rewrites the same buffers
        if T == 1:
            o = lib_env.step(policy="greedy")
            got = dict(obs=o.obs, reward=o.reward, agent_flags=o.agent_flags, agent_info=o.agent_info, env_flags=o.env_flags, actions=o.actions)
            _native.check(raw_env._lib.cc_step(raw_env._h, C.byref(io), stream))
        else:
            got = lib_env.rollout_trajectory(T, policy="greedy")
            _native.check(raw_env._lib.cc_rollout_fused(raw_env._h, C.byref(io), T, stream))
        torch.cuda.synchronize()
        for f in FIELDS:
            if raw[f] is None:
                assert got[f] is None, f
            else:
                assert got[f].shape == raw[f].shape and got[f].dtype == raw[f].dtype, f
                assert torch.equal(got[f], raw[f]), f
    assert (raw["agent_flags"] != 0).any() and (raw["actions"] != 0).any()
    for k in ("x", "y", "flags", "step_count", "episode_return"):
        assert torch.equal(getattr(lib_env, k), getattr(raw_env, k)), k
    lib_env.check_error()
    raw_env.check_error()
    lib_env.close()
    raw_env.close()


def compression_of(ptr):
    """CUmemAllocationProp.allocFlags.compressionType of the allocation at `ptr` (0 for cudaMalloc memory)."""
    cuda = C.CDLL("libcuda.so.1")
    handle = C.c_ulonglong()
    if cuda.cuMemRetainAllocationHandle(C.byref(handle), C.c_void_p(ptr)) != 0:
        return 0   # not a cuMemCreate allocation
    prop = (C.c_ubyte * 32)()   # CUmemAllocationProp: allocFlags.compressionType is the byte at offset 24
    try:
        assert cuda.cuMemGetAllocationPropertiesFromHandle(prop, handle) == 0
    finally:
        cuda.cuMemRelease(handle)
    return prop[24]


def test_outputs_compressed_reports_the_allocation():
    env = make_env(4096, "float32")
    traj = env.rollout_trajectory(4, policy="greedy")
    tensors = [env.obs, env.reward, env.agent_flags, env.agent_info, env.env_flags, env.actions_out] + [traj[f] for f in FIELDS]
    kinds = {compression_of(t.data_ptr()) for t in tensors}
    assert kinds == {1 if env.outputs_compressed else 0}, kinds
    supported = C.c_int()
    cuda = C.CDLL("libcuda.so.1")
    assert cuda.cuDeviceGetAttribute(C.byref(supported), 107, 0) == 0   # CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED
    if not supported.value:
        assert not env.outputs_compressed
    env.close()
    if not env.outputs_compressed:
        pytest.skip("the device granted plain memory for the outputs (compression not supported or refused)")


def test_output_tensor_outlives_the_env_and_its_memory_returns():
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free0, _ = torch.cuda.mem_get_info()
    env = make_env(1048576, "float32")
    env.step(policy="greedy")
    obs, expect = env.obs, env.obs.clone()
    obs_bytes = obs.numel() * obs.element_size()
    env.close()
    del env
    gc.collect()
    torch.cuda.empty_cache()
    assert torch.equal(obs, expect)
    obs.add_(1.0)   # still writable device memory
    assert torch.equal(obs, expect + 1.0)
    del expect
    torch.cuda.empty_cache()
    held, _ = torch.cuda.mem_get_info()
    assert free0 - held >= obs_bytes
    del obs
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free1, _ = torch.cuda.mem_get_info()
    assert free1 >= free0 - (64 << 20), (free0, free1)


@pytest.mark.parametrize("obs", ["float32", "table"])
def test_host_path_equals_the_device_step(obs):
    host_env, dev_env = make_env(50000, obs), make_env(50000, obs)
    host = host_env.make_host_buffers()
    for _ in range(3):
        out = host_env.step_host(host, policy="greedy")
        o = dev_env.step(policy="greedy")
        torch.cuda.synchronize()
        assert torch.equal(out["obs"], o.obs.cpu())
        assert torch.equal(out["reward"], o.reward.cpu())
        assert torch.equal(out["agent_flags"], o.agent_flags.cpu())
        assert torch.equal(out["env_flags"], o.env_flags.cpu())
    host_env.close()
    dev_env.close()


def test_new_trajectory_buffers_on_a_side_stream():
    """rollout_trajectory allocates (and zero-fills) new buffers for a new T and launches at once on the caller's stream:
    on a non-blocking side stream the results equal those of the default stream."""
    ref_env, side_env = make_env(1048576, "float32"), make_env(1048576, "float32")
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    for T in (20, 7):
        ref = ref_env.rollout_trajectory(T, policy="greedy")
        with torch.cuda.stream(side):
            got = side_env.rollout_trajectory(T, policy="greedy")
        side.synchronize()
        torch.cuda.synchronize()
        for f in FIELDS:
            assert torch.equal(got[f], ref[f]), (T, f)
        assert (got["agent_flags"][-1] != 0).any()
    ref_env.close()
    side_env.close()
