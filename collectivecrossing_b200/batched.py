"""Batched tensor interface over N independent CollectiveCrossing envs on one B200.

``BatchedCollectiveCrossing`` owns torch tensors for the persistent state and the step outputs
and hands their ``data_ptr()`` plus the current CUDA stream to the C-ABI library
(``include/ccb200.h``); every ``step`` is one launch of the fused sm_100a kernel.  It replaces,
for N envs at once, ``CollectiveCrossingEnv.step/reset`` of the reference
(``collectivecrossing.py:91-261``).

Encoding (see the ``CC_*`` enums in the header, mirrored in ``_abi``):

* state  ``x, y`` int8 [N, A]; ``flags`` uint8 [N, A] (active|terminated|truncated);
  ``step_count`` int32 [N]; ``episode_return`` float32 [N]
* agent order is the reference's: ``boarding_0..B-1`` then ``exiting_0..E-1``
* outputs are overwritten in place by every step (the returned ``StepOutput`` aliases them)

The output tensors (``obs``, ``reward``, flags, infos, applied actions, and the ``[T, N, ...]`` buffers of
``rollout_trajectory``) live in memory from the library's ``cc_device_alloc``: compressible device memory where the
GPU grants it (``outputs_compressed``), else plain device memory.  Compression changes no value; it cuts the DRAM
bytes of the very regular observation rows.  Two limits follow: ``torch.cuda.memory_allocated`` does not count these
tensors, and they cannot be shared through CUDA IPC (``torch.multiprocessing``).  Releasing one waits for the
device, like ``cudaFree``, so do not drop the last reference to an env or its output tensors while capturing a CUDA
graph.  The state tensors are ordinary torch allocations.
"""

from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Any

import torch

from . import _abi, _native
from .lowering import lower_config

_OBS_TORCH = {"none": (None, _abi.OBS_NONE), "int8": (torch.int8, _abi.OBS_INT8), "float32": (torch.float32, _abi.OBS_FP32),
              "table": (torch.int8, _abi.OBS_TABLE)}
_REW_TORCH = {"float32": (torch.float32, _abi.REWARD_F32), "float64": (torch.float64, _abi.REWARD_F64)}
_TYPESTR = {torch.float32: "<f4", torch.float64: "<f8", torch.int8: "|i1", torch.uint8: "|u1"}


class _DeviceBuffer:
    """Zeroed memory from ``cc_device_alloc`` exposed through ``__cuda_array_interface__``.  A tensor made from it
    holds a reference to it, so the memory goes back to the library (``cc_device_free``) when the last view dies."""

    def __init__(self, lib, device_index: int, shape: tuple, dtype: torch.dtype):
        nbytes = dtype.itemsize
        for d in shape:
            nbytes *= d
        self._lib, self.ptr = lib, None
        ptr, compressed = C.c_void_p(), C.c_int32()
        _native.check(lib.cc_device_alloc(device_index, max(nbytes, 1), C.byref(ptr), C.byref(compressed)))
        self.ptr, self.compressed = ptr.value, bool(compressed.value)
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": _TYPESTR[dtype], "data": (ptr.value, False),
                                         "strides": None, "version": 2}

    def __del__(self):
        if self.ptr is not None:
            self._lib.cc_device_free(self.ptr)


@dataclass
class StepOutput:
    """Views of the env's output tensors after a step (valid until the next step)."""

    obs: torch.Tensor | None      # [N, A, 6+4A]; [N, A, 4] int8 (x, y, type, active) with obs_dtype="table"
    reward: torch.Tensor          # [N, A]; 0 where the agent had no reward entry
    agent_flags: torch.Tensor     # [N, A] CC_O_* bits
    agent_info: torch.Tensor | None  # [N, A] CC_I_* bits
    env_flags: torch.Tensor       # [N]    CC_E_* bits
    actions: torch.Tensor | None  # [N, A] actions that were applied (policy output)

    # decoded views (each is a small elementwise torch op; not part of the hot path)
    @property
    def terminated(self) -> torch.Tensor:
        return (self.agent_flags & _abi.O_TERM_VALUE) != 0

    @property
    def truncated(self) -> torch.Tensor:
        return (self.agent_flags & _abi.O_TRUNC_VALUE) != 0

    @property
    def alive_prev(self) -> torch.Tensor:
        return (self.agent_flags & _abi.O_ALIVE_PREV) != 0

    @property
    def obs_present(self) -> torch.Tensor:
        return (self.agent_flags & _abi.O_OBS_PRESENT) != 0

    @property
    def terminated_all(self) -> torch.Tensor:
        return (self.env_flags & _abi.E_TERMINATED_ALL) != 0

    @property
    def truncated_all(self) -> torch.Tensor:
        return (self.env_flags & _abi.E_TRUNCATED_ALL) != 0

    @property
    def was_reset(self) -> torch.Tensor:
        return (self.env_flags & _abi.E_WAS_RESET) != 0


def _policy_code(policy: Any) -> int:
    if isinstance(policy, str):
        if policy not in _abi.POLICIES:
            raise ValueError(f"Unknown policy '{policy}'. Available: {', '.join(_abi.POLICIES)}")
        return _abi.POLICIES[policy]
    return int(policy)


class BatchedCollectiveCrossing:
    """N independent CollectiveCrossing envs stepped by one fused CUDA kernel.

    Parameters mirror ``CollectiveCrossingEnv(config)``; ``global_env_offset`` is this shard's
    first env in the whole job (the counter-based RNG is keyed on the global env index, so a run
    sharded over 8 GPUs reproduces the 1-GPU run env by env).

    ``reset_rng`` chooses where unseeded placements (the auto-reset and ``reset(mask)``) come from: "philox"
    (default, counter-based) or "numpy": the reference's ``reset()`` without a seed, env n continuing the numpy
    generator ``reset_seeded`` gave it — N envs seeded once and stepped with auto-reset then reproduce N reference
    envs episode after episode.  In "numpy" mode a call that may place envs raises until ``reset_seeded(seeds)`` or
    ``load_state`` has seeded the generators.
    """

    def __init__(self, config: Any, num_envs: int, device: Any = "cuda:0", *, seed: int = 0,
                 global_env_offset: int = 0, obs_dtype: str = "float32", reward_dtype: str = "float32",
                 auto_reset: bool = True, with_info: bool = False, kernel: str = "auto", reset_rng: str = "philox"):
        self._lib = _native.library()  # raises ImportError when the CUDA library is not built
        if not torch.cuda.is_available():
            raise RuntimeError("collectivecrossing_b200 needs a CUDA device (no CPU fallback exists)")
        if obs_dtype not in _OBS_TORCH:
            raise ValueError(f"obs_dtype must be one of {list(_OBS_TORCH)}")
        if reward_dtype not in _REW_TORCH:
            raise ValueError(f"reward_dtype must be one of {list(_REW_TORCH)}")
        if reset_rng not in _abi.RESET_RNG:
            raise ValueError(f"reset_rng must be one of {list(_abi.RESET_RNG)}")
        self.config = config
        self.cfg = config if isinstance(config, _abi.CCConfig) else lower_config(config)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("device must be a CUDA device")
        self.device_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.num_envs = int(num_envs)
        self.num_agents = self.cfg.num_agents
        self.obs_len = self.cfg.obs_len
        self.seed = int(seed)
        self.global_env_offset = int(global_env_offset)
        self.auto_reset = bool(auto_reset)
        self.obs_dtype = obs_dtype
        self.obs_torch_dtype, self.obs_code = _OBS_TORCH[obs_dtype]
        self.reward_torch_dtype, self.reward_code = _REW_TORCH[reward_dtype]

        n, a, dev = self.num_envs, self.num_agents, self.device
        self.x = torch.zeros((n, a), dtype=torch.int8, device=dev)
        self.y = torch.zeros((n, a), dtype=torch.int8, device=dev)
        self.flags = torch.zeros((n, a), dtype=torch.uint8, device=dev)
        self.step_count = torch.zeros((n,), dtype=torch.int32, device=dev)
        self.episode_return = torch.zeros((n,), dtype=torch.float32, device=dev)
        # last axis of the obs output: the reference's row (6+4A) or one block of the compact table
        self.obs_width = 4 if self.obs_code == _abi.OBS_TABLE else self.obs_len
        self.outputs_compressed = True   # cleared by _output_tensor when the device does not grant compressible memory
        self.obs = None if self.obs_code == _abi.OBS_NONE else self._output_tensor((n, a, self.obs_width), self.obs_torch_dtype)
        self.reward = self._output_tensor((n, a), self.reward_torch_dtype)
        self.agent_flags = self._output_tensor((n, a), torch.uint8)
        self.agent_info = self._output_tensor((n, a), torch.uint8) if with_info else None
        self.env_flags = self._output_tensor((n,), torch.uint8)
        self.actions_out = self._output_tensor((n, a), torch.int8)

        handle = C.c_void_p()
        _native.check(self._lib.cc_create(C.byref(self.cfg), n, self.device_index, self.global_env_offset, self.seed, C.byref(handle)))
        self._h = handle
        _native.check(self._lib.cc_attach_state(self._h, self.x.data_ptr(), self.y.data_ptr(), self.flags.data_ptr(),
                                                self.step_count.data_ptr(), self.episode_return.data_ptr()))
        self._io = _abi.CCStepIO()
        self.set_kernel(kernel)
        _native.check(self._lib.cc_set_reset_rng(self._h, _abi.RESET_RNG[reset_rng]))

    @property
    def reset_rng(self) -> str:
        """Where unseeded placements come from: "philox" or "numpy" (``cc_reset_rng``)."""
        code = int(self._lib.cc_reset_rng(self._h))
        return next(k for k, v in _abi.RESET_RNG.items() if v == code)

    def set_kernel(self, kernel: str) -> None:
        """Work mapping of ``step``: "auto" (default), "lanes" (one lane per agent) or "threads" (one
        thread per env; crews of 4 or 8).  Both mappings return identical results."""
        if kernel not in _abi.KERNEL_VARIANTS:
            raise ValueError(f"kernel must be one of {list(_abi.KERNEL_VARIANTS)}")
        _native.check(self._lib.cc_set_kernel_variant(self._h, _abi.KERNEL_VARIANTS[kernel]))

    @property
    def last_kernel(self) -> str:
        """Mapping the last ``step`` launch used ("none" before the first)."""
        code = int(self._lib.cc_last_kernel_variant(self._h))
        return {0: "none", 1: "lanes", 2: "threads"}[code]

    @property
    def last_kernel_name(self) -> str:
        """Instantiation the last ``step`` launch ran, e.g. ``ccb::cc_step_tpe_kernel<8,4>``."""
        return self._lib.cc_last_kernel_name(self._h).decode()

    def _output_tensor(self, shape: tuple, dtype: torch.dtype) -> torch.Tensor:
        """A zeroed output tensor in memory from ``cc_device_alloc`` (compressible where the device grants it)."""
        buf = _DeviceBuffer(self._lib, self.device_index, shape, dtype)
        self.outputs_compressed = self.outputs_compressed and buf.compressed
        t = torch.as_tensor(buf)
        assert t.device == self.x.device and t.dtype == dtype and t.is_contiguous()
        return t

    # ------------------------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.cc_destroy(self._h)
            self._h = None

    def __del__(self):  # pragma: no cover - best effort
        try:
            self.close()
        except Exception:
            pass

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _check_tensor(self, t: torch.Tensor, dtype: torch.dtype, shape: tuple, name: str) -> torch.Tensor:
        if t.dtype != dtype or tuple(t.shape) != shape or t.device != self.x.device or not t.is_contiguous():
            raise ValueError(f"{name} must be a contiguous {dtype} tensor of shape {shape} on {self.x.device}")
        return t

    # ---- state injection / checkpoint ----------------------------------------------------------
    def set_state(self, x, y, flags, step_count) -> None:
        """Inject a state (what the reference's tests do by writing ``env._agents[id]``)."""
        self.x.copy_(torch.as_tensor(x).reshape(self.x.shape))
        self.y.copy_(torch.as_tensor(y).reshape(self.y.shape))
        self.flags.copy_(torch.as_tensor(flags).reshape(self.flags.shape))
        self.step_count.copy_(torch.as_tensor(step_count).reshape(self.step_count.shape))
        self.episode_return.zero_()

    def get_state(self) -> dict:
        """Checkpoint: env state, the Philox counter and — once ``reset_seeded`` has seeded them — the per-env
        numpy-compatible generators (what gymnasium keeps in ``env.np_random``), so that a resumed run's
        unseeded ``reset()`` continues the saved run's stream."""
        state = {"x": self.x.clone(), "y": self.y.clone(), "flags": self.flags.clone(), "step_count": self.step_count.clone(),
                 "episode_return": self.episode_return.clone(), "t": int(self._lib.cc_step_counter(self._h)), "rng": None}
        if int(self._lib.cc_rng_seeded(self._h)):
            rng = torch.zeros((self.num_envs, 6), dtype=torch.int64, device=self.device)   # uint64 bit patterns
            _native.check(self._lib.cc_get_rng_state(self._h, rng.data_ptr(), self._stream()))
            state["rng"] = rng
        return state

    def load_state(self, state: dict) -> None:
        self.set_state(state["x"], state["y"], state["flags"], state["step_count"])
        self.episode_return.copy_(state["episode_return"])
        _native.check(self._lib.cc_set_step_counter(self._h, int(state["t"])))
        if state.get("rng") is not None:
            rng = self._check_tensor(state["rng"].to(self.device), torch.int64, (self.num_envs, 6), "rng")
            _native.check(self._lib.cc_set_rng_state(self._h, rng.data_ptr(), self._stream()))
            torch.cuda.current_stream(self.device).synchronize()   # `rng` may be a temporary

    # ---- reset ---------------------------------------------------------------------------------
    def reset(self, mask: torch.Tensor | None = None) -> torch.Tensor | None:
        """Re-sample the initial placement (reference ``reset()``, collectivecrossing.py:91-159) of
        all envs, or of those with ``mask[n] != 0``; returns the observation tensor."""
        mptr = None
        if mask is not None:
            mask = self._check_tensor(mask, torch.uint8, (self.num_envs,), "mask")
            mptr = mask.data_ptr()
        optr = self.obs.data_ptr() if self.obs is not None else None
        _native.check(self._lib.cc_reset(self._h, mptr, optr, self.obs_code, self._stream()))
        return self.obs

    def reset_seeded(self, seeds: torch.Tensor | None) -> torch.Tensor | None:
        """``reset(seed=seeds[n])`` per env, bit-exact with the reference's PCG64 placement;
        ``seeds=None`` is ``reset()``: every env continues the generator it was last seeded with."""
        sptr = None
        if seeds is not None:
            sptr = self._check_tensor(seeds, torch.int64, (self.num_envs,), "seeds").data_ptr()
        optr = self.obs.data_ptr() if self.obs is not None else None
        _native.check(self._lib.cc_reset_seeded(self._h, sptr, optr, self.obs_code, self._stream()))
        return self.obs

    # ---- the hot path --------------------------------------------------------------------------
    def _fill_io(self, actions, order, policy, auto_reset) -> _abi.CCStepIO:
        io = self._io
        code = _policy_code(policy)
        shape = (self.num_envs, self.num_agents)
        if code == _abi.POLICIES["external"]:
            if actions is None:
                raise ValueError("step() needs `actions` unless an on-device policy is selected")
            io.actions = self._check_tensor(actions, torch.int8, shape, "actions").data_ptr()
        else:
            io.actions = None
        io.order = None if order is None else self._check_tensor(order, torch.int8, shape, "order").data_ptr()
        io.actions_out = self.actions_out.data_ptr()
        io.obs = None if self.obs is None else self.obs.data_ptr()
        io.reward = self.reward.data_ptr()
        io.agent_flags = self.agent_flags.data_ptr()
        io.agent_info = None if self.agent_info is None else self.agent_info.data_ptr()
        io.env_flags = self.env_flags.data_ptr()
        io.obs_dtype, io.reward_dtype = self.obs_code, self.reward_code
        io.policy = code
        io.auto_reset = int(self.auto_reset if auto_reset is None else auto_reset)
        return io

    def _output(self) -> StepOutput:
        return StepOutput(self.obs, self.reward, self.agent_flags, self.agent_info, self.env_flags, self.actions_out)

    def step(self, actions: torch.Tensor | None = None, *, order: torch.Tensor | None = None,
             policy: Any = "external", auto_reset: bool | None = None) -> StepOutput:
        """One env step for all N envs: ONE kernel launch on the current stream, no host sync.

        ``actions`` int8 [N, A] in {0..4} (reference ``step(action_dict)``; an absent dict entry
        is WAIT).  ``order`` int8 [N, A] optionally gives the caller's dict order (agent indices,
        negative = end of list).  ``policy`` in {"external","random","greedy","waiting"} selects an
        on-device action source instead.  Out-of-range actions raise ``ValueError`` at the next
        ``check_error()``."""
        io = self._fill_io(actions, order, policy, auto_reset)
        _native.check(self._lib.cc_step(self._h, C.byref(io), self._stream()))
        return self._output()

    def rollout(self, n_steps: int, policy: Any = "greedy", auto_reset: bool | None = None) -> StepOutput:
        """``n_steps`` fused steps with an on-device policy and no host round trip."""
        io = self._fill_io(None, None, policy, auto_reset)
        _native.check(self._lib.cc_rollout(self._h, C.byref(io), int(n_steps), self._stream()))
        return self._output()

    def rollout_trajectory(self, n_steps: int, policy: Any = "greedy", actions: torch.Tensor | None = None,
                           auto_reset: bool | None = None) -> dict:
        """``n_steps`` steps whose outputs are all kept, time-major: ``obs [T, N, A, L]``, ``reward``,
        ``agent_flags``, ``agent_info``, ``actions`` ``[T, N, A]``, ``env_flags [T, N]`` — the loop
        "policy -> step -> reset on done" of the reference's rollout scripts for N envs.  With the
        thread-per-env kernel (crews of 4 or 8) this is ONE launch that keeps each env's state in
        registers for the T steps; results equal T calls of ``step``.  ``policy="external"`` reads
        ``actions`` int8 ``[T, N, A]``.  The returned tensors are reused by the next call with the same T."""
        T, n, a = int(n_steps), self.num_envs, self.num_agents
        if T < 1:
            raise ValueError("n_steps must be positive")
        buf = getattr(self, "_traj", None)
        if buf is None or buf["reward"].shape[0] != T:
            out = self._output_tensor
            buf = self._traj = dict(
                obs=None if self.obs is None else out((T, n, a, self.obs_width), self.obs_torch_dtype),
                reward=out((T, n, a), self.reward_torch_dtype),
                agent_flags=out((T, n, a), torch.uint8),
                agent_info=None if self.agent_info is None else out((T, n, a), torch.uint8),
                env_flags=out((T, n), torch.uint8),
                actions=out((T, n, a), torch.int8))
        io = _abi.CCStepIO()
        code = _policy_code(policy)
        if code == _abi.POLICIES["external"]:
            if actions is None:
                raise ValueError("policy='external' needs `actions` [T, N, A]")
            io.actions = self._check_tensor(actions, torch.int8, (T, n, a), "actions").data_ptr()
        io.order = None
        io.actions_out = buf["actions"].data_ptr()
        io.obs = None if buf["obs"] is None else buf["obs"].data_ptr()
        io.reward = buf["reward"].data_ptr()
        io.agent_flags = buf["agent_flags"].data_ptr()
        io.agent_info = None if buf["agent_info"] is None else buf["agent_info"].data_ptr()
        io.env_flags = buf["env_flags"].data_ptr()
        io.obs_dtype, io.reward_dtype, io.policy = self.obs_code, self.reward_code, code
        io.auto_reset = int(self.auto_reset if auto_reset is None else auto_reset)
        _native.check(self._lib.cc_rollout_fused(self._h, C.byref(io), T, self._stream()))
        return buf

    def policy_actions(self, policy: Any, out: torch.Tensor | None = None) -> torch.Tensor:
        """Actions of a baseline policy for the current state (``policy.get_action`` for every agent)."""
        out = self.actions_out if out is None else self._check_tensor(out, torch.int8, (self.num_envs, self.num_agents), "out")
        _native.check(self._lib.cc_policy_actions(self._h, _policy_code(policy), out.data_ptr(), self._stream()))
        return out

    def observe(self) -> torch.Tensor:
        if self.obs is None:
            raise ValueError("this env was created with obs_dtype='none'")
        _native.check(self._lib.cc_observe(self._h, self.obs.data_ptr(), self.obs_code, self._stream()))
        return self.obs

    # ---- host-buffer path (what a numpy / RLlib caller binds) --------------------------------------
    def make_host_buffers(self, pinned: bool = True, n_steps: int | None = None, obs: str | None = "same", actions_out: bool = True) -> dict:
        """Host tensors for ``step_host`` (``n_steps=None``: per-step shapes) or ``rollout_host``
        (time-major ``[n_steps, ...]``).  ``obs``: "same" = the env's obs dtype, or "float32" / "int8" /
        "table" / None for another delivery format of the same step.  ``actions_out=False``: the applied actions are not
        copied back (a caller that supplies the actions has them)."""
        n, a = self.num_envs, self.num_agents
        lead = () if n_steps is None else (int(n_steps),)
        mk = lambda shape, dt: torch.zeros(lead + shape, dtype=dt, pin_memory=pinned)  # noqa: E731
        if obs == "same":
            obs_t = None if self.obs is None else mk((n, a, self.obs_width), self.obs_torch_dtype)
        elif obs is None or obs == "none":
            obs_t = None
        else:
            dt, code = _OBS_TORCH[obs]
            obs_t = mk((n, a, 4 if code == _abi.OBS_TABLE else self.obs_len), dt)
        return dict(
            actions=mk((n, a), torch.int8), obs=obs_t,
            reward=mk((n, a), self.reward_torch_dtype), agent_flags=mk((n, a), torch.uint8),
            agent_info=None if self.agent_info is None else mk((n, a), torch.uint8),
            env_flags=mk((n,), torch.uint8), actions_out=mk((n, a), torch.int8) if actions_out else None,
        )

    def _host_io(self, host: dict, policy: Any, auto_reset: bool | None) -> _abi.CCStepIO:
        io = _abi.CCStepIO()
        code = _policy_code(policy)
        io.actions = host["actions"].data_ptr() if code == 0 else None
        io.order = None
        io.actions_out = None if host.get("actions_out") is None else host["actions_out"].data_ptr()
        obs = host["obs"]
        io.obs = None if obs is None else obs.data_ptr()
        io.reward = host["reward"].data_ptr()
        io.agent_flags = host["agent_flags"].data_ptr()
        io.agent_info = None if host.get("agent_info") is None else host["agent_info"].data_ptr()
        io.env_flags = host["env_flags"].data_ptr()
        if obs is None:
            io.obs_dtype = _abi.OBS_NONE
        elif obs.dtype == torch.float32:
            io.obs_dtype = _abi.OBS_FP32
        else:
            io.obs_dtype = _abi.OBS_TABLE if obs.shape[-1] == 4 else _abi.OBS_INT8
        io.reward_dtype = self.reward_code
        io.policy = code
        io.auto_reset = int(self.auto_reset if auto_reset is None else auto_reset)
        # everything enqueued on the current torch stream so far (set_state copies, earlier steps) happens first
        _native.check(self._lib.cc_order_after(self._h, self._stream()))
        return io

    def step_host(self, host: dict, *, policy: Any = "external", auto_reset: bool | None = None) -> dict:
        """``cc_step_host``: actions are read from HOST memory (``host['actions']``), the outputs
        land in the HOST tensors of ``host``; the call returns when they are complete.  Chunks of envs
        are pipelined over three streams (copy in / kernel / copy out)."""
        io = self._host_io(host, policy, auto_reset)
        _native.check(self._lib.cc_step_host(self._h, C.byref(io)))
        return host

    def rollout_host(self, host: dict, n_steps: int, *, policy: Any = "greedy", auto_reset: bool | None = None) -> dict:
        """``cc_rollout_host``: ``n_steps`` env-steps per env, every output time-major in the HOST tensors of
        ``host`` (``make_host_buffers(n_steps=T)``); chunks of envs are rolled out on the device while the
        previous chunk's slices stream to the host."""
        if host["reward"].shape[0] != int(n_steps):
            raise ValueError("host buffers must be time-major with n_steps slices: make_host_buffers(n_steps=T)")
        io = self._host_io(host, policy, auto_reset)
        _native.check(self._lib.cc_rollout_host(self._h, C.byref(io), int(n_steps)))
        return host

    def last_host_call(self) -> dict:
        """What the last ``step_host`` / ``rollout_host`` did (``cc_last_host_call``): chunks, envs per chunk, host threads that
        rebuilt rows (0: rows crossed PCIe), bytes copied in each direction."""
        out = (C.c_int64 * 5)()
        _native.check(self._lib.cc_last_host_call(self._h, out))
        return dict(zip(("chunks", "chunk_envs", "expand_threads", "h2d_bytes", "d2h_bytes"), (int(v) for v in out)))

    def set_host_chunk(self, chunk_envs: int) -> None:
        """Envs per chunk of the host pipeline (0 = automatic)."""
        _native.check(self._lib.cc_set_host_chunk(self._h, int(chunk_envs)))

    def set_host_expand(self, n_threads: int) -> None:
        """Rows of the host path rebuilt on the host from the compact table: ``n_threads`` host threads, -1 = all,
        0 = off (rows cross PCIe as the kernel wrote them), -2 = automatic (the default of a new env: all threads when
        the host has at least 8 and a call delivers at least 16 MiB of rows).  Same bytes either way."""
        _native.check(self._lib.cc_set_host_expand(self._h, int(n_threads)))

    def expand_table_host(self, table: torch.Tensor, out: torch.Tensor | None = None, dtype: torch.dtype = torch.float32,
                          n_threads: int = 0) -> torch.Tensor:
        """``cc_expand_obs_host``: HOST table ``[..., A, 4]`` int8 -> the reference's rows ``[..., A, 6+4A]``
        (observations.py:62-94), bit-identical to the kernels' ``float32`` / ``int8`` rows."""
        if table.device.type != "cpu" or table.dtype != torch.int8 or not table.is_contiguous() or tuple(table.shape[-2:]) != (self.num_agents, 4):
            raise ValueError(f"table must be a contiguous int8 CPU tensor of shape [..., {self.num_agents}, 4]")
        shape = tuple(table.shape[:-1]) + (self.obs_len,)
        if out is None:
            out = torch.empty(shape, dtype=dtype)
        if out.device.type != "cpu" or tuple(out.shape) != shape or not out.is_contiguous() or out.dtype not in (torch.float32, torch.int8):
            raise ValueError(f"out must be a contiguous float32 / int8 CPU tensor of shape {shape}")
        code = _abi.OBS_FP32 if out.dtype == torch.float32 else _abi.OBS_INT8
        n = table.numel() // (4 * self.num_agents)
        _native.check(self._lib.cc_expand_obs_host(C.byref(self.cfg), n, table.data_ptr(), out.data_ptr(), code, int(n_threads)))
        return out

    # ---- bookkeeping -----------------------------------------------------------------------------
    def stats(self) -> dict:
        """Episode statistics accumulated on the device (synchronises the current stream)."""
        st = _abi.CCStats()
        _native.check(self._lib.cc_stats_read(self._h, C.byref(st), self._stream()))
        return st.as_dict()

    def stats_device(self, out: torch.Tensor | None = None) -> torch.Tensor:
        """The statistics block as a float64 [8] DEVICE tensor (``distributed.STAT_KEYS`` order), with no host round trip:
        what the multi-GPU reduction all-reduces behind the step kernels."""
        raw = getattr(self, "_stats_raw", None)
        if raw is None:
            raw = self._stats_raw = torch.zeros(8, dtype=torch.int64, device=self.device)
        _native.check(self._lib.cc_stats_copy(self._h, raw.data_ptr(), self._stream()))
        vals = torch.cat([raw[:6].to(torch.float64), raw[6:].view(torch.float64)])
        if out is not None:
            out.copy_(vals)
            return out
        return vals

    def reset_stats(self) -> None:
        _native.check(self._lib.cc_stats_reset(self._h, self._stream()))

    def check_error(self) -> None:
        """Raise ``ValueError`` if any launch since the last call saw an invalid action (the
        reference raises inside ``step``, collectivecrossing.py:707-711)."""
        _native.check(self._lib.cc_check_error(self._h, self._stream()))

    @property
    def launch_count(self) -> int:
        return int(self._lib.cc_launch_count(self._h))

    @property
    def step_counter(self) -> int:
        return int(self._lib.cc_step_counter(self._h))

    def timing_begin(self) -> None:
        _native.check(self._lib.cc_timing_begin(self._h, self._stream()))

    def timing_end(self) -> float:
        ms = C.c_float()
        _native.check(self._lib.cc_timing_end(self._h, self._stream(), C.byref(ms)))
        return float(ms.value)

    # algorithmic bytes of one env-step (SURVEY.md §8d / DESIGN.md §5)
    def algorithmic_bytes_per_env_step(self) -> int:
        a = self.num_agents
        if self.obs_code == _abi.OBS_TABLE:   # s_obs = 0 plus the 4A-byte table
            return 12 * a + 17 + 4 * a
        return 12 * a + 17 + self.obs_code * a * (6 + 4 * a)
