"""The C oracle with numpy-mode placements (``tests/native/cc_oracle_np.c``) — TEST INFRASTRUCTURE.

``NumpyOracleEnvs`` is ``oracle.OracleEnvs`` whose auto-reset and ``reset(mask)`` continue each env's numpy generator
``gen`` (seeded by ``reset_seeded``), as the device does under ``reset_rng="numpy"``.  The library is compiled once
per process into a temporary directory, so the source tree stays untouched."""

from __future__ import annotations

import atexit
import ctypes as C
import functools
import shutil
import subprocess
import tempfile
from pathlib import Path

import numpy as np

import oracle
from collectivecrossing_b200 import _abi
from oracle import _ptr

SRC = Path(__file__).resolve().parent / "native" / "cc_oracle_np.c"
_P, _I32, _I64, _U64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
_EXPORTS = {
    "cc_oracle_np_step": (C.c_int, [C.POINTER(_abi.CCConfig), _I64, _I64, _U64, _U64, _P, _P, _P, _P, _P,
                                    C.POINTER(_abi.CCStepIO), C.POINTER(_abi.CCStats), _P]),
    "cc_oracle_np_reset": (C.c_int, [C.POINTER(_abi.CCConfig), _I64, _P, _P, _P, _P, _P, _P, _P, _P, _I32]),
}


@functools.lru_cache(maxsize=None)
def lib() -> C.CDLL:
    tmp = tempfile.mkdtemp(prefix="cc_oracle_np_")
    atexit.register(shutil.rmtree, tmp, True)
    out = Path(tmp) / "libcc_oracle_np.so"
    subprocess.run(["gcc", "-O2", "-fPIC", "-fopenmp", "-std=c11", "-shared", "-o", str(out), str(SRC), "-lm"], check=True)
    return _abi.bind(C.CDLL(str(out)), _EXPORTS)


class NumpyOracleEnvs(oracle.OracleEnvs):
    def _gen(self):
        if not hasattr(self, "gen"):
            raise ValueError("numpy-mode placements continue the generators reset_seeded(seeds) seeds: seed them first")
        return self.gen

    def step(self, actions=None, *, order=None, policy="external", auto_reset=False,
             obs_dtype=_abi.OBS_INT8, reward_dtype=_abi.REWARD_F32, check=True):
        b = self._bufs(obs_dtype, reward_dtype)
        io = _abi.CCStepIO()
        if actions is not None:
            actions = np.ascontiguousarray(actions, np.int8).reshape(self.n, self.a)
        if order is not None:
            order = np.ascontiguousarray(order, np.int8).reshape(self.n, self.a)
        io.actions, io.order = _ptr(actions), _ptr(order)
        io.actions_out = _ptr(b["actions_out"])
        io.obs, io.reward = _ptr(b["obs"]), _ptr(b["reward"])
        io.agent_flags, io.agent_info, io.env_flags = _ptr(b["agent_flags"]), _ptr(b["agent_info"]), _ptr(b["env_flags"])
        io.obs_dtype, io.reward_dtype = obs_dtype, reward_dtype
        io.policy = _abi.POLICIES[policy] if isinstance(policy, str) else int(policy)
        io.auto_reset = int(bool(auto_reset))
        gen = self._gen()
        rc = lib().cc_oracle_np_step(C.byref(self.cfg), self.n, self.offset, self.seed, self.t, _ptr(self.x), _ptr(self.y),
                                     _ptr(self.flags), _ptr(self.step_count), _ptr(self.episode_return), C.byref(io),
                                     C.byref(self.stats), _ptr(gen))
        self.t += 1
        if check and rc != _abi.OK:
            raise ValueError(f"oracle step failed with status {rc}")
        out = dict(b)
        out["status"] = rc
        return out

    def reset(self, mask=None, obs_dtype=_abi.OBS_INT8):
        b = self._bufs(obs_dtype, _abi.REWARD_F32)
        if mask is not None:
            mask = np.ascontiguousarray(mask, np.uint8)
        gen = self._gen()
        rc = lib().cc_oracle_np_reset(C.byref(self.cfg), self.n, _ptr(mask), _ptr(gen), _ptr(self.x), _ptr(self.y),
                                      _ptr(self.flags), _ptr(self.step_count), _ptr(self.episode_return), _ptr(b["obs"]), obs_dtype)
        self.t += 1
        if rc != _abi.OK:
            raise RuntimeError(f"oracle reset failed with status {rc}")
        return b["obs"]
