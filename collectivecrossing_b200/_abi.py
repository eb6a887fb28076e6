"""ctypes mirrors of ``include/ccb200.h`` (structs, enums, flag bits).  Keep in lock-step with
the header; ``tests/test_abi.py`` checks sizes and exported symbols."""

from __future__ import annotations

import ctypes as C

ABI_VERSION = 2
MAX_AGENTS = 128

# cc_status
OK, ERR_INVALID_ARG, ERR_CUDA, ERR_UNSUPPORTED, ERR_INVALID_ACTION, ERR_RESET_STUCK, ERR_NOMEM = 0, -1, -2, -3, -4, -5, -6

REWARD_KINDS = {"default": 0, "simple_distance": 1, "binary": 2, "constant_negative": 3}
TERMINATED_KINDS = {"individual_at_destination": 0, "all_at_destination": 1}
OBS_NONE, OBS_INT8, OBS_FP32, OBS_TABLE = 0, 1, 4, 16
REWARD_F32, REWARD_F64 = 4, 8
POLICIES = {"external": 0, "random": 1, "greedy": 2, "waiting": 3}

F_ACTIVE, F_TERMINATED, F_TRUNCATED = 1, 2, 4
O_ACTIVE, O_TERMINATED, O_TRUNCATED, O_ALIVE_PREV, O_TERM_VALUE, O_TRUNC_VALUE, O_OBS_PRESENT = 1, 2, 4, 8, 16, 32, 64
I_IN_TRAM_AREA, I_AT_DOOR, I_ACTIVE, I_AT_DESTINATION = 1, 2, 4, 8
E_TERMINATED_ALL, E_TRUNCATED_ALL, E_WAS_RESET = 1, 2, 4
KERNEL_VARIANTS = {"auto": 0, "lanes": 1, "threads": 2}
RESET_RNG = {"philox": 0, "numpy": 1}


class CCConfig(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("division_y", C.c_int32),
        ("tram_left", C.c_int32), ("tram_right", C.c_int32), ("door_left", C.c_int32), ("door_right", C.c_int32),
        ("boarding_dest_y", C.c_int32), ("exiting_dest_y", C.c_int32),
        ("num_boarding", C.c_int32), ("num_exiting", C.c_int32),
        ("max_steps", C.c_int32), ("reward_kind", C.c_int32), ("terminated_kind", C.c_int32),
        ("reward_params", C.c_double * 4),
    ]

    @property
    def num_agents(self) -> int:
        return self.num_boarding + self.num_exiting

    @property
    def obs_len(self) -> int:
        return 6 + 4 * self.num_agents


class CCStepIO(C.Structure):
    _fields_ = [
        ("actions", C.c_void_p), ("order", C.c_void_p), ("actions_out", C.c_void_p),
        ("obs", C.c_void_p), ("reward", C.c_void_p),
        ("agent_flags", C.c_void_p), ("agent_info", C.c_void_p), ("env_flags", C.c_void_p),
        ("obs_dtype", C.c_int32), ("reward_dtype", C.c_int32), ("policy", C.c_int32), ("auto_reset", C.c_int32),
    ]


class CCStats(C.Structure):
    _fields_ = [
        ("env_steps", C.c_int64), ("episodes", C.c_int64), ("terminated_all", C.c_int64),
        ("truncated_all", C.c_int64), ("arrivals", C.c_int64), ("episode_length_sum", C.c_int64),
        ("episode_return_sum", C.c_double), ("reward_sum", C.c_double),
    ]

    def as_dict(self) -> dict:
        return {name: getattr(self, name) for name, _ in self._fields_}


# name -> (restype, argtypes); every symbol include/ccb200.h declares
_P, _I32, _I64, _U64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
EXPORTS = {
    "cc_create": (C.c_int, [C.POINTER(CCConfig), _I64, C.c_int, _I64, _U64, C.POINTER(_P)]),
    "cc_destroy": (None, [_P]),
    "cc_attach_state": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "cc_set_state": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "cc_get_state": (C.c_int, [_P, _P, _P, _P, _P, _P]),
    "cc_set_state_host": (C.c_int, [_P, _P, _P, _P, _P]),
    "cc_get_state_host": (C.c_int, [_P, _P, _P, _P, _P]),
    "cc_step": (C.c_int, [_P, C.POINTER(CCStepIO), _P]),
    "cc_step_host": (C.c_int, [_P, C.POINTER(CCStepIO)]),
    "cc_rollout_host": (C.c_int, [_P, C.POINTER(CCStepIO), _I32]),
    "cc_set_host_chunk": (C.c_int, [_P, _I64]),
    "cc_set_host_expand": (C.c_int, [_P, _I32]),
    "cc_order_after": (C.c_int, [_P, _P]),
    "cc_expand_obs_host": (C.c_int, [C.POINTER(CCConfig), _I64, _P, _P, _I32, _I32]),
    "cc_get_rng_state": (C.c_int, [_P, _P, _P]),
    "cc_set_rng_state": (C.c_int, [_P, _P, _P]),
    "cc_rng_seeded": (_I32, [_P]),
    "cc_set_reset_rng": (C.c_int, [_P, _I32]),
    "cc_reset_rng": (_I32, [_P]),
    "cc_rollout": (C.c_int, [_P, C.POINTER(CCStepIO), _I32, _P]),
    "cc_rollout_fused": (C.c_int, [_P, C.POINTER(CCStepIO), _I32, _P]),
    "cc_reset": (C.c_int, [_P, _P, _P, _I32, _P]),
    "cc_reset_seeded": (C.c_int, [_P, _P, _P, _I32, _P]),
    "cc_policy_actions": (C.c_int, [_P, _I32, _P, _P]),
    "cc_observe": (C.c_int, [_P, _P, _I32, _P]),
    "cc_stats_read": (C.c_int, [_P, C.POINTER(CCStats), _P]),
    "cc_stats_reset": (C.c_int, [_P, _P]),
    "cc_stats_copy": (C.c_int, [_P, _P, _P]),
    "cc_check_error": (C.c_int, [_P, _P]),
    "cc_num_envs": (_I64, [_P]),
    "cc_num_agents": (_I32, [_P]),
    "cc_obs_len": (_I32, [_P]),
    "cc_step_counter": (_U64, [_P]),
    "cc_set_step_counter": (C.c_int, [_P, _U64]),
    "cc_launch_count": (_I64, [_P]),
    "cc_set_kernel_variant": (C.c_int, [_P, _I32]),
    "cc_last_kernel_variant": (_I32, [_P]),
    "cc_last_kernel_name": (C.c_char_p, [_P]),
    "cc_last_host_call": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "cc_timing_begin": (C.c_int, [_P, _P]),
    "cc_timing_end": (C.c_int, [_P, _P, C.POINTER(C.c_float)]),
    "cc_device_alloc": (C.c_int, [C.c_int, C.c_size_t, C.POINTER(_P), C.POINTER(_I32)]),
    "cc_device_free": (C.c_int, [_P]),
    "cc_last_error": (C.c_char_p, []),
    "cc_abi_version": (C.c_int, []),
}


def bind(lib: C.CDLL, table: dict = EXPORTS) -> C.CDLL:
    """Attach restype/argtypes; raises AttributeError naming the first missing symbol."""
    for name, (res, args) in table.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib
