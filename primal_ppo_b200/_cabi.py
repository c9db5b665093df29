"""ctypes binding of ``libmapf_b200.so`` (the C ABI in ``include/mapf_b200.h``).

There is NO fallback: if the shared library is missing or a CUDA call fails, an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libmapf_b200.so")

EXPORTED = ["mapf_abi_version", "mapf_last_error", "mapf_create", "mapf_destroy", "mapf_reset", "mapf_evaluate",
            "mapf_joint_step", "mapf_step", "mapf_observe", "mapf_bfs", "mapf_bfs_refresh", "mapf_gae", "mapf_gae2",
            "mapf_get_state", "mapf_get_counters", "mapf_step_observe_host", "mapf_step_observe",
            "mapf_sample_actions", "mapf_generate_scenario",
            "mapf_observe_bf16", "mapf_step_observe_bf16", "mapf_state_bytes", "mapf_save_state", "mapf_load_state",
            "mapf_get_human", "mapf_host_layout", "mapf_step_observe_host_begin", "mapf_step_observe_host_wait", "mapf_decode_results_host", "mapf_checksum_rows", "mapf_adv_moments", "mapf_ppo_loss",
            "mapf_observe_bits", "mapf_step_observe_bits", "mapf_unpack_obs", "mapf_unpack_obs_host", "mapf_astar4_paths"]
ABI_VERSION = 2

def obs_bits_words(C: int, F: int) -> int:
    """MAPF_OBS_BITS_WORDS(C, F): u32 words of one agent's record in the bit-packed observation format."""
    return (C * F * F + 31) // 32


ERR_NO_VIABLE, ERR_FIX_ITER_CAP, ERR_BAD_ACTION, ERR_TAPE, ERR_NO_FREE_CELL = 1, 2, 4, 8, 64


class MapfConfig(C.Structure):
    _fields_ = [("num_worlds", C.c_int32), ("height", C.c_int32), ("width", C.c_int32), ("num_agents", C.c_int32),
                ("fov", C.c_int32), ("num_channel", C.c_int32), ("use_da", C.c_int32), ("use_hp", C.c_int32),
                ("queue_len", C.c_int32), ("trace_len", C.c_int32), ("tape_stride", C.c_int32),
                ("hp5_per_tick", C.c_int32), ("seed", C.c_uint64), ("device", C.c_int32), ("world_offset", C.c_int32),
                ("goal_sampling", C.c_int32), ("reserved0", C.c_int32)]


class MapfGenConfig(C.Structure):
    _fields_ = [("num_worlds", C.c_int32), ("height", C.c_int32), ("width", C.c_int32), ("num_agents", C.c_int32),
                ("kind", C.c_int32), ("density_mode", C.c_int32), ("density_lo", C.c_float), ("density_hi", C.c_float),
                ("size_lo", C.c_int32), ("size_hi", C.c_int32), ("queue_len", C.c_int32), ("trace_len", C.c_int32),
                ("human_loops", C.c_int32), ("human_path", C.c_int32), ("seed", C.c_uint64), ("world_offset", C.c_int32), ("device", C.c_int32)]


class MapfScenario(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("obst", "starts", "goal_queue", "htrace", "hlen", "hp5", "tape", "tape_len", "dims")]


class MapfStepOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("status", "reward", "cost", "train_valid", "goals_reached", "violated", "shadow_goals",
                 "fixed_actions", "packed", "good_actions")]


MapfStepOutHost = MapfStepOut   # same layout, host pointers


class MapfHostLayout(C.Structure):
    _fields_ = [(n, C.c_int64) for n in
                ("slot_bytes", "off_reward", "off_cost", "off_shadow_goals", "off_status", "off_goals_reached",
                 "off_violated", "off_fixed_actions", "off_train_valid", "off_packed")]


HOST_TRAIN_VALID, HOST_COMPACT, HOST_OBS_BF16, HOST_OBS_BITS, HOST_OBS = 1, 2, 4, 8, 16


class MapfPpoLossConfig(C.Structure):
    _fields_ = [("clip_range", C.c_float), ("entropy_coef", C.c_float), ("value_coef", C.c_float), ("valid_coef", C.c_float),
                ("cost_value_coef", C.c_float), ("cost_coef", C.c_float), ("lagrangian", C.c_float),
                ("minus_adv_with_cadv", C.c_int32), ("n_global", C.c_double), ("adv_mean", C.c_double),
                ("adv_std", C.c_double), ("cadv_mean", C.c_double), ("cadv_std", C.c_double)]


PPO_LOSS_MAX_BLOCKS, PPO_LOSS_STATS = 1024, 10


class MapfError(RuntimeError):
    pass


_lib = None


def load_library():
    """Loads the CUDA library; raises if it has not been built (python -m primal_ppo_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MapfError(f"{LIB_PATH} is missing: build it with `python -m primal_ppo_b200.build` "
                        f"(nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    lib.mapf_abi_version.restype = C.c_int
    lib.mapf_last_error.restype = C.c_char_p
    lib.mapf_create.argtypes = [C.POINTER(MapfConfig), C.POINTER(vp)]
    lib.mapf_destroy.argtypes = [vp]
    lib.mapf_reset.argtypes = [vp, C.POINTER(MapfScenario), vp]
    lib.mapf_evaluate.argtypes = [vp, vp, C.POINTER(MapfStepOut), vp]
    lib.mapf_joint_step.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    lib.mapf_step.argtypes = [vp, vp, C.POINTER(MapfStepOut), vp]
    lib.mapf_observe.argtypes = [vp, vp, vp, vp]
    lib.mapf_step_observe.argtypes = [vp, vp, C.POINTER(MapfStepOut), vp, vp, vp]
    lib.mapf_observe_bf16.argtypes = [vp, vp, vp, vp]
    lib.mapf_step_observe_bf16.argtypes = [vp, vp, C.POINTER(MapfStepOut), vp, vp, vp]
    lib.mapf_observe_bits.argtypes = [vp, vp, vp, vp]
    lib.mapf_step_observe_bits.argtypes = [vp, vp, C.POINTER(MapfStepOut), vp, vp, vp]
    lib.mapf_unpack_obs.argtypes = [vp, i64, i32, i32, i32, vp, i64, i32, vp, vp]
    lib.mapf_unpack_obs_host.argtypes = [vp, i64, i32, i32, i32, vp, i64, i32, vp]
    lib.mapf_bfs.argtypes = [vp, vp, i64, vp, vp]
    lib.mapf_bfs_refresh.argtypes = [vp, vp, vp, vp]
    lib.mapf_gae.argtypes = [vp, vp, vp, vp, C.c_double, C.c_double, i32, i64, vp, vp, vp]
    lib.mapf_gae2.argtypes = [vp] * 7 + [C.c_double, C.c_double, i32, i64, vp, vp, vp, vp, vp]
    lib.mapf_adv_moments.argtypes = [vp, vp, vp, vp, i64, vp, vp]
    lib.mapf_ppo_loss.argtypes = [C.POINTER(MapfPpoLossConfig), i64] + [vp] * 17
    lib.mapf_sample_actions.argtypes = [vp, i64, C.c_uint64, C.c_uint32, vp, vp, vp]
    lib.mapf_generate_scenario.argtypes = [C.POINTER(MapfGenConfig)] + [vp] * 9
    lib.mapf_astar4_paths.argtypes = [vp, i64, i32, i32, vp, i32, vp, vp, vp]
    lib.mapf_state_bytes.argtypes = [vp]
    lib.mapf_save_state.argtypes = [vp, vp, vp]
    lib.mapf_load_state.argtypes = [vp, vp, vp]
    lib.mapf_get_state.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.mapf_get_counters.argtypes = [vp, vp, vp]
    lib.mapf_get_human.argtypes = [vp, vp, vp, vp]
    lib.mapf_step_observe_host.argtypes = [vp, vp, C.POINTER(MapfStepOutHost), vp, vp, vp, vp, vp, vp]
    lib.mapf_host_layout.argtypes = [vp, C.c_int, C.POINTER(MapfHostLayout)]
    lib.mapf_step_observe_host_begin.argtypes = [vp, vp, vp, C.c_int, vp, vp, vp, vp]
    lib.mapf_step_observe_host_wait.argtypes = [vp, C.c_int]
    lib.mapf_checksum_rows.argtypes = [vp, i64, i64, vp, vp]
    lib.mapf_decode_results_host.argtypes = [vp, i64, C.POINTER(MapfStepOutHost)]
    for n in EXPORTED:
        if n not in ("mapf_last_error",):
            getattr(lib, n).restype = C.c_int
    lib.mapf_state_bytes.restype = C.c_int64
    lib.mapf_last_error.restype = C.c_char_p
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load_library().mapf_last_error().decode("utf-8", "replace")
        raise MapfError(f"{what} failed (code {rc}): {msg}")
