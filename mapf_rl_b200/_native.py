"""ctypes binding of libmapf_b200.so (include/mapf_b200.h).  No fallback: if the CUDA library is
missing and cannot be built, importing a compute entry point raises."""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

_lib = None

MAPF_OK, MAPF_EINVAL, MAPF_ECUDA, MAPF_EACTION, MAPF_EUNIQUE, MAPF_ENOMEM, MAPF_ENOSPACE = 0, -1, -2, -3, -4, -5, -6
MAPF_ESTATE, MAPF_EINTERNAL, MAPF_EINDEX, MAPF_EPRIORITY = -7, -8, -9, -10
ABI_VERSION = 2
# element types of mapf_obs_unpack (MAPF_DTYPE_*)
DTYPE_U8, DTYPE_F16, DTYPE_BF16 = 0, 1, 2
# reward codes (MAPF_RCODE_*): index into reward_fn in config.REWARD_ORDER; 5 = reset step (reward 0), and on a sized
# handle an absent agent slot
RCODE_RESET = 5


class EnvConfig(C.Structure):
    _fields_ = [("num_envs", C.c_int32), ("num_agents", C.c_int32), ("map_length", C.c_int32),
                ("obs_radius", C.c_int32), ("device", C.c_int32), ("reward_fn", C.c_float * 5)]


class ReplayView(C.Structure):
    _fields_ = [("obs_buf", C.c_void_p), ("comm_buf", C.c_void_p), ("hid_buf", C.c_void_p), ("act_buf", C.c_void_p),
                ("rew_buf", C.c_void_p), ("done_buf", C.c_void_p), ("size_buf", C.c_void_p),
                ("num_agents", C.c_int32), ("max_steps", C.c_int32), ("bt_steps", C.c_int32),
                ("forward_steps", C.c_int32), ("latent_dim", C.c_int32)]


class ReplayViewCompact(C.Structure):
    _fields_ = [("obs_bits", C.c_void_p), ("comm_bits", C.c_void_p), ("hid_buf", C.c_void_p), ("act_buf", C.c_void_p),
                ("rew_buf", C.c_void_p), ("done_buf", C.c_void_p), ("size_buf", C.c_void_p),
                ("num_agents", C.c_int32), ("max_steps", C.c_int32), ("bt_steps", C.c_int32),
                ("forward_steps", C.c_int32), ("latent_dim", C.c_int32)]


class RolloutIO(C.Structure):
    _fields_ = [("T", C.c_int32), ("d_actions", C.c_void_p), ("action_slots", C.c_int32), ("d_obs", C.c_void_p),
                ("obs_slots", C.c_int32), ("d_rewards", C.c_void_p), ("d_codes", C.c_void_p), ("d_done", C.c_void_p),
                ("d_steps", C.c_void_p), ("out_slots", C.c_int32), ("chains", C.c_int32)]


class PerCycleArgs(C.Structure):
    _fields_ = [("d_q_online", C.c_void_p), ("d_q_target_next", C.c_void_p), ("d_q_online_next", C.c_void_p),
                ("d_action", C.c_void_p), ("d_reward", C.c_void_p), ("d_done", C.c_void_p), ("d_steps", C.c_void_p),
                ("d_idx", C.c_void_p), ("n_update", C.c_int64), ("gamma", C.c_float), ("alpha", C.c_double),
                ("old_ptr", C.c_int64), ("ptr", C.c_int64), ("slot_steps", C.c_int64), ("d_td_out", C.c_void_p),
                ("d_prio_out", C.c_void_p),
                ("d_uniforms", C.c_void_p), ("n_sample", C.c_int64), ("d_sample_idx_out", C.c_void_p),
                ("d_sample_prio_out", C.c_void_p), ("d_sample_weight_out", C.c_void_p), ("beta", C.c_double)]


class ReplayBatch(C.Structure):
    _fields_ = [("obs", C.c_void_p), ("comm_mask", C.c_void_p), ("hidden", C.c_void_p), ("action", C.c_void_p),
                ("reward", C.c_void_p), ("done", C.c_void_p), ("steps", C.c_void_p), ("bt_steps", C.c_void_p)]


# name -> (restype, argtypes); must list every symbol include/mapf_b200.h declares
_vp, _i32, _i64, _f32, _f64, _u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double, C.c_uint64
SIGNATURES = {
    "mapf_abi_version": (C.c_int, []),
    "mapf_last_error": (C.c_char_p, []),
    "mapf_env_create": (C.c_int, [C.POINTER(EnvConfig), C.POINTER(_vp)]),
    "mapf_env_destroy": (C.c_int, [_vp]),
    "mapf_env_arena_bytes": (_i64, [_vp]),
    "mapf_env_load": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _vp, _vp]),
    "mapf_env_bfs_navi": (C.c_int, [_vp, _vp, _i32, _vp, _vp]),
    "mapf_env_plan_prioritized": (C.c_int, [_vp, _i32, _vp, _vp, _vp]),
    "mapf_env_plan_prioritized_orders": (C.c_int, [_vp, _i32, _i32, _u64, _u64, _vp, _vp, _vp, _vp, _vp]),
    "mapf_env_plan_lns": (C.c_int, [_vp, _i32, _i32, _i32, _u64, _u64, C.c_uint32, _vp, _vp, _vp, _vp]),
    "mapf_env_plan_repair": (C.c_int, [_vp, _i32, _i32, _i32, _u64, _u64, _vp, _vp, _vp, _vp]),
    "mapf_env_step_observe": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mapf_env_step_observe_ex": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mapf_env_observe": (C.c_int, [_vp, _vp, _vp, _vp]),
    "mapf_env_step_observe_rows": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mapf_env_observe_rows": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "mapf_env_step_observe_packed": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mapf_env_observe_packed": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "mapf_obs_unpack": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _vp, _vp]),
    "mapf_obs_unpack_present": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _i64, _i32, _vp, _vp]),
    "mapf_env_rollout": (C.c_int, [_vp, _i32, _vp, _i32, _vp, _i32, _vp, _vp, _vp, _i32, _i32, _vp]),
    "mapf_env_rollout_ex": (C.c_int, [_vp, C.POINTER(RolloutIO), _vp]),
    "mapf_env_set_autoreset": (C.c_int, [_vp, _i32, _u64, _u64, _u64, _f32, _vp]),
    "mapf_env_set_checks": (C.c_int, [_vp, _i32]),
    "mapf_env_episode_counts": (C.c_int, [_vp, _vp, _vp]),
    "mapf_env_rollout_plan": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "mapf_env_step_host": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mapf_env_step_host_codes": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mapf_debug_step_tuning": (C.c_int, [_i32, _i32, _i32]),
    "mapf_debug_step_host_mode": (C.c_int, [_i32]),
    "mapf_debug_rollout_tuning": (C.c_int, [_i32, _i32, _i32, _i32, _i32]),
    "mapf_debug_rollout_pregen": (C.c_int, [_i32]),
    "mapf_debug_rollout_tasks": (C.c_int, [_i32]),
    "mapf_env_comm_mask": (C.c_int, [_vp, _i32, _vp, _vp]),
    "mapf_env_comm_mask_packed": (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp]),
    "mapf_env_get_state": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mapf_env_set_state": (C.c_int, [_vp, _vp, _vp, _vp]),
    "mapf_env_status": (C.c_int, [_vp, _vp]),
    "mapf_env_reset": (C.c_int, [_vp, _vp, _u64, _u64, _f32, _vp]),
    "mapf_env_enable_sizes": (C.c_int, [_vp]),
    "mapf_env_load_sized": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mapf_env_reset_levels": (C.c_int, [_vp, _vp, _u64, _u64, _f32, _vp, _i32, _vp]),
    "mapf_env_get_sizes": (C.c_int, [_vp, _vp, _vp, _vp]),
    "mapf_per_create": (C.c_int, [_i64, _i32, C.POINTER(_vp)]),
    "mapf_per_destroy": (C.c_int, [_vp]),
    "mapf_per_tree_ptr": (_vp, [_vp]),
    "mapf_per_update": (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "mapf_per_sample": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, _f64, _vp]),
    "mapf_per_td_update": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _f32, _f64, _i64, _i64, _i64,
                                     _vp, _vp, _vp]),
    "mapf_replay_gather": (C.c_int, [C.POINTER(ReplayView), _vp, _i64, C.POINTER(ReplayBatch), _vp, _vp]),
    "mapf_replay_gather_compact": (C.c_int, [C.POINTER(ReplayViewCompact), _vp, _i64, C.POINTER(ReplayBatch), _vp, _vp]),
    "mapf_replay_gather_present": (C.c_int, [C.POINTER(ReplayViewCompact), _vp, _vp, _vp, _i64, _i64, C.POINTER(ReplayBatch),
                                             _vp, _vp]),
    "mapf_actor_td": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp]),
    "mapf_actor_td_n": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _f64, _vp, _vp]),
    "mapf_per_cycle": (C.c_int, [_vp, C.POINTER(PerCycleArgs), _vp]),
    "mapf_per_status": (C.c_int, [_vp, _vp]),
    "mapf_cbs_solve": (C.c_int, [_vp, _i32, _i32, _vp, _vp, _vp, _i32, _i32, _i64, _vp, _i32, _vp, _vp, _vp]),
    "mapf_cbs_solve_batch": (C.c_int, [_i32, _vp, _i32, _i32, _vp, _vp, _vp, _i32, _i32, _i64, _vp, _i32, _vp, _vp, _vp, _i32]),
}


class MapfError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libmapf_b200 error {code}: {msg}")
        self.code = code


def lib():
    """Load (building first if the in-tree .so is missing or stale and nvcc is present)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    if _build.is_stale():
        try:
            _build.build()
        except Exception as e:  # no nvcc on this box: use the shipped .so if there is one
            if not os.path.exists(path):
                raise ImportError(f"libmapf_b200.so is missing and could not be built ({e}); "
                                  "there is no CPU fallback") from e
    L = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)  # AttributeError = ABI mismatch, fail loudly
        fn.restype = res
        fn.argtypes = args
    if L.mapf_abi_version() != ABI_VERSION:
        raise ImportError("libmapf_b200.so ABI version mismatch")
    _lib = L
    return L


def check(code: int):
    if code != MAPF_OK:
        msg = lib().mapf_last_error().decode("utf-8", "replace")
        if code == MAPF_EACTION:
            raise AssertionError("action index out of range")  # environment.py:290
        if code in (MAPF_EUNIQUE, MAPF_ENOSPACE):
            raise RuntimeError(msg)  # 'unique' (environment.py:428) / 'no empty position' (environment.py:31)
        if code in (MAPF_ESTATE, MAPF_EINDEX):
            raise IndexError(msg)    # what numpy raises on an out-of-range coordinate / leaf index
        if code == MAPF_EPRIORITY:
            raise AssertionError(msg)  # assert np.all(priorities > 0) (buffer.py:74)
        raise MapfError(code, msg)
