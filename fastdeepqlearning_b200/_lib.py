"""ctypes binding of libfdql.so (C ABI declared in include/fdql.h).

There is no CPU fallback: if the library is missing, `lib()` raises.  Build it with
`python __graft_entry__.py` (or `make -C fastdeepqlearning_b200/csrc`)."""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfdql.so")

FDQL_OK, FDQL_EINVAL, FDQL_ECUDA, FDQL_EOVERSAMPLE, FDQL_ENOMEM = 0, -1, -2, -3, -4
MAX_KEYS = 24

ROLE_NONE, ROLE_REWARD, ROLE_TASK_DONE, ROLE_EPISODE_DONE, ROLE_EPISODE_STEP, ROLE_MC_RETURN, ROLE_ACHIEVED_GOAL, \
    ROLE_DESIRED_GOAL = range(8)
ROLE_BY_NAME = {"reward": ROLE_REWARD, "task_done": ROLE_TASK_DONE, "episode_done": ROLE_EPISODE_DONE,
                "episode_step": ROLE_EPISODE_STEP, "mc_return": ROLE_MC_RETURN, "achieved_goal": ROLE_ACHIEVED_GOAL,
                "desired_goal": ROLE_DESIRED_GOAL}
REWARD_NONE, REWARD_BITFLIP, REWARD_ALL_GEQ, REWARD_FIRST_GEQ, REWARD_WEIGHTED_PNORM = range(5)
GOAL_FINAL, GOAL_RANDOM, GOAL_FUTURE = range(3)
OPT_EXACT_EPISODE_STEP, OPT_EMIT_LEARNER_AUX, OPT_CORESIDENT = 1, 2, 4
APPEND_SQUASH_REWARDS = 1


class FdqlError(RuntimeError):
    pass


class OversampleError(Exception):
    """franQ/Replay/replay_memory.py:6"""


_lib = None
_lock = threading.Lock()

_p = C.c_void_p
_i64, _i32, _u32, _u64, _f32, _f64 = C.c_int64, C.c_int32, C.c_uint32, C.c_uint64, C.c_float, C.c_double
_pp = C.POINTER(C.c_void_p)

_SIGNATURES = {
    "fdql_last_error": (C.c_char_p, []),
    "fdql_version": (C.c_int, []),
    "fdql_arena_create": (C.c_int, [_i64, _i32, C.POINTER(_i32), C.POINTER(_i32), _i32, C.POINTER(_p)]),
    "fdql_arena_destroy": (C.c_int, [_p]),
    "fdql_arena_info": (C.c_int, [_p, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64)]),
    "fdql_arena_set_cursor": (C.c_int, [_p, _i64, _i64]),
    "fdql_arena_key_view": (C.c_int, [_p, _i32, C.POINTER(_p), C.POINTER(_i64), C.POINTER(_i32)]),
    "fdql_arena_meta_view": (C.c_int, [_p, _i32, C.POINTER(_p), C.POINTER(_i64), C.POINTER(_i32)]),
    "fdql_arena_link_state": (C.c_int, [_p, _i32, C.POINTER(_f64), C.POINTER(_i32)]),
    "fdql_arena_append": (C.c_int, [_p, _i64, _pp, _p]),
    "fdql_arena_append_host": (C.c_int, [_p, _i64, _pp, _p]),
    "fdql_arena_append_packed_host": (C.c_int, [_p, _i64, _p, _i32, C.POINTER(_i32), _u32, _p]),
    "fdql_commit_episodes": (C.c_int, [_p, _i32, _p, _p, _f64, _i32, _i32, C.POINTER(_f32), _i32, _p]),
    "fdql_her_flush_episodes": (C.c_int, [_p, _i32, _p, _p, _p, _p, _i32, C.POINTER(_f32), _i32, _f64, _i32, _p]),
    "fdql_action_onehot": (C.c_int, [_i64, _i32, _p, _p, _p, _p]),
    "fdql_vmap_flush_episodes": (C.c_int, [_p, _i32, _p, _p, _p, _i32, _i32, _i32, _i32, _i32, C.POINTER(_f32), _i32, _f64, _i32, _i32, _p]),
    "fdql_vmap_select_column": (C.c_int, [_p, _i64, _i32, _i64, _p, _i32, _i32, _i32, _i32, _i32, _i32, _p, _p, _p, _p, _p, _p, _p, _p]),
    "fdql_q3_duplicate": (C.c_int, [_p, _i64, _i32, _i64, _f64, _p]),
    "fdql_her_flush_episodes_given": (C.c_int, [_p, _i32, _p, _p, _p, _p, _i64, _p, _p, _p, _f64, _i32, _p]),
    "fdql_vmap_flush_episodes_given": (C.c_int, [_p, _i32, _p, _p, _p, _i32, _i32, _i32, _i32, _i64, _p, _p, _f64, _i32, _i32, _p]),
    "fdql_arena_reserve": (C.c_int, [_p, _i64, C.POINTER(_i64)]),
    "fdql_sample_streams": (C.c_int, [_p, _i64, _i32, _i32, _f32, _u64, _u64, _p, _p, _p, _p, _p]),
    "fdql_gather_rows": (C.c_int, [_p, _i64, _p, _pp, _p]),
    "fdql_sample_gather": (C.c_int, [_p, _i64, _i32, _i64, _p, _p, _p, _i32, C.POINTER(_f32), _i32, _f64, _u32, _i32, _pp,
                                     _p, _p, _p, _p]),
    "fdql_sample_gather_draw": (C.c_int, [_p, _i64, _i32, _i32, _f32, _u64, _u64, _p, _p, _p, _p, _i32, C.POINTER(_f32), _i32, _f64, _u32, _i32,
                                          _pp, _p, _p, _p, _p]),
    "fdql_fused_pass": (C.c_int, [_p, _i64, _i32, _i32, _f32, _u64, _u64, _p, _p, _p, _p, _i32, C.POINTER(_f32), _i32, _f64, _u32, _i32,
                                  _pp, _p, _p, _p, _i64, _i32, _i32, _p, _p, _p, _p, _p, _p, _p, _f32, _f32, _p, _p, _p, _p]),
    "fdql_debug_force_generic_gather": (C.c_int, [C.c_int]),
    "fdql_set_coresident": (C.c_int, [C.c_int]),
    "fdql_debug_tqc_warp_kernel": (C.c_int, [C.c_int]),
    "fdql_tqc_loss": (C.c_int, [_i64, _i32, _i32, _p, _p, _p, _p, _p, _p, _p, _f32, _f32, _p, _p, _p, _p, _p]),
    "fdql_tqc_loss_dev_alpha": (C.c_int, [_i64, _i32, _i32, _p, _p, _p, _p, _p, _p, _p, _p, _f32, _p, _p, _p, _p, _p]),
    "fdql_quantile_huber": (C.c_int, [_i64, _i32, _i32, _p, _p, _p, _p, _p, _p]),
    "fdql_sac_min_target_loss": (C.c_int, [_i64, _i32, _p, _p, _p, _p, _p, _p, _p, _f32, _f32, _p, _p, _p, _p]),
    "fdql_sac_min_target_loss_dev_alpha": (C.c_int, [_i64, _i32, _p, _p, _p, _p, _p, _p, _p, _p, _f32, _p, _p, _p, _p]),
    "fdql_hotpath_step_host": (C.c_int, [_p, _i64, _i32, _i64, _p, _p, _p, _i32, C.POINTER(_f32), _i32, _f64, _u32, _pp,
                                         _i32, _i32, _p, _p, _p, _f32, _p, _p, _p]),
    "fdql_per_create": (C.c_int, [_p, _i32, _f32, _f32, _f32, C.POINTER(_p)]),
    "fdql_per_destroy": (C.c_int, [_p]),
    "fdql_per_sample": (C.c_int, [_p, _i64, _i32, _f32, _u64, _u64, _p, _p, _p, _p, _p, _p, _p, _p]),
    "fdql_per_update": (C.c_int, [_p, _i64, _p, _p, _p, _p]),
    "fdql_per_apply_pending": (C.c_int, [_p, _p]),
    "fdql_per_view": (C.c_int, [_p, C.POINTER(_p), C.POINTER(_p)]),
    "fdql_per_level_view": (C.c_int, [_p, _i32, C.POINTER(_p), C.POINTER(_p), C.POINTER(_i64)]),
    "fdql_per_rebuild": (C.c_int, [_p, _p]),
    "fdql_fused_pass_per": (C.c_int, [_p, _i64, _i32, _f32, _u64, _u64, _p, _p, _p, _p, _p, _p, _p, _p, _i32, C.POINTER(_f32), _i32, _f64,
                                      _u32, _i32, _pp, _p, _p, _p, _i64, _i32, _i32, _p, _p, _p, _p, _p, _p, _p, _f32, _f32, _p, _p, _p,
                                      _p, _p, _p]),
}
EXPORTS = tuple(_SIGNATURES)


def lib():
    """Load libfdql.so once; raise (never fall back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise FdqlError(f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` "
                                f"(nvcc, sm_100a). This package has no CPU or PyTorch fallback.")
            h = C.CDLL(LIB_PATH)
            for name, (res, args) in _SIGNATURES.items():
                fn = getattr(h, name)  # AttributeError if the library does not export what fdql.h declares
                fn.restype, fn.argtypes = res, args
            _lib = h
    return _lib


def check(rc):
    if rc == FDQL_OK:
        return
    msg = lib().fdql_last_error().decode("utf-8", "replace")
    if rc == FDQL_EOVERSAMPLE:
        raise OversampleError(msg)
    if rc == FDQL_EINVAL:
        raise ValueError(msg)
    if rc == FDQL_ENOMEM:
        raise MemoryError(msg)
    raise FdqlError(f"libfdql error {rc}: {msg}")


def ptr_array(ptrs):
    arr = (C.c_void_p * len(ptrs))()
    for i, p in enumerate(ptrs):
        arr[i] = p
    return arr


def f32_array(vals):
    vals = list(vals) if vals is not None else []
    arr = (C.c_float * max(len(vals), 1))(*vals)
    return arr, len(vals)
