"""ctypes binding of include/sy_env.h (libsy_env.so).  No CPU fallback: if the CUDA library
has not been built this module raises, and so does everything that depends on it."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SY_LIB_PATH: profiling experiments only (kernel variants built side by side); the product loads the in-tree library
LIB_PATH = os.environ.get("SY_LIB_PATH") or os.path.join(_HERE, "libsy_env.so")

SY_ABI_VERSION = 4
SY_NUM_REWARD_WEIGHTS = 11
SY_MAX_AGENTS = 16
SY_NUM_STATS = 16
SY_MAX_GROUPS = 1024
SY_MAX_TOLL = 1048576
SY_MAX_TIMESTEP = 65533
INT32_MAX = 2 ** 31 - 1
SY_REWARD_FP64, SY_REWARD_FP32 = 0, 1
STAT_NAMES = [
    "env_steps", "episodes", "mrx_wins", "police_wins", "truncations", "out_of_money",
    "sum_episode_length", "sum_budget_spent", "sum_sq_episode_length", "sum_length_police_wins",
    "sum_length_mrx_wins", "sum_episode_budget_spent", "police_moves",
    "reveals", "sum_belief_ce_q24", "sum_sq_belief_ce_q24",
]
BELIEF_CE_SCALE = float(1 << 24)  # fixed-point scale of the two belief cross-entropy sums (include/sy_env.h)


class SyConfig(C.Structure):
    _fields_ = [
        ("struct_bytes", C.c_int32), ("device", C.c_int32), ("num_envs", C.c_int32), ("num_nodes", C.c_int32),
        ("num_police", C.c_int32), ("agent_money", C.c_int32), ("mrx_money", C.c_int32), ("max_timestep", C.c_int32),
        ("reveal_interval", C.c_int32), ("toll", C.c_int32), ("belief", C.c_int32), ("reward_mode", C.c_int32),
        ("auto_reset", C.c_int32), ("resample_graph", C.c_int32), ("env_offset", C.c_int64), ("seed", C.c_uint64),
        ("reward_weights", C.c_double * SY_NUM_REWARD_WEIGHTS), ("reveal_skip_prob", C.c_float), ("reserved0", C.c_int32),
    ]


class _PtrStruct(C.Structure):
    """pointer struct of include/sy_env.h: `struct_bytes` (ABI guard, filled in here) followed by void* members,
    constructed with the members positionally or by name"""

    def __init__(self, *args, **kw):
        names = [n for n, _ in self._fields_[1:]]
        super().__init__(C.sizeof(type(self)), *args, **{k: v for k, v in kw.items() if k in names})


class SyState(_PtrStruct):
    _fields_ = [("struct_bytes", C.c_uint64)] + [(n, C.c_void_p) for n in (
        "pos", "money", "timestep", "graph_id", "episode", "done", "visits", "belief", "belief_hint")]


class SyObs(_PtrStruct):
    _fields_ = [("struct_bytes", C.c_uint64)] + [(n, C.c_void_p) for n in (
        "action_mask", "node_features", "agent_budget", "mrx_revealed", "node_features_u8")]


class SyOut(_PtrStruct):
    _fields_ = [("struct_bytes", C.c_uint64)] + [(n, C.c_void_p) for n in (
        "reward", "reward64", "terminated", "truncated", "done", "winner", "stats", "status")]


class SyHostOut(_PtrStruct):
    _fields_ = [("struct_bytes", C.c_uint64)] + [(n, C.c_void_p) for n in (
        "reward", "terminated", "truncated", "done", "winner", "status")]


class SyGroup(C.Structure):
    _fields_ = [
        ("struct_bytes", C.c_uint64), ("reward_weights", C.c_double * SY_NUM_REWARD_WEIGHTS),
        ("agent_money", C.c_int32), ("reveal_interval", C.c_int32), ("reveal_skip_prob", C.c_float), ("reserved0", C.c_int32),
    ]


SY_HEUR_NONE, SY_HEUR_RANDOM, SY_HEUR_EVADE, SY_HEUR_CHASE, SY_HEUR_CHASE_BELIEF = 0, 1, 2, 3, 4


class SyHeuristic(C.Structure):
    _fields_ = [
        ("struct_bytes", C.c_uint64), ("mrx_kind", C.c_int32), ("police_kind", C.c_int32), ("explore_mrx", C.c_uint64),
        ("explore_police", C.c_uint64), ("last_seen", C.c_void_p),
    ]


# name -> (restype, argtypes); must list every function include/sy_env.h declares
SIGNATURES = {
    "sy_abi_version": (C.c_int, []),
    "sy_last_error": (C.c_char_p, []),
    "sy_launch_count": (C.c_int64, []),
    "sy_create": (C.c_int, [C.POINTER(SyConfig), C.POINTER(C.c_void_p)]),
    "sy_destroy": (None, [C.c_void_p]),
    "sy_set_option": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32]),
    "sy_set_seed": (C.c_int, [C.c_void_p, C.c_uint64]),
    "sy_set_reward_tables": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]),
    "sy_load_graphs": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "sy_read_graph_tables": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sy_generate_graphs": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_uint64, C.c_uint32,
                                     C.c_uint32, C.c_void_p, C.c_void_p]),
    "sy_read_graph_edges": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "sy_reset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(SyState),
                           C.POINTER(SyObs), C.c_void_p]),
    "sy_step": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(SyState), C.POINTER(SyObs), C.POINTER(SyOut), C.c_void_p]),
    "sy_step_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(SyState), C.POINTER(SyObs), C.POINTER(SyOut),
                               C.POINTER(SyHostOut), C.c_void_p]),
    "sy_step_i16": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(SyState), C.POINTER(SyObs), C.POINTER(SyOut), C.c_void_p]),
    "sy_step_host_i16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(SyState), C.POINTER(SyObs),
                                   C.POINTER(SyOut), C.POINTER(SyHostOut), C.c_void_p]),
    "sy_sample_actions_i16": (C.c_int, [C.c_void_p, C.POINTER(SyState), C.c_uint32, C.c_void_p, C.c_void_p]),
    "sy_step_deferred": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(SyState), C.POINTER(SyObs), C.POINTER(SyOut), C.c_void_p]),
    "sy_flush_observations": (C.c_int, [C.c_void_p, C.POINTER(SyState), C.POINTER(SyObs), C.c_void_p]),
    "sy_observations_pending": (C.c_int, [C.c_void_p]),
    "sy_step_i32": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(SyState), C.POINTER(SyObs), C.POINTER(SyOut), C.c_void_p]),
    "sy_step_host_i32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(SyState), C.POINTER(SyObs),
                                   C.POINTER(SyOut), C.POINTER(SyHostOut), C.c_void_p]),
    "sy_set_host_overlap": (C.c_int, [C.c_void_p, C.c_int32]),
    "sy_host_rollout_random": (C.c_int, [C.c_void_p, C.c_int32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(SyState),
                                         C.POINTER(SyObs), C.POINTER(SyOut), C.POINTER(SyHostOut), C.c_void_p]),
    "sy_sample_actions_host": (C.c_int, [C.c_void_p, C.POINTER(SyState), C.c_uint32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "sy_sample_actions_i32": (C.c_int, [C.c_void_p, C.POINTER(SyState), C.c_uint32, C.c_void_p, C.c_void_p]),
    "sy_sample_actions": (C.c_int, [C.c_void_p, C.POINTER(SyState), C.c_uint32, C.c_void_p, C.c_void_p]),
    "sy_heuristic_actions": (C.c_int, [C.c_void_p, C.POINTER(SyHeuristic), C.POINTER(SyState), C.POINTER(SyObs), C.c_uint32,
                                       C.c_void_p, C.c_void_p]),
    "sy_copy_segments": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sy_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "sy_set_groups": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(SyGroup), C.c_void_p, C.c_void_p]),
    "sy_group_stats": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "sy_set_group_tolls": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.c_void_p]),
    "sy_set_group_rules": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_void_p]),
    "sy_allreduce_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "sy_rollout_random_dev": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(SyState), C.POINTER(SyObs),
                                        C.POINTER(SyOut), C.c_void_p]),
    "sy_rollout_random": (C.c_int, [C.c_void_p, C.c_int32, C.c_uint32, C.c_void_p, C.POINTER(SyState), C.POINTER(SyObs),
                                    C.POINTER(SyOut), C.c_void_p]),
    "sy_action_mask_dense": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
}

_lib = None


class SyError(RuntimeError):
    pass


def load_library() -> C.CDLL:
    """dlopen libsy_env.so (built in-tree by `__graft_entry__.build()`); raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise SyError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built. Run "
            "`python -c 'import __graft_entry__ as g; g.build()'` at the repo root. There is no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    if lib.sy_abi_version() != SY_ABI_VERSION:
        raise SyError(f"ABI mismatch: library {lib.sy_abi_version()} vs binding {SY_ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise SyError(f"libsy_env error {rc}: {load_library().sy_last_error().decode()}")
