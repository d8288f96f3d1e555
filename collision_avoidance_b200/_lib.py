"""ctypes binding of the C ABI in ``include/orca_b200.h``.

This is the thin layer the north star asks for: Python reaches the hand-written sm_100a
kernels only through ``liborca_b200.so``.  There is NO fallback: if the library is missing
or a call fails, an exception is raised (``OrcaLibraryError`` / ``RuntimeError`` /
``ValueError``), mirroring how ``rvo2`` surfaces C++ errors (SURVEY.md 8b conventions).
"""
from __future__ import annotations

import ctypes
import os

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# ORCA_B200_LIB lets a developer point at an experimental build of the same library
LIB_PATH = os.environ.get("ORCA_B200_LIB") or os.path.join(PKG_DIR, "liborca_b200.so")

ORCA_OK = 0
ORCA_ERR_INVALID = -1
ORCA_ERR_CUDA = -2
ORCA_ERR_UNSUPPORTED = -3
ORCA_ERR_STATE = -4

POLICY_EXTERNAL, POLICY_GOAL, POLICY_RL, POLICY_ALAN = 0, 1, 2, 3
DONE_NONE, DONE_GOAL_RADIUS, DONE_X_BELOW, DONE_GOAL_RADIUS_DEFERRED = 0, 1, 2, 3

STAT_AGENT_STEPS, STAT_FINISHED, STAT_COLLISIONS, STAT_LP3_CALLS, STAT_OVERFLOW = 0, 1, 2, 3, 4
STAT_SUM_ARRIVAL, STAT_SUM_ARRIVAL2, STAT_SUM_REWARD, STAT_COUNT = 5, 6, 7, 8

HOST_UPLOAD_STATE, HOST_AUX_UNCHANGED = 1, 2

MAX_OBST_NEIGHBORS = 16
MAX_OBST_LINES = 6         # obstacle lines of the step's fast path (orca_b200.h ORCA_MAX_OBST_LINES)
SLOW_MAX_OBST = 64         # obstacle lines the uncapped path holds (ORCA_SLOW_MAX_OBST)
MAX_ACTIONS = 16

# every symbol include/orca_b200.h declares (tests check the .so exports all of them)
EXPORTED_SYMBOLS = (
    "orca_abi_version", "orca_last_error", "orca_create", "orca_destroy", "orca_get_params", "orca_set_agent_params",
    "orca_set_obstacles", "orca_obstacle_vertex_count", "orca_get_obstacle_vertices",
    "orca_query_visibility", "orca_set_roadmap", "orca_get_roadmap", "orca_roadmap_pref_velocity",
    "orca_step", "orca_env_step", "orca_env_step_many", "orca_neighbors", "orca_agent_lines", "orca_observe", "orca_step_host", "orca_step_host_ex", "orca_policy_mlp", "orca_policy_mlp_fp32", "orca_launch_count",
)


class OrcaLibraryError(ImportError):
    pass


class OrcaParams(ctypes.Structure):
    _fields_ = [
        ("time_step", ctypes.c_float),
        ("neighbor_dist", ctypes.c_float),
        ("max_neighbors", ctypes.c_int32),
        ("time_horizon", ctypes.c_float),
        ("time_horizon_obst", ctypes.c_float),
        ("radius", ctypes.c_float),
        ("max_speed", ctypes.c_float),
    ]


_vp = ctypes.c_void_p


class OrcaEnvStepArgs(ctypes.Structure):
    _fields_ = [
        ("struct_size", ctypes.c_uint32),
        ("policy", ctypes.c_int32),
        ("done_mode", ctypes.c_int32),
        ("_pad0", ctypes.c_int32),
        ("pos_dev", _vp),
        ("vel_dev", _vp),
        ("pref_dev", _vp),
        ("goal_dev", _vp),
        ("goal2_dev", _vp),
        ("action_theta_dev", _vp),
        ("rl_reward_scale", ctypes.c_float),
        ("done_x_threshold", ctypes.c_float),
        ("alan_weights_dev", _vp),
        ("alan_actions_dev", _vp),
        ("alan_action_out_dev", _vp),
        ("alan_uniform_in_dev", _vp),
        ("alan_num_actions", ctypes.c_int32),
        ("alan_window_steps", ctypes.c_int32),
        ("alan_gamma", ctypes.c_float),
        ("alan_temp", ctypes.c_float),
        ("rng_seed", ctypes.c_uint64),
        ("alan_num_actions_env_dev", _vp),
        ("alan_actions_env_stride", ctypes.c_int32),
        ("_pad1", ctypes.c_int32),
        ("reward_dev", _vp),
        ("agent_done_dev", _vp),
        ("arrival_time_dev", _vp),
        ("env_step_dev", _vp),
        ("env_done_cnt_dev", _vp),
        ("nbr_idx_dev", _vp),
        ("nbr_cnt_dev", _vp),
        ("obst_nbr_idx_dev", _vp),
        ("obst_nbr_cnt_dev", _vp),
        ("stats_dev", _vp),
    ]


class OrcaMlpWeights(ctypes.Structure):
    _fields_ = [
        ("struct_size", ctypes.c_uint32),
        ("in_dim", ctypes.c_int32),
        ("hidden_dim", ctypes.c_int32),
        ("out_dim", ctypes.c_int32),
        ("w1_dev", _vp), ("b1_dev", _vp), ("w2_dev", _vp), ("b2_dev", _vp), ("w3_dev", _vp), ("b3_dev", _vp),
    ]


_lib = None


def load() -> ctypes.CDLL:
    """Load liborca_b200.so (built in-tree by ``collision_avoidance_b200.build``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise OrcaLibraryError(
            f"{LIB_PATH} is missing: build it with `python -m collision_avoidance_b200.build` "
            "(nvcc, sm_100a).  There is no CPU fallback.")
    L = ctypes.CDLL(LIB_PATH)
    i, f = ctypes.c_int, ctypes.c_float
    hp = ctypes.c_void_p
    L.orca_abi_version.restype = i
    L.orca_last_error.restype = ctypes.c_char_p
    L.orca_create.argtypes = [ctypes.POINTER(OrcaParams), i, i, i, ctypes.POINTER(hp)]
    L.orca_destroy.argtypes = [hp]
    L.orca_get_params.argtypes = [hp, ctypes.POINTER(OrcaParams), ctypes.POINTER(i), ctypes.POINTER(i)]
    L.orca_set_agent_params.argtypes = [hp, _vp, _vp, _vp, _vp, _vp, _vp]
    L.orca_set_obstacles.argtypes = [hp, _vp, _vp, i, _vp]
    L.orca_obstacle_vertex_count.argtypes = [hp, i]
    L.orca_get_obstacle_vertices.argtypes = [hp, i, _vp, _vp, _vp, _vp]
    L.orca_query_visibility.argtypes = [hp, _vp, _vp, _vp, f, i, _vp, _vp]
    L.orca_set_roadmap.argtypes = [hp, _vp, i, i, i, f]
    L.orca_get_roadmap.argtypes = [hp, i, _vp, _vp]
    L.orca_roadmap_pref_velocity.argtypes = [hp, _vp, _vp, _vp, _vp, _vp]
    L.orca_step.argtypes = [hp, _vp, _vp, _vp, _vp]
    L.orca_env_step.argtypes = [hp, ctypes.POINTER(OrcaEnvStepArgs), _vp]
    L.orca_env_step_many.argtypes = [hp, ctypes.POINTER(OrcaEnvStepArgs), i, _vp]
    L.orca_neighbors.argtypes = [hp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]
    L.orca_agent_lines.argtypes = [hp, _vp, _vp, i, _vp, _vp, _vp, _vp]
    L.orca_observe.argtypes = [hp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, i, i, _vp, _vp]
    L.orca_step_host.argtypes = [hp, _vp, _vp, _vp, i, i, i]
    L.orca_step_host_ex.argtypes = [hp, _vp, _vp, _vp, i, i, i]
    L.orca_step_host_ex.restype = i
    L.orca_policy_mlp.argtypes = [hp, _vp, ctypes.c_int64, ctypes.POINTER(OrcaMlpWeights), _vp, _vp]
    L.orca_policy_mlp_fp32.argtypes = [hp, _vp, ctypes.c_int64, ctypes.POINTER(OrcaMlpWeights), _vp, _vp]
    L.orca_launch_count.argtypes = [hp]
    L.orca_launch_count.restype = ctypes.c_int64
    for name in EXPORTED_SYMBOLS:
        if name not in ("orca_last_error", "orca_launch_count"):
            getattr(L, name).restype = i
    if L.orca_abi_version() != 2:
        raise OrcaLibraryError(f"ABI version mismatch: library reports {L.orca_abi_version()}, binding expects 2")
    _lib = L
    return L


def check(rc: int) -> int:
    """Turn a negative OrcaStatus into the exception the rvo2 wrapper would raise."""
    if rc >= 0:
        return rc
    msg = load().orca_last_error().decode("utf-8", "replace")
    if rc == ORCA_ERR_INVALID:
        raise ValueError(msg)
    if rc == ORCA_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise RuntimeError(msg)
