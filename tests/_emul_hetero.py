"""Test-only driver of tests/host_emul/emul_hetero.cpp: the step with per-agent ORCA parameters
(the HETERO instantiation of the library's per-agent device code) compiled for the host.
Reuses the StepArgs mirror and the obstacle tables of _emul."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

import _emul

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "host_emul", "emul_hetero.cpp")
_LIB = os.path.join(_HERE, "host_emul", "libemul_hetero.so")
_CSRC = os.path.join(_HERE, "..", "collision_avoidance_b200", "csrc")

NAMES = ("neighbor_dist", "max_neighbors", "time_horizon", "time_horizon_obst", "radius", "max_speed")

_lib = None


def lib():
    global _lib
    if _lib is None:
        deps = [_SRC] + [os.path.join(_CSRC, f) for f in os.listdir(_CSRC)]
        if not os.path.exists(_LIB) or os.path.getmtime(_LIB) < max(os.path.getmtime(d) for d in deps):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-Wno-unknown-pragmas",
                                   "-I" + os.path.join(_HERE, "host_emul"), "-o", _LIB, _SRC])
        L = ctypes.CDLL(_LIB)
        assert L.emul_hetero_stepargs_size() == ctypes.sizeof(_emul.StepArgs)
        L.emul_hetero_step.argtypes = [ctypes.POINTER(_emul.StepArgs), ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
        L.emul_hetero_step.restype = ctypes.c_int
        _lib = L
    return _lib


def agent_param_table(params, E, N, arrays):
    """The records orca_set_agent_params packs (float32 [E*N, 8], same float32 expressions) and the
    largest neighbor distance.  arrays: {name: [E, N] array}; a missing name takes the handle value."""
    f32 = np.float32
    col = {}
    for name in NAMES:
        v = arrays.get(name)
        dt = np.int32 if name == "max_neighbors" else np.float32
        col[name] = np.full(E * N, params[name], dt) if v is None else np.asarray(v, dt).reshape(E * N)
    nd, th, tho = col["neighbor_dist"], col["time_horizon"], col["time_horizon_obst"]
    r, vmax = col["radius"], col["max_speed"]
    orange = tho * vmax + r
    t = np.zeros((E * N, 8), np.float32)
    t[:, 0], t[:, 1], t[:, 2], t[:, 3] = r, vmax, f32(1.0) / th, f32(1.0) / tho
    t[:, 4], t[:, 5] = nd * nd, orange * orange
    t[:, 6] = col["max_neighbors"].view(np.float32)
    return t, f32(nd.max())


def emul_step_hetero(params, pos, vel, agent_params, *, pref, world=None, want_neighbors=True, stats=None, grid=False,
                     nbr_hint=None):
    """One EXTERNAL-policy step of the heterogeneous body on host arrays, in place (pos/vel float32
    [E, N, 2]); returns the neighbor lists.  Handle values and grid sizes as orca_api.cu sets them."""
    E, N = pos.shape[0], pos.shape[1]
    f32 = np.float32
    table, nd = agent_param_table(params, E, N, agent_params)
    a = _emul.StepArgs()
    a.E, a.N, a.envs_per_block, a.k = E, N, 1, int(params["max_neighbors"])
    a.tile_grid_inv_cell = f32(1.0) / (nd * f32(1.001)) if (N > 32 and not grid and nd > 0) else f32(0.0)
    dt = f32(params["time_step"])
    a.dt, a.inv_dt, a.nd_sq = dt, f32(1.0) / dt, nd * nd
    a.inv_th = f32(1.0) / f32(params["time_horizon"])
    a.inv_tho = f32(1.0) / f32(params["time_horizon_obst"])
    a.radius, a.vmax = f32(params["radius"]), f32(params["max_speed"])
    orange = f32(params["time_horizon_obst"]) * f32(params["max_speed"]) + f32(params["radius"])
    a.obst_range_sq = orange * orange
    for arr in (pos, vel, pref):
        assert arr.flags["C_CONTIGUOUS"]
    p = _emul._ptr
    a.pos, a.vel, a.pref = p(pos), p(vel), p(pref)
    out = {}
    if want_neighbors:
        out["nbr_idx"] = np.full((E, N, a.k), -1, np.int32)
        out["nbr_cnt"] = np.zeros((E, N), np.int32)
        out["onbr_idx"] = np.full((E, N, 16), -1, np.int32)
        out["onbr_cnt"] = np.zeros((E, N), np.int32)
        a.nbr_idx, a.nbr_cnt = p(out["nbr_idx"]), p(out["nbr_cnt"])
        a.onbr_idx, a.onbr_cnt = p(out["onbr_idx"]), p(out["onbr_cnt"])
    a.stats = p(stats)
    if nbr_hint is not None:
        assert nbr_hint.dtype == np.float32 and nbr_hint.flags["C_CONTIGUOUS"]
        a.nbr_hint = p(nbr_hint)
        a.hint_slack = f32(2.5) * f32(params["max_speed"]) * dt + f32(1e-4)
    if world is not None and world.nv > 0:
        a.vert_pd, a.vert_link, a.bsp, a.bsp_seg = p(world.pd), p(world.link), p(world.bsp), p(world.seg)
        a.shared_nodes, a.vert_stride = world.nv, 0
        a.cull_rows, a.cull_geo = p(world.cull_rows), p(world.cull_geo)
    assert lib().emul_hetero_step(ctypes.byref(a), table.ctypes.data, 0, 1 if grid else 0) == 0
    return out
