"""Test-only driver of tests/host_emul/emul_lines.cpp: the ORCA-line query of csrc/orca_lines.cuh
compiled for the host, with the StepArgs mirror and obstacle tables of _emul and the per-agent
parameter records of _emul_hetero."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

import _emul
import _emul_hetero

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "host_emul", "emul_lines.cpp")
_LIB = os.path.join(_HERE, "host_emul", "libemul_lines.so")
_CSRC = os.path.join(_HERE, "..", "collision_avoidance_b200", "csrc")

COVERED, COLLISION_LINES = 9, 10   # counter slots (emul_lines.cpp)

_lib = None


def lib():
    global _lib
    if _lib is None:
        deps = [_SRC, os.path.join(_HERE, "host_emul", "host_vec_types.h")] + [os.path.join(_CSRC, f) for f in os.listdir(_CSRC)]
        if not os.path.exists(_LIB) or os.path.getmtime(_LIB) < max(os.path.getmtime(d) for d in deps):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-DORCA_EMUL_COUNT",
                                   "-Wno-unknown-pragmas", "-I" + os.path.join(_HERE, "host_emul"), "-o", _LIB, _SRC])
        L = ctypes.CDLL(_LIB)
        assert L.emul_lines_stepargs_size() == ctypes.sizeof(_emul.StepArgs)
        p, i = ctypes.c_void_p, ctypes.c_int
        L.emul_agent_lines.argtypes = [ctypes.POINTER(_emul.StepArgs), p, i, i, p, p, p]
        L.emul_agent_lines.restype = i
        L.emul_lines_counters.argtypes = [p, i]
        _lib = L
    return _lib


def counters(reset=True):
    out = np.zeros(16, np.int64)
    lib().emul_lines_counters(out.ctypes.data, 1 if reset else 0)
    return out


def agent_lines(params, pos, vel, *, world=None, agent_params=None, grid=False, max_lines=None):
    """(lines float32 [E, N, L, 4], count int32 [E, N], n_obst int32 [E, N]) of orca_agent_lines on host
    arrays.  params: snake-case handle parameters; agent_params: {name: [E, N]} or None; world: an
    _emul.World shared by the batch (its obstacle-free map built for the largest obstacle range).
    L = max_lines (default maxNeighbors + 64: every line).  Rows not written stay NaN."""
    pos = np.ascontiguousarray(pos, np.float32)
    vel = np.ascontiguousarray(vel, np.float32)
    E, N = pos.shape[0], pos.shape[1]
    f32 = np.float32
    a = _emul.StepArgs()
    a.E, a.N, a.envs_per_block, a.k = E, N, 1, int(params["max_neighbors"])
    dt = f32(params["time_step"])
    a.dt, a.inv_dt = dt, f32(1.0) / dt
    nd = f32(params["neighbor_dist"])
    a.nd_sq = nd * nd
    a.inv_th = f32(1.0) / f32(params["time_horizon"])
    a.inv_tho = f32(1.0) / f32(params["time_horizon_obst"])
    a.radius, a.vmax = f32(params["radius"]), f32(params["max_speed"])
    orange = f32(params["time_horizon_obst"]) * f32(params["max_speed"]) + f32(params["radius"])
    a.obst_range_sq = orange * orange
    table = None
    if agent_params is not None:
        table, max_nd = _emul_hetero.agent_param_table(params, E, N, agent_params)
        a.nd_sq = max_nd * max_nd
    p = _emul._ptr
    a.pos, a.vel = p(pos), p(vel)
    if world is not None and world.nv > 0:
        a.vert_pd, a.vert_link, a.bsp, a.bsp_seg = p(world.pd), p(world.link), p(world.bsp), p(world.seg)
        a.shared_nodes, a.vert_stride = world.nv, 0
        a.cull_rows, a.cull_geo = p(world.cull_rows), p(world.cull_geo)
    L = a.k + 64 if max_lines is None else int(max_lines)
    lines = np.full((E, N, max(L, 1), 4), np.nan, np.float32)
    count = np.full((E, N), -7, np.int32)
    n_obst = np.full((E, N), -7, np.int32)
    rc = lib().emul_agent_lines(ctypes.byref(a), p(table), 1 if grid else 0, L, p(lines), p(count), p(n_obst))
    assert rc == 0
    return lines[:, :, :L], count, n_obst
