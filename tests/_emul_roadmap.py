"""Test-only driver of tests/host_emul/emul_roadmap.cpp: the roadmap device functions of
csrc/orca_roadmap.cuh compiled for the host, built the way _emul_hetero.py builds its library."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "host_emul", "emul_roadmap.cpp")
_LIB = os.path.join(_HERE, "host_emul", "libemul_roadmap.so")
_CSRC = os.path.join(_HERE, "..", "collision_avoidance_b200", "csrc")

_lib = None


def lib():
    global _lib
    if _lib is None:
        deps = [_SRC] + [os.path.join(_CSRC, f) for f in os.listdir(_CSRC)]
        if not os.path.exists(_LIB) or os.path.getmtime(_LIB) < max(os.path.getmtime(d) for d in deps):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-DORCA_EMUL_COUNT",
                                   "-Wno-unknown-pragmas", "-I" + os.path.join(_HERE, "host_emul"), "-o", _LIB, _SRC])
        L = ctypes.CDLL(_LIB)
        p, i = ctypes.c_void_p, ctypes.c_int
        L.emul_rm_world_new.restype = p
        L.emul_rm_world_new.argtypes = [p, p, i]
        L.emul_rm_world_free.argtypes = [p]
        L.emul_rm_world_depth.argtypes = [p]
        L.emul_rm_counters.argtypes = [p, i]
        L.emul_rm_visibility.argtypes = [p, p, p, p, i, p]
        L.emul_rm_dist.argtypes = [p, p, i, i, p]
        L.emul_rm_dist.restype = i
        L.emul_rm_pref.argtypes = [p, p, i, i, p, p, p, p, i, p, p]
        _lib = L
    return _lib


class World:
    """Processed obstacle tables of one world, as orca_set_obstacles builds them."""

    def __init__(self, polygons):
        polys = [np.asarray(p, np.float32).reshape(-1, 2) for p in polygons]
        xy = np.ascontiguousarray(np.concatenate(polys) if polys else np.zeros((0, 2), np.float32))
        sizes = np.asarray([p.shape[0] for p in polys], np.int32)
        self._h = lib().emul_rm_world_new(xy.ctypes.data, sizes.ctypes.data, len(polys))
        assert self._h, "BSP too deep"

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            lib().emul_rm_world_free(h)

    def visibility(self, q1, q2, radii):
        q1 = np.ascontiguousarray(q1, np.float32).reshape(-1, 2)
        q2 = np.ascontiguousarray(q2, np.float32).reshape(-1, 2)
        radii = np.ascontiguousarray(np.broadcast_to(np.asarray(radii, np.float32), (q1.shape[0],)))
        out = np.zeros(q1.shape[0], np.uint8)
        lib().emul_rm_visibility(self._h, q1.ctypes.data, q2.ctypes.data, radii.ctypes.data, q1.shape[0], out.ctypes.data)
        return out.astype(bool)

    def pref(self, vertices, dist, pos, goals, radii):
        """(pref [n, 2], vertex [n]) of roadmap_pref_kernel's body."""
        xy = np.ascontiguousarray(vertices, np.float32).reshape(-1, 2)
        dist = np.ascontiguousarray(dist, np.float32)
        pos = np.ascontiguousarray(pos, np.float32).reshape(-1, 2)
        n = pos.shape[0]
        goals = np.ascontiguousarray(goals, np.int32).reshape(n)
        radii = np.ascontiguousarray(np.broadcast_to(np.asarray(radii, np.float32), (n,)))
        pref = np.zeros((n, 2), np.float32)
        vertex = np.zeros(n, np.int32)
        lib().emul_rm_pref(self._h, xy.ctypes.data, xy.shape[0], dist.shape[0], dist.ctypes.data, pos.ctypes.data,
                           goals.ctypes.data, radii.ctypes.data, n, pref.ctypes.data, vertex.ctypes.data)
        return pref, vertex


def counters(reset=True):
    """Case counts of the visibility walks since the last reset (see emul_roadmap.cpp)."""
    out = np.zeros(16, np.int64)
    lib().emul_rm_counters(out.ctypes.data, 1 if reset else 0)
    return out


def pack_adjacency(adj):
    """bool [R, R] -> the library's rows of ceil(R / 32) uint32 words (row u bit v)."""
    R = adj.shape[0]
    words = (R + 31) // 32
    padded = np.zeros((R, words * 32), np.uint8)
    padded[:, :R] = adj
    return np.ascontiguousarray(np.packbits(padded, axis=1, bitorder="little").view(np.uint32))


def relax_dist(vertices, adj, goal):
    """roadmap_dist_kernel's relaxation for one goal: (dist float32 [R], rounds)."""
    xy = np.ascontiguousarray(vertices, np.float32).reshape(-1, 2)
    words = pack_adjacency(np.asarray(adj, bool))
    out = np.zeros(xy.shape[0], np.float32)
    rounds = lib().emul_rm_dist(xy.ctypes.data, words.ctypes.data, xy.shape[0], int(goal), out.ctypes.data)
    return out, rounds
