"""Test-only front-end of tests/host_emul/roadmap_oracle.cpp: the CPU oracle with RVO2's
queryVisibility and the roadmap of RVO2's obstacle example (Roadmap.cpp), restated literally.

``OracleSim`` is the oracle's ``PyRVOSimulator`` running on that library (the oracle compiled in
unchanged), plus ``queryVisibility``, ``roadmap_build`` and ``roadmap_pref``."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

from oracle.rvo2_oracle import PyRVOSimulator

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "host_emul", "roadmap_oracle.cpp")
_ORACLE_SRC = os.path.join(_HERE, "..", "oracle", "rvo2_oracle.cpp")
_LIB = os.path.join(_HERE, "host_emul", "libroadmap_oracle.so")

_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB) or os.path.getmtime(_LIB) < max(os.path.getmtime(_SRC), os.path.getmtime(_ORACLE_SRC)):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-shared",
                                   "-o", _LIB, _SRC])
        L = ctypes.CDLL(_LIB)
        f, i, p = ctypes.c_float, ctypes.c_int, ctypes.c_void_p
        fp = ctypes.POINTER(ctypes.c_float)
        sig = {
            "rvo_create": (p, [f, f, i, f, f, f, f, f, f]),
            "rvo_destroy": (None, [p]),
            "rvo_add_agent": (i, [p, f, f, f, i, f, f, f, f, f, f]),
            "rvo_add_agent_default": (i, [p, f, f]),
            "rvo_add_obstacle": (i, [p, fp, i]),
            "rvo_process_obstacles": (None, [p]),
            "rvo_num_agents": (i, [p]),
            "rvo_query_visibility": (i, [p, f, f, f, f, f]),
            "rvo_roadmap_build": (None, [p, p, i, i, f, p, p]),
            "rvo_roadmap_pref": (None, [p, p, i, i, p, p, p, p]),
        }
        for name, (res, args) in sig.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class OracleSim(PyRVOSimulator):
    """The oracle simulator with queryVisibility and Roadmap.cpp's roadmap."""

    def __init__(self, timeStep, neighborDist, maxNeighbors, timeHorizon, timeHorizonObst, radius, maxSpeed,
                 velocity=(0.0, 0.0)):
        self._L = lib()
        self._h = self._L.rvo_create(timeStep, neighborDist, int(maxNeighbors), timeHorizon, timeHorizonObst,
                                     radius, maxSpeed, float(velocity[0]), float(velocity[1]))
        self._buf = (ctypes.c_float * 4)()

    def queryVisibility(self, point1, point2, radius=0.0):
        return bool(self._L.rvo_query_visibility(self._h, float(point1[0]), float(point1[1]), float(point2[0]),
                                                 float(point2[1]), float(radius)))

    def roadmap_build(self, vertices, num_goals, radius):
        """Roadmap.cpp buildRoadmap: (adjacency bool [R, R], distToGoal float32 [G, R])."""
        xy = np.ascontiguousarray(vertices, np.float32).reshape(-1, 2)
        R, G = xy.shape[0], int(num_goals)
        adj = np.zeros((R, R), np.uint8)
        dist = np.zeros((G, R), np.float32)
        self._L.rvo_roadmap_build(self._h, xy.ctypes.data, R, G, float(radius), adj.ctypes.data, dist.ctypes.data)
        return adj.astype(bool), dist

    def roadmap_pref(self, vertices, dist, goals):
        """Roadmap.cpp setPreferredVelocities without the perturbation, for every agent (its own radius):
        (pref float32 [n, 2], minVertex int32 [n])."""
        xy = np.ascontiguousarray(vertices, np.float32).reshape(-1, 2)
        dist = np.ascontiguousarray(dist, np.float32)
        goals = np.ascontiguousarray(goals, np.int32)
        n = self.getNumAgents()
        pref = np.zeros((n, 2), np.float32)
        vertex = np.zeros(n, np.int32)
        self._L.rvo_roadmap_pref(self._h, xy.ctypes.data, xy.shape[0], dist.shape[0], dist.ctypes.data,
                                 goals.ctypes.data, pref.ctypes.data, vertex.ctypes.data)
        return pref, vertex


def oracle_world(polygons, params=None, process=True) -> OracleSim:
    """An oracle simulator holding ``polygons`` (processed unless ``process`` is False) and no agents."""
    p = params or dict(timeStep=0.25, neighborDist=15.0, maxNeighbors=10, timeHorizon=5.0, timeHorizonObst=5.0,
                       radius=2.0, maxSpeed=2.0)
    s = OracleSim(p["timeStep"], p["neighborDist"], p["maxNeighbors"], p["timeHorizon"], p["timeHorizonObst"],
                  p["radius"], p["maxSpeed"])
    for poly in polygons:
        s.addObstacle(poly)
    if process:
        s.processObstacles()
    return s
