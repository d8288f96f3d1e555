"""Test-only driver of tests/host_emul/emul_lp.cpp: the library's LP2 -> LP3 (lp3 or lp3_stored)
compiled for the host with branch counters (ORCA_EMUL_COUNT)."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "host_emul", "emul_lp.cpp")
_LIB = os.path.join(_HERE, "host_emul", "libemul_lp.so")
_CSRC = os.path.join(_HERE, "..", "collision_avoidance_b200", "csrc")

# counter slots (orca_core.cuh)
LP3_ROUNDS, LP1_CALLS, PROJ_FETCHES, LP3_INFEASIBLE, PARALLEL_SKIPPED, ANTIPARALLEL, LP3_STORED_ROUNDS = 0, 2, 4, 5, 6, 7, 8
LP3, LP3_STORED = 0, 1

_lib = None


def lib():
    global _lib
    if _lib is None:
        deps = [_SRC, os.path.join(_HERE, "host_emul", "host_vec_types.h")] + [os.path.join(_CSRC, f) for f in os.listdir(_CSRC)]
        if not os.path.exists(_LIB) or os.path.getmtime(_LIB) < max(os.path.getmtime(d) for d in deps):
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-DORCA_EMUL_COUNT",
                                   "-Wno-unknown-pragmas", "-I" + os.path.join(_HERE, "host_emul"), "-o", _LIB, _SRC])
        L = ctypes.CDLL(_LIB)
        f, i, p = ctypes.c_float, ctypes.c_int, ctypes.c_void_p
        L.emul_solve.argtypes = [p, i, i, f, f, f, i, p]
        L.emul_solve.restype = i
        L.emul_lp_counters.argtypes = [p, i]
        _lib = L
    return _lib


def emul_solve(lines, n, n_obst, radius, pref, variant):
    """(fail index, result float32[2]) of LP2 -> lp3 (variant 0) / lp3_stored (variant 1)."""
    lines = np.ascontiguousarray(lines, np.float32).reshape(-1, 4)
    assert lines.shape[0] == n
    out = np.zeros(2, np.float32)
    fail = lib().emul_solve(lines.ctypes.data, int(n), int(n_obst), float(np.float32(radius)), float(np.float32(pref[0])),
                            float(np.float32(pref[1])), int(variant), out.ctypes.data)
    return fail, out


def counters(reset=False):
    out = np.zeros(16, np.int64)
    lib().emul_lp_counters(out.ctypes.data, 1 if reset else 0)
    return out


def reset_counters():
    counters(reset=True)
