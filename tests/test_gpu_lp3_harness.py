"""LP3 on the device, programme by programme: tests/device_harness/lp_harness.cu runs the library's
lp2 -> lp3 / lp3_stored (csrc/orca_core.cuh) with one programme per lane, in warps that mix short and
long programmes and lanes without one.  Every lane must return the oracle's fail index and result
bits, whichever lane and warp its programme sits in."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import _lp3_worlds as W
from oracle.rvo2_oracle import solve_lp

pytestmark = pytest.mark.gpu

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "device_harness", "lp_harness.cu")
_LIB = os.path.join(_HERE, "device_harness", "liblp_harness.so")
_CSRC = os.path.join(_HERE, "..", "collision_avoidance_b200", "csrc")
TPB = 64  # two warps per block; 2 x 22 shared line slots per thread


def _lib():
    from collision_avoidance_b200 import build
    deps = [_SRC] + [os.path.join(_CSRC, f) for f in os.listdir(_CSRC)]
    if not os.path.exists(_LIB) or os.path.getmtime(_LIB) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call([build.nvcc_path(), *build.NVCC_FLAGS, "-o", _LIB, _SRC])
    L = ctypes.CDLL(_LIB)
    L.lp_harness_run.argtypes = [ctypes.c_void_p] * 5 + [ctypes.c_int] * 3 + [ctypes.c_void_p] * 2
    L.lp_harness_run.restype = ctypes.c_int
    return L


def _oracle(progs):
    fails, res = [], []
    for lines, n_obst, vmax, pref in progs:
        f, r = solve_lp(lines, n_obst, vmax, pref)
        fails.append(f)
        res.append(r)
    return np.array(fails, np.int32), np.stack(res)


def _run(L, progs, lane_prog, variant):
    import torch
    kmax = L.lp_harness_max_lines()
    P = len(progs)
    lines = np.zeros((P, kmax, 4), np.float32)
    meta = np.zeros(P, np.int32)
    for j, (ln, n_obst, _, _) in enumerate(progs):
        assert len(ln) <= kmax
        lines[j, :len(ln)] = ln
        meta[j] = len(ln) | (n_obst << 8)
    radius = np.array([p[2] for p in progs], np.float32)
    pref = np.stack([p[3] for p in progs]).astype(np.float32)
    dev = [torch.from_numpy(a).cuda() for a in (lines, meta, radius, pref, np.asarray(lane_prog, np.int32))]
    T = len(lane_prog)
    out = torch.zeros(T, 2, dtype=torch.float32, device="cuda")
    fail = torch.full((T,), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    rc = L.lp_harness_run(*(t.data_ptr() for t in dev), T, variant, TPB, out.data_ptr(), fail.data_ptr())
    assert rc == 0, rc
    return fail.cpu().numpy(), out.cpu().numpy()


def _layouts(P, seed):
    """Lane -> programme maps: every programme in at least three different lanes and warps, about a
    quarter of the lanes without a programme."""
    rng = np.random.default_rng(seed)
    maps = []
    for rep in range(3):
        order = list(rng.permutation(P))
        lanes = []
        for p in order:
            while rng.random() < 0.25:
                lanes.append(-1)
            lanes.append(int(p))
        maps.append(lanes)
    return maps


@pytest.mark.parametrize("variant", [0, 1], ids=["lp3", "lp3_stored"])
@pytest.mark.parametrize("source", ["synthetic", "worlds"])
def test_device_lp_matches_oracle_in_every_lane(source, variant):
    progs = W.synthetic_programmes() if source == "synthetic" else W.library_programmes(k_values=(10, 16))
    if source == "worlds":
        # every LP3 programme and an equal number of the others (LP2 feasible: need = false in LP3's votes)
        rng = np.random.default_rng(5)
        fo = np.array([solve_lp(*p)[0] < len(p[0]) for p in progs])
        lp3 = np.flatnonzero(fo)
        rest = rng.choice(np.flatnonzero(~fo), size=min(len(lp3), int((~fo).sum())), replace=False)
        progs = [progs[j] for j in np.concatenate([lp3, rest])]
    ofail, ores = _oracle(progs)
    assert (ofail < np.array([len(p[0]) for p in progs])).sum() > 500
    L = _lib()
    for lanes in _layouts(len(progs), seed=variant):
        fail, res = _run(L, progs, lanes, variant)
        lanes = np.asarray(lanes)
        has = lanes >= 0
        idx = lanes[has]
        bad = np.flatnonzero((fail[has] != ofail[idx]) | (res[has].view(np.int32) != ores[idx].view(np.int32)).any(1))
        assert len(bad) == 0, [(int(idx[b]), int(fail[has][b]), int(ofail[idx[b]]), res[has][b], ores[idx[b]])
                               for b in bad[:3]]
