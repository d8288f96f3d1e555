"""CPU check of the step-kernel choice (csrc/step_plan.h compiled for the host): for every handle shape,
the path (tile or uniform grid) and the template arguments (K, KFULL, OL, HETERO) are the ones the
library has always launched.  Slim and full kernels give the same bits, so no parity test would notice
a wrong choice; this one does."""
import ctypes
import itertools
import os
import subprocess

import pytest

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "collision_avoidance_b200", "csrc")

SHIM = r"""
#include "step_plan.h"
extern "C" void plan(int N, int k, int grid_min_agents, int vert_stride, int per_env, int hetero, int no_slim, int* out) {
  orca_host::StepPlanInputs in;
  in.N = N;
  in.max_neighbors = k;
  in.grid_min_agents = grid_min_agents;
  in.vert_stride = vert_stride;
  in.per_env = per_env != 0;
  in.hetero = hetero != 0;
  in.no_slim = no_slim != 0;
  const orca_host::StepPlan p = orca_host::step_plan(in);
  out[0] = p.grid;
  out[1] = p.K;
  out[2] = p.kfull;
  out[3] = p.ol;
  out[4] = p.hetero;
}
extern "C" int pick_k(int k) { return orca_host::pick_k(k); }
"""


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("step_plan")
    src, so = d / "shim.cpp", d / "libstep_plan.so"
    src.write_text(SHIM)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-Werror", "-I" + CSRC, "-o", str(so),
                           str(src)])
    L = ctypes.CDLL(str(so))
    L.plan.argtypes = [ctypes.c_int] * 7 + [ctypes.c_void_p]
    return L


def plan(lib, N, k, gmin=257, vs=0, per_env=False, hetero=False, no_slim=False):
    out = (ctypes.c_int * 5)()
    lib.plan(N, k, gmin, vs, int(per_env), int(hetero), int(no_slim), out)
    return bool(out[0]), out[1], bool(out[2]), out[3], bool(out[4])


def expected(N, k, gmin, vs, per_env, hetero, no_slim):
    """The launchers' choice, restated: per-agent parameters first (K from the 5 / 10 / 16 ladder,
    lists never full, OL = 6 on both paths), then the uniform K ladder, then the slim K + 2 kernel,
    whose condition differs between the tile and the grid path."""
    grid = N >= gmin
    if hetero:
        return grid, 5 if k <= 5 else 10 if k <= 10 else 16, False, 6, True
    K, kfull = {5: (5, True), 10: (10, True)}.get(k, (16, False))
    ol = 6
    if k == 10 and not no_slim:
        if grid:
            world_verts, args_vert_stride = vs, (vs if per_env else 0)  # StepArgs.world_verts / .vert_stride
            if world_verts <= 4 and args_vert_stride == 0:
                ol = 2
        elif vs <= 4 and N <= 32:
            ol = 2
    return grid, K, kfull, ol, False


# (N, grid_min_agents): both sides of the default 257, and a lowered threshold that puts worlds of
# 32 agents or fewer on the grid path
SHAPES = [(16, 257), (32, 257), (33, 257), (256, 257), (257, 257), (1000, 257), (1, 2), (16, 2), (32, 32),
          (32, 33), (33, 33), (31, 30)]


def test_every_input_combination_matches_the_launchers(lib):
    seen = set()
    for (N, gmin), k, vs, per_env, hetero, no_slim in itertools.product(SHAPES, (0, 3, 5, 9, 10, 16), (0, 4, 5),
                                                                         (False, True), (False, True), (False, True)):
        got = plan(lib, N, k, gmin, vs, per_env, hetero, no_slim)
        assert got == expected(N, k, gmin, vs, per_env, hetero, no_slim), (N, gmin, k, vs, per_env, hetero, no_slim)
        seen.add(got[1:])
    # the (K, KFULL, OL, HETERO) combinations the library instantiates, and no other
    assert seen == {(5, True, 6, False), (10, True, 6, False), (10, True, 2, False), (16, False, 6, False),
                    (5, False, 6, True), (10, False, 6, True), (16, False, 6, True)}


@pytest.mark.parametrize("row", [
    # uniform k = 5: 5, full, never slim
    ((16, 5), (False, 5, True, 6, False)),
    ((300, 5), (True, 5, True, 6, False)),
    # uniform k = 10: slim on the tile up to 32 agents in worlds of at most 4 vertices
    ((32, 10, 257, 4), (False, 10, True, 2, False)),
    ((32, 10, 257, 4, True), (False, 10, True, 2, False)),
    ((33, 10), (False, 10, True, 6, False)),
    ((16, 10, 257, 5), (False, 10, True, 6, False)),
    ((16, 10, 257, 0, False, False, True), (False, 10, True, 6, False)),
    # ... and on the grid at any N, but per-env worlds only without vertices
    ((1000, 10, 257, 4), (True, 10, True, 2, False)),
    ((16, 10, 2, 0), (True, 10, True, 2, False)),
    ((16, 10, 2, 0, True), (True, 10, True, 2, False)),
    ((16, 10, 2, 4, True), (True, 10, True, 6, False)),
    ((1000, 10, 257, 5), (True, 10, True, 6, False)),
    ((1000, 10, 257, 0, False, False, True), (True, 10, True, 6, False)),
    # any other uniform k runs K = 16 with lists of k < K entries, k < 5 included
    ((16, 0), (False, 16, False, 6, False)),
    ((16, 3), (False, 16, False, 6, False)),
    ((16, 9), (False, 16, False, 6, False)),
    ((300, 16), (True, 16, False, 6, False)),
    # per-agent parameters: K = pick_k(k), never full, never slim
    ((16, 3, 257, 0, False, True), (False, 5, False, 6, True)),
    ((16, 0, 257, 0, False, True), (False, 5, False, 6, True)),
    ((16, 9, 257, 0, False, True), (False, 10, False, 6, True)),
    ((16, 10, 257, 0, False, True), (False, 10, False, 6, True)),
    ((300, 10, 257, 0, False, True), (True, 10, False, 6, True)),
    ((300, 16, 257, 4, True, True), (True, 16, False, 6, True)),
])
def test_table_rows(lib, row):
    args, want = row
    assert plan(lib, *args) == want


def test_pick_k(lib):
    assert [lib.pick_k(k) for k in range(18)] == [5] * 6 + [10] * 5 + [16] * 6 + [-1]
