"""CPU check of the ORCA-line query (csrc/orca_lines.cuh compiled for the host by
tests/host_emul/emul_lines.cpp) against the oracle: for every agent of every world, the lines, their
count and the number of obstacle lines equal ``Simulator::orca_lines`` after one oracle doStep from
the same state, bit for bit -- through the tile source and through the grid source."""
import functools

import numpy as np
import pytest

import _emul
import _emul_lines as el
from _agent_params import max_obstacle_range
from _lines_worlds import cpu_cases


@functools.lru_cache(maxsize=None)
def _cases():
    return cpu_cases()


def _env_lines(case, e, grid, max_lines=None):
    """The host build's (lines, count, n_obst) of env e, over that env's own obstacle world."""
    scn, P = case["scn"], case["params"]
    ap = case["agent_params"]
    orange = max_obstacle_range(scn, ap) if ap is not None else \
        P["time_horizon_obst"] * P["max_speed"] + P["radius"]
    world = _emul.World(case["polys"][e], obst_range=float(orange)) if case["polys"][e] else None
    sub = None if ap is None else {k: np.ascontiguousarray(v[e:e + 1]) for k, v in ap.items()}
    lines, cnt, n_obst = el.agent_lines(P, case["pos"][e:e + 1], case["vel"][e:e + 1], world=world, agent_params=sub,
                                        grid=grid, max_lines=max_lines)
    return lines[0], cnt[0], n_obst[0]


def _compare(case, grid):
    stats = dict(max_obst=0, collisions=0)
    for e in range(case["scn"].num_envs):
        lines, cnt, n_obst = _env_lines(case, e, grid)
        for i, (want, want_obst) in enumerate(case["progs"][e]):
            where = (case["name"], "grid" if grid else "tile", e, i)
            assert cnt[i] == want.shape[0], where + (int(cnt[i]), want.shape[0])
            assert n_obst[i] == want_obst, where + (int(n_obst[i]), want_obst)
            got = lines[i, :cnt[i]]
            assert got.view(np.uint32).tolist() == want.view(np.uint32).tolist(), where
            stats["max_obst"] = max(stats["max_obst"], int(want_obst))
    return stats


def test_lines_equal_the_oracle_bit_for_bit():
    el.counters(reset=True)
    max_obst = 0
    names = set()
    for case, grid in _cases():
        s = _compare(case, grid)
        max_obst = max(max_obst, s["max_obst"])
        names.add(case["name"])
    c = el.counters(reset=True)
    # the cases the worlds are there for all occurred
    assert max_obst > 6, max_obst                     # more obstacle lines than the step's fast path holds
    assert c[el.COVERED] > 0, c                       # an obstacle edge skipped as already covered
    assert c[el.COLLISION_LINES] > 0, c               # a line of the collision branch
    assert {"circle16", "circle32", "crowd256_blocks", "pillar_hall", "deadlock", "congested", "mixed_params",
            "lonely", "overlap", "grid_crowd1024"} <= names


def test_cases_cover_empty_programmes_and_per_agent_k0():
    cases = {c["name"]: c for c, _ in _cases()}
    lonely = cases["lonely"]["progs"][0][-1]
    assert lonely[0].shape[0] == 0 and lonely[1] == 0        # the lonely agent has no line at all
    mixed = cases["mixed_params"]
    k0 = mixed["agent_params"]["max_neighbors"] == 0
    assert k0.any()
    for e, i in zip(*np.nonzero(k0)):
        lines, n_obst = mixed["progs"][e][i]
        assert lines.shape[0] == n_obst                       # k = 0: obstacle lines only


@pytest.mark.parametrize("max_lines", [0, 1, 3])
def test_rows_past_max_lines_are_not_written(max_lines):
    case = next(c for c, _ in _cases() if c["name"] == "pillar_hall")
    full, cnt_full, obst_full = _env_lines(case, 0, False)
    lines, cnt, n_obst = _env_lines(case, 0, False, max_lines=max_lines)
    assert (cnt == cnt_full).all() and (n_obst == obst_full).all()   # counts are complete
    assert lines.shape[1] == max_lines
    for i in range(lines.shape[0]):
        m = min(max_lines, int(cnt[i]))
        assert lines[i, :m].view(np.uint32).tolist() == full[i, :m].view(np.uint32).tolist()
        assert np.isnan(lines[i, m:]).all()   # rows at and past max_lines (or count): untouched
    assert (cnt > max_lines).any()               # some programme really is cut
