"""CPU check of the roadmap device code (csrc/orca_roadmap.cuh compiled for the host by
tests/host_emul/emul_roadmap.cpp) against the oracle's literal queryVisibility recursion, Roadmap.cpp's
Dijkstra and its preferred-velocity loop (tests/host_emul/roadmap_oracle.cpp)."""
import numpy as np
import pytest

import _emul_roadmap as em
from _roadmap_common import RADII, query_points, random_roadmap, worlds
from _roadmap_oracle import oracle_world
from collision_avoidance_b200 import scenarios

def test_query_visibility_matches_oracle_bit_for_bit():
    rng = np.random.default_rng(0)
    em.counters(reset=True)
    n = 20000
    for name, polys in worlds().items():
        o = oracle_world(polys)
        w = em.World(polys)
        q1, q2 = query_points(polys, n, rng), query_points(polys, n, rng)
        # some degenerate queries: q1 == q2
        q2[:200] = q1[:200]
        r = rng.choice(RADII, n)
        got = w.visibility(q1, q2, r)
        want = np.array([o.queryVisibility(a, b, float(rr)) for a, b, rr in zip(q1, q2, r)])
        bad = np.flatnonzero(got != want)
        assert bad.size == 0, (name, bad[:5], q1[bad[:5]], q2[bad[:5]], r[bad[:5]])
        assert want.any() and not want.all(), name
    c = em.counters(reset=True)
    # every case of the recursion, and both outcomes of every clearance test, occurred
    assert (c[:10] > 0).all(), c[:10]


@pytest.mark.parametrize("R", [1, 7, 33, 200, 512])
def test_relaxation_equals_dijkstra(R):
    rng = np.random.default_rng(R)
    polys = worlds()["random_b"]
    o = oracle_world(polys)
    w = em.World(polys)
    xy = random_roadmap(polys, R, rng)
    G = min(R, 4)
    radius = float(rng.choice(RADII))
    adj, dist = o.roadmap_build(xy, G, radius)
    # the device edges are the device visibility of every ordered pair
    uu, vv = np.meshgrid(np.arange(R), np.arange(R), indexing="ij")
    got_adj = w.visibility(xy[uu.ravel()], xy[vv.ravel()], radius).reshape(R, R)
    assert (got_adj == adj).all()
    if R > 2:
        assert not (adj == adj.T).all() or R < 20  # visibility is not symmetric in general
    for g in range(G):
        d, _ = em.relax_dist(xy, adj, g)
        assert d.view(np.uint32).tolist() == dist[g].view(np.uint32).tolist(), g
    assert (dist == np.float32(9e9)).any() or R < 20


def test_pref_choice_matches_oracle():
    rng = np.random.default_rng(5)
    for name, polys in (("roadmap_blocks", worlds()["roadmap_blocks"]), ("random_a", worlds()["random_a"])):
        if name == "roadmap_blocks":
            _, xy, _ = scenarios.roadmap_blocks(1)
        else:
            xy = random_roadmap(polys, 40, rng)
        R, G = xy.shape[0], 4
        o = oracle_world(polys)
        _, dist = o.roadmap_build(xy, G, 0.5)
        n = 600
        pos = query_points(polys, n, rng)
        pos[:40] = xy[rng.integers(0, R, 40)]   # agents standing on roadmap vertices
        on_goal = rng.integers(0, G, 10)
        pos[40:50] = xy[on_goal]                 # ... on goal vertices
        goals = rng.integers(0, G, n).astype(np.int32)
        goals[40:45] = on_goal[:5]               # half of them on their own goal: pref (0, 0)
        radii = rng.choice(RADII, n)  # a per-agent radius table
        P = scenarios.ROADMAP_PARAMS
        for i in range(n):
            o.addAgent(tuple(pos[i]), P["neighborDist"], P["maxNeighbors"], P["timeHorizon"], P["timeHorizonObst"],
                       float(radii[i]), P["maxSpeed"], (0.0, 0.0))
        want_pref, want_vertex = o.roadmap_pref(xy, dist, goals)
        w = em.World(polys)
        pref, vertex = w.pref(xy, dist, pos, goals, radii)
        assert (vertex == want_vertex).all(), name
        assert pref.view(np.uint32).tolist() == want_pref.view(np.uint32).tolist(), name
        assert (want_vertex >= 0).any() and (want_vertex == -1).any() or name == "roadmap_blocks"
        # goal ids outside [0, G): pref (0, 0), vertex -1
        bad = np.array([-1, G, 1000], np.int32)
        pref, vertex = w.pref(xy, dist, pos[:3], bad, radii[:3])
        assert (vertex == -1).all() and (pref == 0).all()
