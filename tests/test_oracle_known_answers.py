"""Pins the CPU oracle: analytic known answers (SURVEY T0), the reference's own golden vectors
for the laser path (generated from the reference's collision_avoidance/envs/utils.py by
tests/golden/make_golden.py) and the reference's action-table fixtures."""
import json
import os

import numpy as np
import pytest

from oracle import shell_oracle
from oracle.rvo2_oracle import PyRVOSimulator, solve_lp

GOLD = os.path.join(os.path.dirname(__file__), "golden")
DT = 1 / 60.


def _sim(nd=5.0, k=10):
    return PyRVOSimulator(DT, nd, k, 1.5, 1.5, 0.5, 1.0)


def test_lone_agent_takes_clamped_pref_velocity():
    s = _sim()
    a = s.addAgent((0, 0))
    s.setAgentPrefVelocity(a, (3, 4))  # |pref| = 5 > vmax = 1 -> unit vector
    s.doStep()
    v = s.getAgentVelocity(a)
    assert v == pytest.approx((0.6, 0.8), abs=1e-7)
    assert s.getAgentPosition(a) == pytest.approx((0.6 * DT, 0.8 * DT), abs=1e-7)
    s.setAgentPrefVelocity(a, (0.25, -0.5))  # inside the disc -> taken as is
    s.doStep()
    assert s.getAgentVelocity(a) == pytest.approx((0.25, -0.5), abs=1e-7)


def test_head_on_pair_analytic():
    """A=(0,0) v=(1,0), B=(2.5,0) v=(-1,0), r=.5, tau=1.5: right-leg projection gives
    v_A = (0.84, -0.36661) and the mirror image for B (SURVEY section 4, T0-ii)."""
    s = _sim()
    a = s.addAgent((0, 0), 5, 10, 1.5, 1.5, 0.5, 1.0, (1, 0))
    b = s.addAgent((2.5, 0), 5, 10, 1.5, 1.5, 0.5, 1.0, (-1, 0))
    s.setAgentPrefVelocity(a, (1, 0))
    s.setAgentPrefVelocity(b, (-1, 0))
    s.doStep()
    va, vb = s.getAgentVelocity(a), s.getAgentVelocity(b)
    leg = np.sqrt(2.5 ** 2 - 1.0)
    d = np.array([2.5 * leg, -2.5]) / 6.25          # right leg direction (before negation)
    rv = np.array([2.0, 0.0])
    u = rv.dot(-d) * (-d) - rv
    expect = np.array([1.0, 0.0]) + 0.5 * u
    assert va == pytest.approx(tuple(expect), abs=1e-6)
    assert va == pytest.approx((0.84, -0.36661), abs=1e-5)
    assert vb == pytest.approx((-0.84, 0.36661), abs=1e-5)
    lines, n_obst = s.orca_lines(a)
    assert n_obst == 0 and lines.shape == (1, 4)
    assert lines[0] == pytest.approx([0.84, -0.36661, -0.91652, 0.4], abs=1e-5)


def test_wall_limits_approach_speed():
    """Agent heading into a wall at distance d: ORCA lets it close (d - r) within tau_obst, so
    the normal speed is (d - r) / tau_obst  (cut-off line of the obstacle VO)."""
    s = _sim()
    a = s.addAgent((1.0, 5.0), 5, 10, 1.5, 1.5, 0.5, 1.0, (-1, 0))
    s.addObstacle([(0, 0), (0, 10), (10, 10), (10, 0)])  # clockwise: inside is visible (Q6)
    s.processObstacles()
    s.setAgentPrefVelocity(a, (-1, 0))
    s.doStep()
    assert s.getAgentVelocity(a) == pytest.approx((-(1.0 - 0.5) / 1.5, 0.0), abs=1e-6)
    assert [v for v, _ in s.obstacle_neighbors(a)] == [0]
    # counter-clockwise wall: the inside is the invisible side -> no obstacle neighbors
    s2 = _sim()
    b = s2.addAgent((1.0, 5.0), 5, 10, 1.5, 1.5, 0.5, 1.0, (-1, 0))
    s2.addObstacle([(0, 0), (10, 0), (10, 10), (0, 10)])
    s2.processObstacles()
    s2.setAgentPrefVelocity(b, (-1, 0))
    s2.doStep()
    assert s2.obstacle_neighbors(b) == []
    assert s2.getAgentVelocity(b) == pytest.approx((-1.0, 0.0), abs=1e-7)


def test_obstacle_ids_and_ring_links():
    """addObstacle returns the id of the first vertex; ids are sequential across polygons;
    getNextObstacleVertexNo walks the ring (env:145-148)."""
    s = _sim()
    assert s.addObstacle([(-15, 0), (-15, 10), (10, 10), (10, 0)]) == 0
    assert s.addObstacle([(2, 0), (2.5, 0), (2.5, 4.4), (2, 4.4)]) == 4
    assert s.addObstacle([(2, 5.6), (2.5, 5.6), (2.5, 10), (2, 10)]) == 8
    ring = [4]
    for _ in range(4):
        ring.append(s.getNextObstacleVertexNo(ring[-1]))
    assert ring == [4, 5, 6, 7, 4]
    with pytest.raises(RuntimeError):
        s.addObstacle([(0, 0)])
    with pytest.raises(ValueError):
        s.addAgent((0, 0), 5.0)  # partial arguments


def test_bsp_splits_straddling_edges():
    """processObstacles may split edges and append vertices (SURVEY A.3 / H5)."""
    s = _sim()
    s.addObstacle([(-15, 0), (-15, 10), (10, 10), (10, 0)])
    s.addObstacle([(2, 0), (2.5, 0), (2.5, 4.4), (2, 4.4)])
    s.addObstacle([(2, 5.6), (2.5, 5.6), (2.5, 10), (2, 10)])
    s.processObstacles()
    n = s.getNumObstacleVertices()
    assert n >= 12
    pts, dirs, nxt, prv, cvx = s.obstacle_vertex_table()
    for v in range(n):  # ring consistency survives the splits
        assert prv[nxt[v]] == v and nxt[prv[v]] == v
    for v in range(12, n):  # appended vertices lie on their parent edge and are convex
        assert cvx[v] == 1
        assert np.allclose(dirs[v], dirs[prv[v]])


def test_lp_infeasible_falls_back_to_min_penetration():
    # two opposing half-planes 0.4 apart in the wrong order: infeasible -> LP3 picks the middle
    lines = np.array([[0.0, 0.2, 1.0, 0.0],    # needs v.y >= 0.2   (left of direction +x)
                      [0.0, -0.2, -1.0, 0.0]],  # needs v.y <= -0.2
                     np.float32)
    fail, res = solve_lp(lines, 0, 1.0, (0.3, 0.0))
    assert fail == 1
    assert res[1] == pytest.approx(0.0, abs=1e-6)


def test_laser_restatement_matches_reference_golden():
    g = np.load(os.path.join(GOLD, "laser_golden.npz"))
    rays = shell_oracle.laser_rays(16, 1.5)
    for c in range(g["seg"].shape[0]):
        n = int(g["nlines"][c])
        lines = [(((g["seg"][c, k, 0], g["seg"][c, k, 1]), (g["seg"][c, k, 2], g["seg"][c, k, 3])),
                  (g["vel"][c, k, 0], g["vel"][c, k, 1])) for k in range(n)]
        if n:
            res = shell_oracle.comp_laser(rays, lines, tuple(g["orient"][c]))
        else:
            res = [((0, 0), (0, 0))] * 16
        got = np.array([[h[0], h[1], v[0], v[1]] for h, v in res])
        np.testing.assert_allclose(got, g["out"][c], rtol=0, atol=1e-12)


def test_line_intersection_matches_reference_golden():
    g = np.load(os.path.join(GOLD, "laser_golden.npz"))
    hits = 0
    for k in range(g["li_in"].shape[0]):
        a = g["li_in"][k]
        d, p = shell_oracle.line_intersection(((a[0], a[1]), (a[2], a[3])), ((a[4], a[5]), (a[6], a[7])))
        if np.isinf(g["li_d"][k]):
            assert np.isinf(d)
        else:
            hits += 1
            assert d == pytest.approx(g["li_d"][k], abs=1e-12)
            assert p == pytest.approx(tuple(g["li_p"][k]), abs=1e-12)
    assert hits > 20


def test_laser_tables_match_reference_constants():
    rays = shell_oracle.laser_rays(16, 1.5)
    assert rays[0][1] == pytest.approx((1.5, 0.0))
    assert rays[4][1] == pytest.approx((0.0, -1.5), abs=1e-12)   # y flipped (env:328)
    oct_ = shell_oracle.circle_approx(8, 0.5)
    assert len(oct_) == 8 and oct_[0][0] == pytest.approx((0.5, 0.0)) and oct_[7][1] == pytest.approx((0.5, 0.0))


def test_alan_window_resets_every_121_steps():
    """All per-action timers advance together; 120 * (1/60.) < 2 in float64, so the reset
    fires on every 121st step (SURVEY Q7).  Checked on the float64 shell restatement."""
    from collision_avoidance_b200 import scenarios
    scn = scenarios.circle(1, 4, seed=0)
    sh = shell_oracle.AlanShellOracle(scn, 0)
    resets = []
    for t in range(1, 260):
        sh.online_step([0.5] * 4)
        if all(x == 0 for x in sh.action_times[0]):
            resets.append(t)
    assert resets == [121, 242]
    from collision_avoidance_b200.alan import alan_window_steps
    assert alan_window_steps(1 / 60., 2) == 121


def test_act_tables_are_unit_vectors_starting_with_forward():
    with open(os.path.join(GOLD, "act_tables.json")) as f:
        tables = json.load(f)
    assert {k: len(v) for k, v in tables.items()} == {"blocks": 8, "circle": 3, "congested": 9, "crowd": 9,
                                                      "deadlock": 2, "incoming": 5}
    for name, t in tables.items():
        assert t[0] == [1.0, 0.0]
        assert np.allclose(np.linalg.norm(np.array(t), axis=1), 1.0, atol=1e-9)
