"""Line-of-sight queries and roadmap navigation on the device (orca_query_visibility, orca_set_roadmap,
orca_get_roadmap, orca_roadmap_pref_velocity) against the oracle's literal queryVisibility recursion
and Roadmap.cpp's buildRoadmap / setPreferredVelocities (tests/host_emul/roadmap_oracle.cpp)."""
import numpy as np
import pytest
import torch

from _roadmap_common import RADII, query_points, random_roadmap, worlds
from _roadmap_oracle import OracleSim, oracle_world
from collision_avoidance_b200 import _lib, rvo2_compat, scenarios
from collision_avoidance_b200.sim import BatchedRVOSimulator

pytestmark = pytest.mark.gpu

P = scenarios.ROADMAP_PARAMS


def make_sim(E, N, params=P):
    return BatchedRVOSimulator(E, N, device="cuda:0", **params)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def oracle_visibility(o, q1, q2, r):
    return np.array([o.queryVisibility(a, b, float(rr)) for a, b, rr in zip(q1, q2, r)])


@pytest.mark.parametrize("per_query_radius", [False, True])
def test_query_visibility_shared_and_per_env_worlds(per_query_radius):
    rng = np.random.default_rng(1)
    ws = worlds()
    names = ["deadlock", "blocks", "random_a"]
    Q = 3000
    for per_env in (False, True):
        E = len(names)
        polys = [ws[n] for n in names] if per_env else ws["deadlock"]
        sim = make_sim(E, 4)
        sim.set_obstacles(polys, per_env=per_env)
        env_polys = polys if per_env else [polys] * E
        q1 = np.stack([query_points(p, Q, rng) for p in env_polys])
        q2 = np.stack([query_points(p, Q, rng) for p in env_polys])
        q2[:, :50] = q1[:, :50]
        r = rng.choice(RADII, (E, Q)) if per_query_radius else np.full((E, Q), np.float32(0.5))
        radius = torch.from_numpy(r).cuda() if per_query_radius else 0.5
        got = sim.query_visibility(torch.from_numpy(q1).cuda(), torch.from_numpy(q2).cuda(), radius).cpu().numpy()
        assert got.dtype == np.bool_ and got.shape == (E, Q)
        for e in range(E):
            want = oracle_visibility(oracle_world(env_polys[e]), q1[e], q2[e], r[e])
            assert (got[e] == want).all(), (per_env, e, np.flatnonzero(got[e] != want)[:5])
            assert want.any() and not want.all()
        sim.close()


def test_no_obstacles_everything_visible():
    sim = make_sim(2, 4)
    rng = np.random.default_rng(2)
    q = torch.from_numpy(rng.uniform(-50, 50, (2, 500, 2)).astype(np.float32)).cuda()
    assert sim.query_visibility(q, q.flip(1), 3.0).all()
    sim.set_roadmap(np.float32([(0, 0), (10, 0), (0, 10)]), 1)
    adj, dist = sim.roadmap()
    assert adj.all()
    assert bits(dist).tolist() == bits([[0.0, 10.0, 10.0]]).tolist()


def check_tables(sim, env, polys, xy, G, radius):
    o = oracle_world(polys)
    adj_w, dist_w = o.roadmap_build(xy, G, radius)
    adj, dist = sim.roadmap(env)
    assert (adj == adj_w).all(), env
    assert bits(dist).tolist() == bits(dist_w).tolist(), env
    return adj_w, dist_w


def test_set_roadmap_matches_buildroadmap():
    rng = np.random.default_rng(3)
    scn, xy, _ = scenarios.roadmap_blocks(2)
    sim = make_sim(2, 8)
    sim.set_obstacles(scn.obstacles)
    sim.set_roadmap(xy, 4)
    for e in range(2):
        adj, dist = check_tables(sim, e, scn.obstacles, xy, 4, P["radius"])
    assert (dist < np.float32(9e9)).all()  # every roadmap vertex of this world reaches every goal
    # a random roadmap of the largest size, a one-way world and unreachable vertices
    polys = worlds()["random_b"]
    xy = random_roadmap(polys, 512, rng)
    sim.set_obstacles(polys)
    sim.set_roadmap(xy, 3, radius=0.1)
    adj, dist = check_tables(sim, 1, polys, xy, 3, 0.1)
    assert (dist == np.float32(9e9)).any() and not (adj == adj.T).all()
    sim.close()


def oracle_prefs(polys, xy, G, pos, goals, radii, radius_tables=0.5):
    o = OracleSim(*(P[k] for k in ("timeStep", "neighborDist", "maxNeighbors", "timeHorizon", "timeHorizonObst",
                                   "radius", "maxSpeed")))
    for p in polys:
        o.addObstacle(p)
    o.processObstacles()
    _, dist = o.roadmap_build(xy, G, radius_tables)
    for i in range(pos.shape[0]):
        o.addAgent(tuple(pos[i]), P["neighborDist"], P["maxNeighbors"], P["timeHorizon"], P["timeHorizonObst"],
                   float(radii[i]), P["maxSpeed"], (0.0, 0.0))
    ok = (goals >= 0) & (goals < G)
    pref, vertex = o.roadmap_pref(xy, dist, np.where(ok, goals, 0))
    pref[~ok] = 0.0
    vertex[~ok] = -1
    return pref, vertex


@pytest.mark.parametrize("agent_radii", [False, True])
def test_roadmap_pref_matches_setpreferredvelocities(agent_radii):
    rng = np.random.default_rng(4)
    polys = worlds()["random_a"]
    E, N, G = 2, 300, 4
    xy = random_roadmap(polys, 40, rng)
    pos = np.stack([query_points(polys, N, rng) for _ in range(E)])
    pos[:, :20] = xy[rng.integers(0, 40, (E, 20))]
    pos[:, 20:25] = xy[:G][rng.integers(0, G, (E, 5))]
    goals = rng.integers(0, G, (E, N)).astype(np.int32)
    goals[:, 25:28] = [-1, G, 99]
    sim = make_sim(E, N)
    sim.set_obstacles(polys)
    sim.set_roadmap(xy, G, radius=0.5)
    radii = np.full((E, N), np.float32(P["radius"]))
    if agent_radii:
        radii = rng.choice(RADII, (E, N))
        sim.set_agent_params(radius=radii)
    sim.pos.copy_(torch.from_numpy(pos))
    pref, vertex = sim.roadmap_pref_velocity(torch.from_numpy(goals).cuda(), return_vertex=True)
    assert pref.data_ptr() == sim.pref.data_ptr()
    pref, vertex = pref.cpu().numpy(), vertex.cpu().numpy()
    for e in range(E):
        want_pref, want_vertex = oracle_prefs(polys, xy, G, pos[e], goals[e], radii[e])
        assert (vertex[e] == want_vertex).all(), (e, np.flatnonzero(vertex[e] != want_vertex)[:5])
        assert bits(pref[e]).tolist() == bits(want_pref).tolist(), e
    assert (vertex[:, 25:28] == -1).all() and (pref[:, 25:28] == 0).all()
    # `out` and an explicit `pos`
    out = torch.zeros(E, N, 2, device="cuda:0")
    sim.pos.zero_()
    sim.roadmap_pref_velocity(torch.from_numpy(goals).cuda(), pos=torch.from_numpy(pos).cuda(), out=out)
    assert bits(out.cpu().numpy()).tolist() == bits(pref).tolist()
    sim.close()


def test_large_per_env_roadmap_blocks():
    E = 2048
    scn, xy, goal_vertex = scenarios.roadmap_blocks(E, jitter=5.0, seed=7)
    assert xy.shape == (E, 20, 2) and scn.per_env_obstacles
    sim = make_sim(E, scn.agents_per_env, scn.params)
    sim.set_obstacles(scn.obstacles, per_env=True)
    sim.set_roadmap(xy, 4)
    # mid-episode positions: the starts moved toward the middle
    rng = np.random.default_rng(8)
    pos = (scn.pos * np.float32(0.6) + rng.normal(0, 3, scn.pos.shape)).astype(np.float32)
    sim.pos.copy_(torch.from_numpy(pos))
    pref, vertex = sim.roadmap_pref_velocity(torch.from_numpy(goal_vertex).cuda(), return_vertex=True)
    pref, vertex = pref.cpu().numpy(), vertex.cpu().numpy()
    assert (vertex >= 0).mean() > 0.9
    for e in (0, 1, 777, E - 1):
        check_tables(sim, e, scn.obstacles[e], xy[e], 4, P["radius"])
        want_pref, want_vertex = oracle_prefs(scn.obstacles[e], xy[e], 4, pos[e], goal_vertex[e],
                                              np.full(scn.agents_per_env, np.float32(P["radius"])), P["radius"])
        assert (vertex[e] == want_vertex).all(), e
        assert bits(pref[e]).tolist() == bits(want_pref).tolist(), e
    sim.close()


def test_roadmap_rebuilt_after_set_obstacles_and_removed():
    scn, xy, goal_vertex = scenarios.roadmap_blocks(1)
    sim = make_sim(1, scn.agents_per_env)
    sim.set_roadmap(xy, 4)
    adj0, _ = sim.roadmap()
    assert adj0.all()  # no obstacles yet
    sim.set_obstacles(scn.obstacles)
    check_tables(sim, 0, scn.obstacles, xy, 4, P["radius"])
    # per-env obstacles after a shared roadmap: tables per env
    sim2 = make_sim(2, 4)
    sim2.set_roadmap(xy, 4)
    sim2.set_obstacles([scn.obstacles, []], per_env=True)
    check_tables(sim2, 0, scn.obstacles, xy, 4, P["radius"])
    assert sim2.roadmap(1)[0].all()
    sim2.close()
    # removal
    sim.set_roadmap(np.zeros((0, 2), np.float32), 0)
    with pytest.raises(RuntimeError):
        sim.roadmap_pref_velocity(torch.from_numpy(goal_vertex).cuda())
    with pytest.raises(RuntimeError):
        sim.roadmap()
    sim.close()


def test_errors():
    sim = make_sim(2, 4)
    xy = np.zeros((513, 2), np.float32)
    with pytest.raises(NotImplementedError):
        sim.set_roadmap(xy, 1)
    with pytest.raises(NotImplementedError):
        sim.set_roadmap(xy[:5], 6)
    with pytest.raises(NotImplementedError):
        sim.set_roadmap(xy[:5], 0)
    bad = xy[:5].copy()
    bad[2, 1] = np.nan
    with pytest.raises(ValueError):
        sim.set_roadmap(bad, 1)
    with pytest.raises(ValueError):
        sim.set_roadmap(xy[:5], 1, radius=-1.0)
    with pytest.raises(ValueError):
        sim.set_roadmap(np.zeros((3, 5, 2), np.float32), 1)  # per-env rows must match num_envs
    goals = torch.zeros(2, 4, dtype=torch.int32, device="cuda:0")
    with pytest.raises(RuntimeError):  # no roadmap yet
        sim.roadmap_pref_velocity(goals)
    sim.set_roadmap(np.float32([(0, 0), (3, 4)]), 2)
    with pytest.raises(ValueError):
        sim.roadmap_pref_velocity(goals.to(torch.int64))
    q = torch.zeros(2, 3, 2, device="cuda:0")
    with pytest.raises(ValueError):
        sim.query_visibility(q, q, -1.0)
    with pytest.raises(ValueError):
        sim.query_visibility(q, q[:, :2], 0.0)
    sim.close()


def test_compat_query_visibility_matches_oracle():
    rng = np.random.default_rng(9)
    polys = worlds()["deadlock"]
    args = (1 / 60., 5.0, 10, 1.5, 1.5, 0.5, 1.0)
    shim = rvo2_compat.PyRVOSimulator(*args)
    ref = OracleSim(*args)
    for p in polys:
        shim.addObstacle(p)
        ref.addObstacle(p)
    q1, q2 = query_points(polys, 40, rng), query_points(polys, 40, rng)
    r = rng.choice(RADII, 40)

    def same():
        for a, b, rr in zip(q1, q2, r):
            assert shim.queryVisibility(tuple(a), tuple(b), float(rr)) == ref.queryVisibility(a, b, float(rr))

    same()  # before processObstacles: everything visible
    assert shim.queryVisibility((0, 0), (1000, 0))
    shim.processObstacles()
    ref.processObstacles()
    same()  # no agents yet: a throw-away handle
    shim.addAgent((1.0, 1.0))
    ref.addAgent((1.0, 1.0))
    same()
    assert any(not shim.queryVisibility(tuple(a), tuple(b), float(rr)) for a, b, rr in zip(q1, q2, r))


# a U-shaped wall open at the bottom, an agent inside it and its goal above the closed top
U_WALL = [[(-5.0, 4.0), (5.0, 4.0), (5.0, 5.0), (-5.0, 5.0)],
          [(-5.0, -4.0), (-4.0, -4.0), (-4.0, 4.0), (-5.0, 4.0)],
          [(4.0, -4.0), (5.0, -4.0), (5.0, 4.0), (4.0, 4.0)]]
U_ROADMAP = np.float32([(0, 12), (0, -6), (-7, -6), (-7, 7), (7, -6), (7, 7)])
U_PARAMS = dict(timeStep=0.1, neighborDist=5.0, maxNeighbors=5, timeHorizon=2.0, timeHorizonObst=2.0, radius=0.5,
                maxSpeed=1.0)


def run_u_wall(roadmap, steps=400):
    sim = make_sim(1, 1, U_PARAMS)
    sim.set_obstacles(U_WALL)
    sim.set_roadmap(U_ROADMAP, 1)
    goal = torch.tensor([[[0.0, 12.0]]], device="cuda:0")
    goal_vertex = torch.zeros(1, 1, dtype=torch.int32, device="cuda:0")
    for _ in range(steps):
        if roadmap:
            sim.roadmap_pref_velocity(goal_vertex)
            sim.env_step(policy=_lib.POLICY_EXTERNAL, collect_stats=False)
        else:
            sim.env_step(policy=_lib.POLICY_GOAL, goal=goal, collect_stats=False)
    out = sim.pos[0, 0].cpu().numpy()
    sim.close()
    return out


def test_closed_loop_u_wall():
    a = run_u_wall(True)
    assert np.linalg.norm(a - (0.0, 12.0)) < 0.5, a
    assert bits(run_u_wall(True)).tolist() == bits(a).tolist()  # deterministic
    b = run_u_wall(False)
    assert np.linalg.norm(b - (0.0, 12.0)) > 5.0, b  # straight to the goal: stuck inside the U
