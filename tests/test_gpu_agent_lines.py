"""orca_agent_lines on the B200: the ORCA half-planes of every agent (RVO2's getAgentNumORCALines /
getAgentORCALine) against the oracle bit for bit on oracle-synchronised states, against the step it
mirrors (the host LP run on the exported lines gives the step's new velocity bit for bit, on every step
kernel variant), its capacity rules, the absence of side effects, the rvo2 shim and the error cases."""
import numpy as np
import pytest

import _lp3_worlds as lw
from _agent_params import mixed_params, oracle_sims_per_agent
from _emul_lp import emul_solve
from _lines_worlds import has_tie
from oracle.helpers import goal_pref, oracle_sims

pytestmark = pytest.mark.gpu

LP3 = 0


def _sim(scn, agent_params=None):
    import torch
    from collision_avoidance_b200.sim import BatchedRVOSimulator
    sim = BatchedRVOSimulator(scn.num_envs, scn.agents_per_env, device="cuda:0", **scn.params)
    if scn.obstacles:
        sim.set_obstacles(scn.obstacles, per_env=scn.per_env_obstacles)
    if agent_params is not None:
        sim.set_agent_params(**agent_params)
    sim.pos.copy_(torch.from_numpy(scn.pos))
    sim.vel.copy_(torch.from_numpy(scn.vel))
    return sim


def _tie_agents(pos, nd):
    """bool [N]: agents with two others at bit-equal squared distance within their range (their order,
    and so their lines, may differ from RVO2's kd-tree order)."""
    p = pos.astype(np.float32)
    nd = np.broadcast_to(np.asarray(nd, np.float32), (len(p),))
    out = np.zeros(len(p), bool)
    for i in range(len(p)):
        d = (p - p[i]).astype(np.float32)
        dsq = np.delete(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1], i)
        dsq = dsq[dsq < nd[i] * nd[i]]
        out[i] = len(np.unique(dsq)) < len(dsq)
    return out


def _check_against_oracle(scn, steps, agent_params=None, agents=None):
    """`steps` oracle-synchronised states: the device lines of the state equal the oracle's programme of
    its next doStep for every agent (of `agents`, default all) without a tie.  Returns agents checked."""
    import torch
    sim = _sim(scn, agent_params)
    sims = oracle_sims(scn) if agent_params is None else oracle_sims_per_agent(scn, agent_params)
    nd = scn.params["neighborDist"] if agent_params is None else agent_params["neighbor_dist"]
    nd = np.broadcast_to(np.asarray(nd, np.float32), scn.pos.shape[:2])
    E, N = scn.pos.shape[:2]
    agents = range(N) if agents is None else agents
    checked = 0
    for t in range(steps):
        pos = np.stack([s.positions() for s in sims]).astype(np.float32)
        vel = np.stack([s.velocities() for s in sims]).astype(np.float32)
        sim.pos.copy_(torch.from_numpy(pos))
        sim.vel.copy_(torch.from_numpy(vel))
        lines, cnt, n_obst = sim.orca_lines(max_lines=scn.params["maxNeighbors"] + 64)
        lines, cnt, n_obst = lines.cpu().numpy(), cnt.cpu().numpy(), n_obst.cpu().numpy()
        for e, s in enumerate(sims):
            s.set_pref_velocities(goal_pref(pos[e], scn.goal[e]).astype(np.float32))
            s.doStep()
            ties = _tie_agents(pos[e], nd[e])
            for i in agents:
                if ties[i]:
                    continue
                want, want_obst = s.orca_lines(i)
                where = (scn.name, t, e, i)
                assert cnt[e, i] == want.shape[0] and n_obst[e, i] == want_obst, where
                assert lines[e, i, :cnt[e, i]].view(np.uint32).tolist() == want.view(np.uint32).tolist(), where
                checked += 1
    return checked


@pytest.mark.parametrize("per_env", [False, True])
@pytest.mark.parametrize("N,k", [(16, 10), (24, 5), (32, 16), (100, 10), (256, 5), (256, 16)])
def test_tile_lines_equal_the_oracle(N, k, per_env):
    from collision_avoidance_b200 import scenarios
    scn = scenarios.crowd(max(2, 256 // N), N, seed=N + k, blocks=4)
    scn.params = dict(scn.params, maxNeighbors=k)
    if not per_env:   # env 0's blocks for every env
        scn.obstacles, scn.per_env_obstacles = scn.obstacles[0], False
    assert _check_against_oracle(scn, 50) > 0.9 * 50 * scn.num_envs * N


@pytest.mark.parametrize("N,grid", [(40, False), (300, True)])
def test_lines_with_per_agent_params_equal_the_oracle(N, grid):
    from collision_avoidance_b200 import scenarios
    scn = scenarios.crowd(2 if not grid else 1, N, seed=N, blocks=2)
    ap = mixed_params(scn.num_envs, N, scn.params["maxNeighbors"], seed=N)
    assert _check_against_oracle(scn, 50, agent_params=ap) > 0.9 * 50 * scn.num_envs * N


def test_grid_lines_equal_the_oracle():
    from collision_avoidance_b200 import scenarios
    scn = scenarios.crowd(1, 1000, seed=21, blocks=4)
    assert _check_against_oracle(scn, 50) > 0.9 * 50 * 1000


def test_million_agent_world_sampled_lines_equal_the_oracle():
    """The 1,000,000-agent world of test_million_agent_world_one_oracle_step, settled by 40 device steps:
    10,000 sampled agents' lines equal the oracle's programme of one doStep from that state."""
    import torch
    from collision_avoidance_b200 import _lib, scenarios
    from oracle import rvo2_oracle
    N = 1_000_000
    scn = scenarios.crowd(1, N, seed=15)
    P = scn.params
    sim = _sim(scn)
    goal = torch.from_numpy(scn.goal).cuda()
    for _ in range(40):
        sim.env_step(policy=_lib.POLICY_GOAL, goal=goal)
    lines, cnt, n_obst = sim.orca_lines(max_lines=P["maxNeighbors"] + 64)
    pos, vel = sim.pos.cpu().numpy()[0], sim.vel.cpu().numpy()[0]
    o = rvo2_oracle.PyRVOSimulator(P["timeStep"], P["neighborDist"], P["maxNeighbors"], P["timeHorizon"],
                                   P["timeHorizonObst"], P["radius"], P["maxSpeed"])
    o.add_agents(pos, vel)
    for poly in scn.obstacles:
        o.addObstacle([tuple(map(float, v)) for v in poly])
    o.processObstacles()
    o.set_pref_velocities(goal_pref(pos, scn.goal[0]).astype(np.float32))
    o.doStep()
    from scipy.spatial import cKDTree
    sample = np.random.default_rng(0).choice(N, 10_000, replace=False)
    rows = lines[0, torch.from_numpy(sample).cuda()].cpu().numpy()
    cnt, n_obst = cnt.cpu().numpy()[0], n_obst.cpu().numpy()[0]
    tree = cKDTree(pos.astype(np.float64))
    nd = np.float32(P["neighborDist"])
    checked = 0
    for r, i in enumerate(sample):
        near = [j for j in tree.query_ball_point(pos[i].astype(np.float64), float(nd) * 1.001) if j != i]
        d = (pos[near] - pos[i]).astype(np.float32)
        dsq = d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]
        dsq = dsq[dsq < nd * nd]
        if len(np.unique(dsq)) < len(dsq):
            continue   # neighbors at bit-equal distance: RVO2's kd-tree order may differ
        want, want_obst = o.orca_lines(int(i))
        assert cnt[i] == want.shape[0] and n_obst[i] == want_obst, i
        assert rows[r, :cnt[i]].view(np.uint32).tolist() == want.view(np.uint32).tolist(), i
        checked += 1
    assert checked >= 9_900, checked


# ----------------------------------------------------------------------------------- lines vs step
def _variant_worlds():
    from collision_avoidance_b200 import scenarios
    batch = lw.assemble(32, 256, 10, seed=2)
    slim = lw.scenario(batch, 10)                                   # 4-vertex wall, N <= 32, K = 10: slim
    full = scenarios.crowd(8, 64, seed=8, blocks=4)                 # full tile kernel, in-block grid
    full5 = scenarios.crowd(8, 24, seed=9, blocks=4)
    full5.params = dict(full5.params, maxNeighbors=5)
    grid = scenarios.crowd(1, 700, seed=10, blocks=4)               # uniform-grid kernel
    het = scenarios.crowd(4, 48, seed=11, blocks=2)                 # HETERO tile kernel
    het_grid = scenarios.crowd(1, 400, seed=12, blocks=2)           # HETERO grid kernel
    return [("slim", slim, None), ("full", full, None), ("full_k5", full5, None), ("grid", grid, None),
            ("hetero", het, mixed_params(4, 48, 10, seed=11)), ("hetero_grid", het_grid, mixed_params(1, 400, 10, seed=12))]


@pytest.mark.parametrize("variant", ["slim", "full", "full_k5", "grid", "hetero", "hetero_grid"])
def test_host_lp_on_the_lines_gives_the_step_velocity(variant):
    """The split check: emul_solve(lines, count, n_obst, maxSpeed_i, pref_i, LP3) on the exported lines
    equals the new velocity of orca_env_step(POLICY_EXTERNAL) from the same state, for every agent."""
    import torch
    from collision_avoidance_b200 import _lib
    name, scn, ap = next(w for w in _variant_worlds() if w[0] == variant)
    sim = _sim(scn, ap)
    E, N = scn.pos.shape[:2]
    vmax = np.full((E, N), scn.params["maxSpeed"], np.float32) if ap is None else ap["max_speed"]
    goal = torch.from_numpy(scn.goal).cuda()
    for t in range(5):
        pref = torch.from_numpy(goal_pref(sim.pos.cpu().numpy(), scn.goal).astype(np.float32)).cuda()
        sim.pref.copy_(pref)
        lines, cnt, n_obst = sim.orca_lines(max_lines=scn.params["maxNeighbors"] + 64)
        sim.env_step(policy=_lib.POLICY_EXTERNAL, collect_stats=True)
        assert sim.read_stats(allow_overflow=False) is not None
        nv = sim.vel.cpu().numpy()
        lines, cnt, n_obst, pref = lines.cpu().numpy(), cnt.cpu().numpy(), n_obst.cpu().numpy(), pref.cpu().numpy()
        for e in range(E):
            for i in range(N):
                n = int(cnt[e, i])
                _, v = emul_solve(lines[e, i, :n], n, int(n_obst[e, i]), vmax[e, i], pref[e, i], LP3)
                assert v.view(np.uint32).tolist() == nv[e, i].view(np.uint32).tolist(), (name, t, e, i)
        for _ in range(3):   # move on to a later state
            sim.env_step(policy=_lib.POLICY_GOAL, goal=goal, collect_stats=False)


# ----------------------------------------------------------------------------------- capacity
def test_capacity_sentinels_and_counts_only():
    import torch
    from collision_avoidance_b200 import _lib
    from _common import pillar_hall
    scn = pillar_hall(num_agents=12, seed=1)
    sim = _sim(scn)
    full, cnt, n_obst = sim.orca_lines(max_lines=64 + scn.params["maxNeighbors"])
    assert (n_obst > 6).any()
    L = sim._L
    E, N = scn.pos.shape[:2]
    for m in (1, 3, 7):
        buf = torch.full((E, N, m, 4), 12345.0, dtype=torch.float32, device="cuda:0")
        c = torch.full((E, N), -9, dtype=torch.int32, device="cuda:0")
        _lib.check(L.orca_agent_lines(sim._h, sim._p(sim.pos), sim._p(sim.vel), m, sim._p(buf), sim._p(c), None,
                                      sim._stream()))
        buf, c = buf.cpu().numpy(), c.cpu().numpy()
        assert (c == cnt.cpu().numpy()).all()
        f = full.cpu().numpy()
        for i in range(N):
            k = min(m, int(c[0, i]))
            assert buf[0, i, :k].view(np.uint32).tolist() == f[0, i, :k].view(np.uint32).tolist()
            assert (buf[0, i, k:] == 12345.0).all()          # rows at and past max_lines (or count) untouched
    c = torch.full((E, N), -9, dtype=torch.int32, device="cuda:0")
    o = torch.full((E, N), -9, dtype=torch.int32, device="cuda:0")
    _lib.check(L.orca_agent_lines(sim._h, sim._p(sim.pos), sim._p(sim.vel), 0, None, sim._p(c), sim._p(o), sim._stream()))
    assert (c == cnt).all() and (o == n_obst).all()
    lines0, c0, _ = sim.orca_lines(max_lines=0)
    assert lines0.shape == (E, N, 0, 4) and (c0 == cnt).all()


# ----------------------------------------------------------------------------------- side effects
def _run(scn, interleave, steps=20):
    import torch
    from collision_avoidance_b200 import _lib
    sim = _sim(scn)
    goal = torch.from_numpy(scn.goal).cuda()
    env_step = torch.zeros(scn.num_envs, dtype=torch.int32, device="cuda:0")
    nbrs = []
    for _ in range(steps):
        if interleave:
            before = env_step.clone()
            sim.orca_lines()
            assert torch.equal(before, env_step)
        sim.env_step(policy=_lib.POLICY_GOAL, goal=goal, env_step=env_step, want_neighbors=True)
        nbrs.append([t.cpu().numpy().copy() for t in (sim.nbr_idx, sim.nbr_cnt, sim.obst_nbr_idx, sim.obst_nbr_cnt)])
    torch.cuda.synchronize()
    return sim.pos.cpu().numpy(), sim.vel.cpu().numpy(), sim.stats.cpu().numpy(), nbrs, env_step.cpu().numpy()


@pytest.mark.parametrize("shape", [(16, 64), (2, 200), (1, 800)])
def test_interleaved_lines_change_nothing(shape):
    from collision_avoidance_b200 import scenarios
    scn = scenarios.crowd(shape[0], shape[1], seed=31, blocks=4)
    a, b = _run(scn, False), _run(scn, True)
    for x, y in zip(a[:3], b[:3]):
        assert x.view(np.uint32).tolist() == y.view(np.uint32).tolist()
    for s1, s2 in zip(a[3], b[3]):
        for x, y in zip(s1, s2):
            assert (x == y).all()
    assert (a[4] == b[4]).all() and (a[4] == 20).all()


def test_interleaved_lines_change_nothing_through_step_host_on_a_grid_handle():
    import torch
    from collision_avoidance_b200 import _lib, scenarios
    scn = scenarios.crowd(1, 600, seed=33, blocks=4)
    results = []
    for interleave in (False, True):
        sim = _sim(scn)
        pos = torch.from_numpy(scn.pos.copy())
        vel = torch.from_numpy(scn.vel.copy())
        goal = torch.from_numpy(scn.goal.copy())
        for t in range(15):
            if interleave:
                p_dev, v_dev = pos.cuda(), vel.cuda()
                sim.orca_lines(pos=p_dev, vel=v_dev)
                # step_host runs on the handle's own streams, which do not wait for torch's stream
                torch.cuda.synchronize()
            sim.step_host(pos, vel, goal, policy=_lib.POLICY_GOAL, upload_state=(t == 0))
        results.append((pos.numpy().copy(), vel.numpy().copy()))
    for x, y in zip(*results):
        assert x.view(np.uint32).tolist() == y.view(np.uint32).tolist()


# ----------------------------------------------------------------------------------- the rvo2 shim
def test_shim_lines_match_the_oracle_through_a_run():
    from collision_avoidance_b200.rvo2_compat import PyRVOSimulator
    from oracle.rvo2_oracle import PyRVOSimulator as Oracle
    P = lw.params(10)
    args = (P["timeStep"], P["neighborDist"], P["maxNeighbors"], P["timeHorizon"], P["timeHorizonObst"], P["radius"], P["maxSpeed"])
    shim, ora = PyRVOSimulator(*args), Oracle(*args)
    rng = np.random.default_rng(5)
    pos = rng.uniform(0, 12, (30, 2)).astype(np.float32)
    while has_tie(pos, P["neighborDist"]):
        pos = rng.uniform(0, 12, (30, 2)).astype(np.float32)
    for p in pos:
        shim.addAgent(tuple(map(float, p)))
        ora.addAgent(tuple(map(float, p)), *args[1:], (0.0, 0.0))
    for s in (shim, ora):
        s.addObstacle([(4.0, 4.0), (4.0, 8.0), (8.0, 8.0), (8.0, 4.0)][::-1])
        s.processObstacles()
    assert shim.getAgentNumORCALines(0) == 0                # before the first step
    with pytest.raises(IndexError):
        shim.getAgentORCALine(0, 0)
    goals = rng.uniform(0, 12, (30, 2))

    def compare(n):
        for i in range(n):
            want, _ = ora.orca_lines(i)
            assert shim.getAgentNumORCALines(i) == want.shape[0], i
            for j in range(want.shape[0]):
                got = shim.getAgentORCALine(i, j)
                assert isinstance(got, tuple) and len(got) == 4    # (point.x, point.y, direction.x, direction.y)
                assert np.asarray(got, np.float32).view(np.uint32).tolist() == want[j].view(np.uint32).tolist()
            with pytest.raises(IndexError):
                shim.getAgentORCALine(i, want.shape[0])

    compared = 0
    for t in range(100):
        n = shim.getNumAgents()
        sp = np.asarray([shim.getAgentPosition(i) for i in range(n)], np.float32)
        if has_tie(sp, P["neighborDist"]):
            break
        pref = goal_pref(sp, goals).astype(np.float32)
        for i in range(n):
            shim.setAgentPrefVelocity(i, tuple(map(float, pref[i])))
        ora.set_pref_velocities(pref)
        shim.doStep()
        ora.doStep()
        if t % 10 == 0 or t in (1, 99):
            compare(n)
            compared += 1
    assert compared >= 6
    # calls that change what the device computes, between the last step and the query: the answers
    # stay those of the step that ran
    shim.setAgentRadius(3, 0.8)
    compare(30)
    shim.addObstacle([(1.0, 1.0), (1.0, 2.0), (2.0, 2.0)])
    shim.processObstacles()
    compare(30)
    new = shim.addAgent((11.5, 0.5))
    assert shim.getAgentNumORCALines(new) == 0             # added after the step: no lines
    compare(30)
    with pytest.raises(IndexError):
        shim.getAgentNumORCALines(new + 1)


# ----------------------------------------------------------------------------------- errors
def test_error_cases():
    import torch
    from collision_avoidance_b200 import _lib, scenarios
    scn = scenarios.circle(2, 16, seed=1)
    sim = _sim(scn)
    L, h, st = sim._L, sim._h, sim._stream()
    c = torch.zeros(2, 16, dtype=torch.int32, device="cuda:0")
    buf = torch.zeros(2, 16, 4, 4, dtype=torch.float32, device="cuda:0")
    P = sim._p
    for call in (lambda: L.orca_agent_lines(None, P(sim.pos), P(sim.vel), 4, P(buf), P(c), None, st),
                 lambda: L.orca_agent_lines(h, None, P(sim.vel), 4, P(buf), P(c), None, st),
                 lambda: L.orca_agent_lines(h, P(sim.pos), None, 4, P(buf), P(c), None, st),
                 lambda: L.orca_agent_lines(h, P(sim.pos), P(sim.vel), 4, P(buf), None, None, st),
                 lambda: L.orca_agent_lines(h, P(sim.pos), P(sim.vel), -1, P(buf), P(c), None, st),
                 lambda: L.orca_agent_lines(h, P(sim.pos), P(sim.vel), 4, None, P(c), None, st)):
        with pytest.raises(ValueError):
            _lib.check(call())
    with pytest.raises(ValueError):
        sim.orca_lines(pos=sim.pos.cpu())
    with pytest.raises(ValueError):
        sim.orca_lines(vel=sim.vel[:, :8].contiguous())
    with pytest.raises(ValueError):
        sim.orca_lines(pos=sim.pos.double())
    with pytest.raises(ValueError):
        sim.orca_lines(max_lines=-2)
