"""Worlds and oracle programmes for the ORCA-line tests (orca_agent_lines, csrc/orca_lines.cuh).

A case is a scenario, a pre-step state (pos, vel) reached by running the oracle, optional per-agent
parameters, and for every agent the oracle's programme of one doStep from that state
(``Simulator::orca_lines``).  States where some agent has two others at bit-equal squared distance
within its neighbor range are rejected, as in _lp3_worlds: there the library's (distSq, id) order and
RVO2's kd-tree order may differ, and the lines with them."""
from __future__ import annotations

import numpy as np

import _lp3_worlds as lw
from _agent_params import full_params, mixed_params, oracle_sims_per_agent
from _common import pillar_hall, snake
from collision_avoidance_b200 import scenarios
from oracle.helpers import goal_pref, oracle_sims


def _polys(scn, e):
    return scn.obstacles[e] if scn.per_env_obstacles else scn.obstacles


def has_tie(pos, nd):
    """Some agent with two others at bit-equal squared distance below nd^2 (nd: scalar or [N])."""
    p = pos.astype(np.float32)
    nd = np.broadcast_to(np.asarray(nd, np.float32), (len(p),))
    for i in range(len(p)):
        d = (p - p[i]).astype(np.float32)
        dsq = np.delete(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1], i)
        dsq = dsq[dsq < nd[i] * nd[i]]
        if len(np.unique(dsq)) < len(dsq):
            return True
    return False


def oracle_case(name, scn, warm=0, agent_params=None, max_tries=40):
    """Run the oracle `warm` steps toward the goals (more while the state has a tie), then one more
    step; returns dict(name, scn, params (snake), pos, vel [E, N, 2] = the state before that step,
    pref, agent_params, progs: per env a list of (lines [n, 4], n_obst))."""
    sims = oracle_sims(scn) if agent_params is None else oracle_sims_per_agent(scn, agent_params)
    nd = scn.params["neighborDist"] if agent_params is None else full_params(scn, agent_params)["neighbor_dist"]
    nd = np.broadcast_to(np.asarray(nd, np.float32), scn.pos.shape[:2])

    def step():
        for e, s in enumerate(sims):
            s.set_pref_velocities(goal_pref(s.positions(), scn.goal[e]).astype(np.float32))
            s.doStep()

    for _ in range(warm):
        step()
    for _ in range(max_tries):
        pos = np.stack([s.positions() for s in sims]).astype(np.float32)
        if not any(has_tie(pos[e], nd[e]) for e in range(scn.num_envs)):
            break
        step()
    else:
        raise AssertionError(f"{name}: no tie-free state")
    vel = np.stack([s.velocities() for s in sims]).astype(np.float32)
    pref = np.stack([goal_pref(pos[e], scn.goal[e]) for e in range(scn.num_envs)]).astype(np.float32)
    progs = []
    for e, s in enumerate(sims):
        s.set_pref_velocities(pref[e])
        s.doStep()
        progs.append([s.orca_lines(i) for i in range(scn.agents_per_env)])
    return dict(name=name, scn=scn, params=snake(scn.params), pos=pos, vel=vel, pref=pref, agent_params=agent_params,
                progs=progs, polys=[_polys(scn, e) for e in range(scn.num_envs)])


def _jam_case(N, c, kind, k, seed):
    pos, vel, goal, _, _ = lw.env(N, c, kind, k, seed)
    scn = scenarios.Scenario("lp3_" + kind, pos[None].copy(), vel[None].copy(), goal[None].copy(), goal[None].copy(),
                             lw.BOX, [list(lw.WALL)], params=lw.params(k))
    return oracle_case(f"lp3_{kind}_{N}_k{k}", scn)


def _lonely(seed=3):
    """20 agents in a 6 x 6 box and one 40 units away from everything: no neighbor, no obstacle."""
    rng = np.random.default_rng(seed)
    pos = np.concatenate([rng.uniform(0, 6, (20, 2)), [[46.0, 46.0]]])[None].astype(np.float32)
    vel = rng.uniform(-1, 1, pos.shape).astype(np.float32)
    goal = (6.0 - pos).astype(np.float32)
    return scenarios.Scenario("lonely", pos, vel, goal, goal.copy(), 50.0, [[(-1.0, -1.0), (-1.0, 7.0), (7.0, 7.0), (7.0, -1.0)]])


def _overlap(seed=4):
    """Agents packed at 0.6 - 0.9 of a diameter apart: every neighbor line takes the collision branch."""
    rng = np.random.default_rng(seed)
    g = np.stack(np.meshgrid(np.arange(5), np.arange(5)), -1).reshape(-1, 2) * 0.8
    pos = (g + rng.uniform(-0.05, 0.05, g.shape))[None].astype(np.float32)
    vel = rng.uniform(-1, 1, pos.shape).astype(np.float32)
    return scenarios.Scenario("overlap", pos, vel, -pos, -pos, 10.0, [])


def cpu_cases():
    """Every world of the host test: (case, grid) pairs."""
    out = []
    c16 = oracle_case("circle16", scenarios.circle(3, 16, seed=1), warm=40)
    c32 = oracle_case("circle32", scenarios.circle(2, 32, seed=2), warm=60)
    crowd = oracle_case("crowd256_blocks", scenarios.crowd(1, 256, seed=3, blocks=4), warm=20)
    hall = oracle_case("pillar_hall", pillar_hall(num_agents=12, seed=1), warm=30)
    dead = oracle_case("deadlock", scenarios.deadlock(2, 10, seed=4), warm=50)
    cong = oracle_case("congested", scenarios.congested(2, 12, seed=5), warm=40)
    jams = [_jam_case(32, 12, "jam", 10, 11), _jam_case(24, 8, "walled", 5, 12), _jam_case(40, 10, "queue", 16, 13)]
    crowd40 = scenarios.crowd(2, 40, seed=6, blocks=2)
    mixed = oracle_case("mixed_params", crowd40, warm=10, agent_params=mixed_params(2, 40, 10, seed=6))
    lonely = oracle_case("lonely", _lonely())
    overlap = oracle_case("overlap", _overlap())
    big = oracle_case("grid_crowd1024", scenarios.crowd(1, 1024, seed=7, blocks=4), warm=5)
    for c in (c16, c32, crowd, hall, dead, cong, *jams, mixed, lonely, overlap):
        out.append((c, False))
        out.append((c, True))
    out.append((big, True))
    return out
