"""CPU check of the heterogeneous step body (per-agent radius, maxSpeed, neighborDist, maxNeighbors,
timeHorizon, timeHorizonObst): the library's device code compiled for the host by
tests/host_emul/emul_hetero.cpp, through the tile source and the grid source, against oracle
simulators built with one addAgent per agent."""
import numpy as np

import _emul
from _emul_hetero import emul_step_hetero
from _agent_params import max_obstacle_range, mixed_params, oracle_sims_per_agent
from _common import goal_pref, neighbor_sets_equal_up_to_ties, pillar_hall, snake
from collision_avoidance_b200 import scenarios


def _compare(scn, ap, steps, grid=False, sample_stride=1, hint=False):
    P = snake(scn.params)
    # the library's threshold hints (agent_front): persistent between steps
    hints = np.full((scn.num_envs, 1, scn.agents_per_env), 3.0e38, np.float32) if hint else None
    orange = max_obstacle_range(scn, ap)
    polys = scn.obstacles
    worlds = ([_emul.World(p, orange) for p in polys] if scn.per_env_obstacles
              else [_emul.World(polys, orange)] * scn.num_envs)
    sims = oracle_sims_per_agent(scn, ap)
    E, N = scn.num_envs, scn.agents_per_env
    worst, exact_agents = 0.0, 0
    stats = np.zeros(8, np.uint64)
    for _ in range(steps):
        pos = np.stack([s.positions() for s in sims])
        vel = np.stack([s.velocities() for s in sims])
        pref = goal_pref(pos, scn.goal).astype(np.float32)
        for e, s in enumerate(sims):
            s.set_pref_velocities(pref[e])
            s.doStep()
        for e in range(E):
            pe, ve = pos[e:e + 1].copy(), vel[e:e + 1].copy()
            ape = {k: v[e:e + 1] for k, v in ap.items()}
            out = emul_step_hetero(P, pe, ve, ape, pref=np.ascontiguousarray(pref[e:e + 1]), world=worlds[e],
                                   stats=stats, grid=grid, nbr_hint=None if hints is None else hints[e])
            op, ov = sims[e].positions(), sims[e].velocities()
            for i in range(0, N, sample_stride):
                o_ids = [x[0] for x in sims[e].agent_neighbors(i)]
                g_ids = list(out["nbr_idx"][0, i, :out["nbr_cnt"][0, i]])
                dsq = lambda j: float(np.float32(((pos[e, i] - pos[e, j]) ** 2).sum()))
                assert neighbor_sets_equal_up_to_ties(o_ids, g_ids, dsq), (i, o_ids, g_ids)
                # (the obstacle-neighbor output holds the 16 nearest edges)
                assert [x[0] for x in sims[e].obstacle_neighbors(i)][:16] == list(out["onbr_idx"][0, i, :out["onbr_cnt"][0, i]])
                diff = max(float(np.abs(pe[0, i] - op[i]).max()), float(np.abs(ve[0, i] - ov[i]).max()))
                if o_ids == g_ids:  # identical ordered lists: bit-identical result
                    worst = max(worst, diff)
                    exact_agents += 1
                elif set(o_ids) == set(g_ids):  # same neighbors, bit-equal distances in another order
                    assert diff <= 1e-4, (i, diff)
                # else: a bit-equal tie at the k-th distance (symmetric rings with an odd maxNeighbors):
                # which of the equally distant agents RVO2 keeps is its kd-tree's visiting order
    assert exact_agents > 0
    return worst, stats


def test_tile_source_mixed_parameters():
    scn = scenarios.crowd(2, 40, seed=11, blocks=4)
    worst, stats = _compare(scn, mixed_params(2, 40, scn.params["maxNeighbors"], seed=1), steps=40)
    assert worst == 0.0
    assert stats[3] > 0 and stats[2] > 0       # LP3 and the collision branch were exercised


def test_tile_source_small_worlds_ranked_selection():
    for scn in (scenarios.circle(2, 16, seed=12), scenarios.circle(1, 32, seed=13), scenarios.deadlock(1, 20, seed=14),
                scenarios.congested(1, 24, seed=15)):
        worst, _ = _compare(scn, mixed_params(scn.num_envs, scn.agents_per_env, scn.params["maxNeighbors"], seed=2),
                            steps=40)
        assert worst == 0.0, scn.name


def test_tile_source_single_parameters_mixed():
    """One array at a time: the others take the handle's values."""
    scn = scenarios.crowd(1, 40, seed=16, blocks=3)
    full = mixed_params(1, 40, scn.params["maxNeighbors"], seed=3)
    for name in full:
        worst, _ = _compare(scn, {name: full[name]}, steps=15)
        assert worst == 0.0, name


def test_grid_source_mixed_parameters():
    scn = scenarios.crowd(1, 600, seed=17)
    worst, _ = _compare(scn, mixed_params(1, 600, scn.params["maxNeighbors"], seed=4), steps=8, grid=True,
                        sample_stride=5)
    assert worst == 0.0


def test_slow_path_world_mixed_parameters():
    """pillar_hall overflows the fast path's obstacle capacities: agent_slow_path with per-agent records."""
    scn = pillar_hall(num_agents=12, seed=3)
    ap = mixed_params(1, 12, scn.params["maxNeighbors"], seed=5)
    for grid in (False, True):
        worst, stats = _compare(scn, ap, steps=30, grid=grid)
        assert worst == 0.0
        assert stats[4] == 0          # ORCA_STAT_OVERFLOW: nothing exceeded the slow path


def test_threshold_hint_scratch_with_per_agent_parameters():
    """With the library's threshold-hint scratch present (worlds of more than 32 agents), the
    heterogeneous body still returns the exact lists (tile and grid)."""
    for scn, grid, stride in ((scenarios.crowd(1, 80, seed=18, blocks=3), False, 1), (scenarios.crowd(1, 500, seed=19), True, 7)):
        K = scn.params["maxNeighbors"]
        ap = mixed_params(1, scn.agents_per_env, K, seed=6)
        ap["max_neighbors"][:, ::2] = K
        ap["neighbor_dist"] = np.minimum(ap["neighbor_dist"], np.float32(scn.params["neighborDist"]))
        worst, _ = _compare(scn, ap, steps=15, grid=grid, sample_stride=stride, hint=True)
        assert worst == 0.0
