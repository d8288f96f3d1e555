"""Per-agent ORCA parameters on the GPU (orca_set_agent_params / BatchedRVOSimulator.set_agent_params /
rvo2_compat's per-agent addAgent and setters):
  - a table that holds the handle's own values gives the uniform kernels' outputs bit for bit,
  - mixed parameters match oracle simulators built with one addAgent per agent (the bar of
    test_gpu_parity_step.py),
  - the collision statistic counts pairs within r_i + r_j,
  - the rvo2 shim, errors, and the return to uniform parameters."""
import numpy as np
import pytest

from _agent_params import NAMES, full_params, max_obstacle_range, mixed_params, oracle_sims_per_agent
from _common import OraclePyRVO, goal_pref, neighbor_sets_equal_up_to_ties, pillar_hall

pytestmark = pytest.mark.gpu

TOL = 1e-4


def _sim(scn, ap=None, obstacles_first=True):
    import torch
    from collision_avoidance_b200.sim import BatchedRVOSimulator
    sim = BatchedRVOSimulator(scn.num_envs, scn.agents_per_env, device="cuda:0", **scn.params)
    if obstacles_first:
        sim.set_obstacles(scn.obstacles, per_env=scn.per_env_obstacles)
    if ap is not None:
        sim.set_agent_params(**ap)
    if not obstacles_first:
        sim.set_obstacles(scn.obstacles, per_env=scn.per_env_obstacles)
    sim.pos.copy_(torch.from_numpy(scn.pos))
    sim.vel.copy_(torch.from_numpy(scn.vel))
    return sim


def _handle_table(scn):
    """All six arrays, every entry the handle's own value."""
    return full_params(scn, {})


# ---------------------------------------------------------------- 1. uniform values, new path
def _drive(sim, scn, kind, steps):
    """`steps` fused steps of one kind; every output the step produces, as numpy arrays."""
    import torch
    from collision_avoidance_b200 import _lib
    E, N = scn.num_envs, scn.agents_per_env
    dev = sim.pos.device
    goal = torch.from_numpy(scn.goal).to(dev)
    goal2 = torch.from_numpy(scn.goal2).to(dev)
    out = {k: [] for k in ("pos", "vel", "nbr_idx", "nbr_cnt", "obst_idx", "obst_cnt", "reward", "w", "act", "done")}
    reward = torch.zeros(E, N, dtype=torch.float32, device=dev)
    done = torch.zeros(E, N, dtype=torch.uint8, device=dev)
    arrival = torch.zeros(E, N, dtype=torch.float32, device=dev)
    env_step = torch.zeros(E, dtype=torch.int32, device=dev)
    env_done = torch.zeros(E, dtype=torch.int32, device=dev)
    g = torch.Generator().manual_seed(3)
    acts = torch.nn.functional.normalize(torch.randn(8, 2, generator=g), dim=1).to(dev)
    w = torch.zeros(E, N, 8, dtype=torch.float32, device=dev)
    act = torch.zeros(E, N, dtype=torch.uint8, device=dev)
    for t in range(steps):
        if kind == "goal":
            sim.env_step(policy=_lib.POLICY_GOAL, goal=goal, want_neighbors=True)
        elif kind == "rl":
            theta = (torch.rand(E, N, generator=g) * 2 - 1).to(dev)
            sim.env_step(policy=_lib.POLICY_RL, goal=goal, goal2=goal2, action_theta=theta, reward=reward,
                         done_mode=_lib.DONE_X_BELOW, agent_done=done, env_step=env_step, env_done_cnt=env_done,
                         want_neighbors=True)
        else:  # alan
            sim.env_step(policy=_lib.POLICY_ALAN, goal=goal, goal2=goal2, alan_weights=w, alan_actions=acts,
                         alan_action_out=act, rng_seed=11, reward=reward, done_mode=_lib.DONE_GOAL_RADIUS,
                         agent_done=done, arrival_time=arrival, env_step=env_step, env_done_cnt=env_done,
                         want_neighbors=True)
        for k, v in (("pos", sim.pos), ("vel", sim.vel), ("nbr_idx", sim.nbr_idx), ("nbr_cnt", sim.nbr_cnt),
                     ("obst_idx", sim.obst_nbr_idx), ("obst_cnt", sim.obst_nbr_cnt), ("reward", reward), ("w", w),
                     ("act", act), ("done", done)):
            out[k].append(v.cpu().numpy().copy())
    out["stats"] = [sim.stats.cpu().numpy().copy()]
    out["arrival"] = [arrival.cpu().numpy()]
    return {k: np.stack(v) for k, v in out.items()}


def _assert_same(a, b):
    for k in a:
        assert a[k].tobytes() == b[k].tobytes(), k


def _uniform_cases():
    from collision_avoidance_b200 import scenarios
    env = scenarios.default_env(64, 10, seed=4)      # the gym env's shape and parameters: maxNeighbors 5
    return [("circle16", scenarios.circle(8, 16, seed=1), "goal", 30),
            ("circle32", scenarios.circle(4, 32, seed=2), "goal", 30),
            ("crowd64_blocks", scenarios.crowd(4, 64, seed=3, blocks=4), "goal", 30),
            ("gym_rl_x_below", env, "rl", 30),
            ("alan_goal_radius", scenarios.crowd(4, 24, seed=5, blocks=2), "alan", 40),
            ("crowd700_grid", scenarios.crowd(1, 700, seed=6), "goal", 8)]


@pytest.mark.parametrize("case", range(6), ids=["circle16", "circle32", "crowd64_blocks", "gym_rl_x_below",
                                                "alan_goal_radius", "crowd700_grid"])
def test_handle_values_through_the_table_are_bit_identical(case):
    name, scn, kind, steps = _uniform_cases()[case]
    if name == "gym_rl_x_below":
        assert scn.params["maxNeighbors"] == 5
    a = _drive(_sim(scn), scn, kind, steps)
    b = _drive(_sim(scn, _handle_table(scn)), scn, kind, steps)
    _assert_same(a, b)
    assert a["stats"][0][0] > 0


@pytest.mark.parametrize("pinned", [True, False], ids=["direct", "staged"])
def test_handle_values_through_the_table_host_step(pinned):
    import torch
    from collision_avoidance_b200 import _lib, scenarios
    scn = scenarios.circle(64, 16, seed=8)
    res = []
    for ap in (None, _handle_table(scn)):
        sim = _sim(scn, ap)
        mk = (lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()) if pinned else \
             (lambda a: torch.from_numpy(np.ascontiguousarray(a)).clone())
        pos, vel, goal = mk(scn.pos), mk(scn.vel), mk(scn.goal)
        traj = []
        for t in range(12):
            sim.step_host(pos, vel, goal, policy=_lib.POLICY_GOAL, upload_state=(t == 0), steps=1 + (t % 3 == 2))
            traj.append(pos.numpy().copy())
            traj.append(vel.numpy().copy())
        res.append(np.stack(traj))
    assert res[0].tobytes() == res[1].tobytes()


# ---------------------------------------------------------------- 2. mixed parameters vs the oracle
def _oracle_case(scn, ap, steps, obstacles_first=True):
    import torch
    sims = oracle_sims_per_agent(scn, ap)
    gpu = _sim(scn, ap, obstacles_first)
    E, N = scn.num_envs, scn.agents_per_env
    worst, n_exact, n_total = 0.0, 0, 0
    for t in range(steps):
        pos = np.stack([s.positions() for s in sims])
        vel = np.stack([s.velocities() for s in sims])
        pref = goal_pref(pos, scn.goal).astype(np.float32)
        for e, s in enumerate(sims):
            s.set_pref_velocities(pref[e])
            s.doStep()
        gpu.pos.copy_(torch.from_numpy(pos))
        gpu.vel.copy_(torch.from_numpy(vel))
        gpu.pref.copy_(torch.from_numpy(pref))
        gpu.env_step(policy=0, want_neighbors=True)
        gp, gv = gpu.pos.cpu().numpy(), gpu.vel.cpu().numpy()
        nbr_idx, nbr_cnt = gpu.nbr_idx.cpu().numpy(), gpu.nbr_cnt.cpu().numpy()
        onbr_idx, onbr_cnt = gpu.obst_nbr_idx.cpu().numpy(), gpu.obst_nbr_cnt.cpu().numpy()
        for e in range(E):
            op, ov = sims[e].positions(), sims[e].velocities()
            for i in range(N):
                o_ids = [x[0] for x in sims[e].agent_neighbors(i)]
                g_ids = list(nbr_idx[e, i, :nbr_cnt[e, i]])
                dsq = lambda j: float(np.float32(((pos[e, i] - pos[e, j]) ** 2).sum()))
                assert neighbor_sets_equal_up_to_ties(o_ids, g_ids, dsq), (t, e, i, o_ids, g_ids)
                o_ob = [x[0] for x in sims[e].obstacle_neighbors(i)][:16]   # the output holds the 16 nearest
                assert o_ob == list(onbr_idx[e, i, :onbr_cnt[e, i]]), (t, e, i)
                diff = max(float(np.abs(gp[e, i] - op[i]).max()), float(np.abs(gv[e, i] - ov[i]).max()))
                if o_ids == g_ids:
                    n_total += 1
                    n_exact += int(diff == 0.0)
                    worst = max(worst, diff)
                elif set(o_ids) == set(g_ids):
                    worst = max(worst, diff)
                # else: bit-equal tie at the k-th distance; RVO2 keeps the one its kd-tree visits first
    assert worst <= TOL, worst
    assert n_total > 0 and n_exact == n_total, (n_exact, n_total)
    assert gpu.read_stats()["overflow"] == 0
    return gpu


def _mixed_cases():
    from collision_avoidance_b200 import scenarios
    return [("circle16", scenarios.circle(4, 16, seed=21), 30), ("circle32", scenarios.circle(2, 32, seed=22), 30),
            ("crowd64_blocks", scenarios.crowd(3, 64, seed=23, blocks=4), 25),
            ("deadlock", scenarios.deadlock(2, 20, seed=24), 30), ("congested", scenarios.congested(2, 24, seed=25), 30),
            ("crowd700_grid", scenarios.crowd(1, 700, seed=26), 6), ("pillar_hall", pillar_hall(12, seed=4), 40)]


@pytest.mark.parametrize("case", range(7), ids=["circle16", "circle32", "crowd64_blocks", "deadlock", "congested",
                                                "crowd700_grid", "pillar_hall"])
def test_mixed_parameters_match_the_oracle(case):
    name, scn, steps = _mixed_cases()[case]
    ap = mixed_params(scn.num_envs, scn.agents_per_env, scn.params["maxNeighbors"], seed=100 + case)
    P = scn.params
    # agents whose obstacle range exceeds the handle's: the obstacle-free maps must be built for the largest
    assert max_obstacle_range(scn, ap) > P["timeHorizonObst"] * P["maxSpeed"] + P["radius"]
    _oracle_case(scn, ap, steps, obstacles_first=(case % 2 == 0))


def test_large_speed_agent_near_walls_with_obstacles_set_after():
    """One fast agent (obstacle range 3 * 4 + 0.5) among default ones, obstacles set after the table."""
    from collision_avoidance_b200 import scenarios
    scn = scenarios.crowd(2, 64, seed=27, blocks=5)
    vmax = np.full((2, 64), scn.params["maxSpeed"], np.float32)
    tho = np.full((2, 64), scn.params["timeHorizonObst"], np.float32)
    vmax[:, ::9] = 4.0
    tho[:, ::9] = 3.0
    _oracle_case(scn, dict(max_speed=vmax, time_horizon_obst=tho), 30, obstacles_first=False)


# ---------------------------------------------------------------- 3. collision statistic
def test_collision_statistic_counts_pairs_within_the_sum_of_radii():
    import torch
    from collision_avoidance_b200 import _lib, scenarios
    for scn in (scenarios.crowd(4, 64, seed=31), scenarios.crowd(1, 600, seed=32)):
        E, N = scn.num_envs, scn.agents_per_env
        rng = np.random.default_rng(7)
        rad = rng.uniform(0.2, 0.8, (E, N)).astype(np.float32)
        gpu = _sim(scn, dict(radius=rad))
        expect = 0
        for t in range(10):
            pos = gpu.pos.cpu().numpy()
            gpu.env_step(policy=_lib.POLICY_GOAL, goal=torch.from_numpy(scn.goal).cuda(), want_neighbors=True)
            idx, cnt = gpu.nbr_idx.cpu().numpy(), gpu.nbr_cnt.cpu().numpy()
            for e in range(E):
                for i in range(N):
                    js = idx[e, i, :cnt[e, i]]
                    d = pos[e, js] - pos[e, i]             # as agent_line: relative position, then distSq
                    dsq = d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]
                    cr = rad[e, i] + rad[e, js]
                    expect += int((dsq <= cr * cr).sum())
        assert expect > 50
        assert gpu.read_stats()["collisions"] == expect


# ---------------------------------------------------------------- 4. rvo2_compat
def _compat_world(seed):
    rng = np.random.default_rng(seed)
    n = 24
    pos = rng.uniform(0, 8, (n, 2)).astype(np.float32)
    goal = (8 - pos).astype(np.float32)
    prm = mixed_params(1, n, 10, seed)
    return pos, goal, prm, [(0.0, 0.0), (0.0, 9.0), (9.0, 9.0), (9.0, 0.0)]


def _add_agents(sim, pos, prm, vel=None):
    for i in range(pos.shape[0]):
        v = (0.0, 0.0) if vel is None else tuple(map(float, vel[i]))
        sim.addAgent(tuple(map(float, pos[i])), float(prm["neighbor_dist"][0, i]), int(prm["max_neighbors"][0, i]),
                     float(prm["time_horizon"][0, i]), float(prm["time_horizon_obst"][0, i]), float(prm["radius"][0, i]),
                     float(prm["max_speed"][0, i]), v)


def _step_both(shim, orc, goal, steps):
    n = goal.shape[0]
    for _ in range(steps):
        p = np.array([orc.getAgentPosition(i) for i in range(n)], np.float32)
        pref = goal_pref(p, goal).astype(np.float32)
        for i in range(n):
            shim.setAgentPrefVelocity(i, tuple(map(float, pref[i])))
            orc.setAgentPrefVelocity(i, tuple(map(float, pref[i])))
        shim.doStep()
        orc.doStep()
        for i in range(n):
            assert np.abs(np.subtract(shim.getAgentPosition(i), orc.getAgentPosition(i))).max() <= TOL
            assert np.abs(np.subtract(shim.getAgentVelocity(i), orc.getAgentVelocity(i))).max() <= TOL


def test_compat_mixed_agents_match_the_oracle_for_200_steps():
    from collision_avoidance_b200 import rvo2_compat
    pos, goal, prm, wall = _compat_world(41)
    args = (1 / 60., 5.0, 10, 1.5, 1.5, 0.5, 1.0)
    shim, orc = rvo2_compat.PyRVOSimulator(*args), OraclePyRVO(*args)
    for s in (shim, orc):
        _add_agents(s, pos, prm)
        s.addObstacle(wall)
        s.processObstacles()
    _step_both(shim, orc, goal, 200)


def test_compat_setters_take_effect_at_the_next_step_and_getters_return_them():
    from collision_avoidance_b200 import rvo2_compat
    pos, goal, prm, wall = _compat_world(42)
    args = (1 / 60., 5.0, 10, 1.5, 1.5, 0.5, 1.0)
    shim, orc = rvo2_compat.PyRVOSimulator(*args), OraclePyRVO(*args)
    for s in (shim, orc):
        _add_agents(s, pos, prm)
        s.addObstacle(wall)
        s.processObstacles()
    _step_both(shim, orc, goal, 40)
    # new parameters for a third of the agents, set on the shim only
    new = {k: v.copy() for k, v in prm.items()}
    rng = np.random.default_rng(43)
    setters = dict(neighbor_dist="setAgentNeighborDist", max_neighbors="setAgentMaxNeighbors",
                   time_horizon="setAgentTimeHorizon", time_horizon_obst="setAgentTimeHorizonObst",
                   radius="setAgentRadius", max_speed="setAgentMaxSpeed")
    fresh = mixed_params(1, pos.shape[0], 10, 44)
    for i in rng.choice(pos.shape[0], 8, replace=False):
        for name, fn in setters.items():
            new[name][0, i] = fresh[name][0, i]
            getattr(shim, fn)(int(i), fresh[name][0, i].item())
    getters = dict(neighbor_dist="getAgentNeighborDist", max_neighbors="getAgentMaxNeighbors",
                   time_horizon="getAgentTimeHorizon", time_horizon_obst="getAgentTimeHorizonObst",
                   radius="getAgentRadius", max_speed="getAgentMaxSpeed")
    for i in range(pos.shape[0]):
        for name, fn in getters.items():
            assert getattr(shim, fn)(i) == new[name][0, i].item(), (i, name)
    # an oracle rebuilt from the shim's state with the new parameters
    n = pos.shape[0]
    p_now = np.array([shim.getAgentPosition(i) for i in range(n)], np.float32)
    v_now = np.array([shim.getAgentVelocity(i) for i in range(n)], np.float32)
    orc2 = OraclePyRVO(*args)
    _add_agents(orc2, p_now, new, v_now)
    orc2.addObstacle(wall)
    orc2.processObstacles()
    _step_both(shim, orc2, goal, 60)


def test_compat_agent_with_other_parameters_after_a_default_agent():
    from collision_avoidance_b200 import rvo2_compat
    sim = rvo2_compat.PyRVOSimulator(1 / 60., 1.5, 5, 1.5, 2.0, 0.4, 1.0)
    sim.addAgent((0.0, 0.0))
    sim.addAgent((1.0, 0.0), 1.5, 5, 1.5, 2.0, 0.3, 1.4, (0, 0))
    sim.setAgentPrefVelocity(0, (1.0, 0.0))
    sim.setAgentPrefVelocity(1, (-1.0, 0.0))
    sim.doStep()
    assert sim.getAgentRadius(1) == np.float32(0.3).item() and sim.getAgentMaxSpeed(0) == 1.0
    assert sim.getAgentNumAgentNeighbors(0) == 1


# ---------------------------------------------------------------- 5. errors and the return to uniform
def test_bad_values_raise_value_error():
    from collision_avoidance_b200 import scenarios
    scn = scenarios.crowd(2, 40, seed=51)
    sim = _sim(scn)
    E, N = 2, 40
    k = scn.params["maxNeighbors"]
    f = lambda v: np.full((E, N), v, np.float32)
    bad = [dict(max_neighbors=np.full((E, N), k + 1, np.int32)), dict(max_neighbors=np.full((E, N), -1, np.int32)),
           dict(radius=f(-0.1)), dict(time_horizon=f(0.0)), dict(time_horizon_obst=f(-1.0)),
           dict(max_speed=f(np.nan)), dict(neighbor_dist=f(np.inf)), dict(radius=np.full((E, N + 1), 0.5, np.float32)),
           dict(max_speed=np.full((E * N,), 1.0, np.float32))]
    for kw in bad:
        with pytest.raises(ValueError):
            sim.set_agent_params(**kw)


def test_no_arguments_returns_to_the_uniform_outputs():
    import torch
    from collision_avoidance_b200 import scenarios
    scn = scenarios.crowd(4, 64, seed=52, blocks=3)
    ref = _drive(_sim(scn), scn, "goal", 15)
    sim = _sim(scn, mixed_params(4, 64, scn.params["maxNeighbors"], seed=53))
    _drive(sim, scn, "goal", 5)
    sim.set_agent_params()
    sim.stats.zero_()
    sim.pos.copy_(torch.from_numpy(scn.pos))
    sim.vel.copy_(torch.from_numpy(scn.vel))
    _assert_same(ref, _drive(sim, scn, "goal", 15))


def test_tensor_arguments_on_the_device():
    import torch
    from collision_avoidance_b200 import scenarios
    scn = scenarios.crowd(2, 40, seed=54)
    ap = mixed_params(2, 40, scn.params["maxNeighbors"], seed=55)
    a = _drive(_sim(scn, ap), scn, "goal", 10)
    b = _drive(_sim(scn, {k: torch.from_numpy(v).cuda() for k, v in ap.items()}), scn, "goal", 10)
    _assert_same(a, b)
    assert set(ap) == set(NAMES)
