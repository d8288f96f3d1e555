"""LP3 of the step kernels under jams: batches whose tile-kernel blocks hold exactly the LP3 totals at
block_lp3's boundaries (tests/_lp3_worlds.py: 0, 1, 31/32/33, half the block and one either side, 5/8,
7/8, all but one, all), stepped on the GPU and compared with the oracle bit for bit -- every agent, no
tie exemption (the worlds have no bit-equal neighbor distances) -- on every kernel variant that runs
block_lp3: tile K = 5 / 10 slim / 10 full / 16, blocks of 32 to 256 threads, the uniform-grid kernel,
and the per-agent-parameter (HETERO) kernels, where a solver thread takes its OWNER's maxSpeed."""
import numpy as np
import pytest

import _lp3_worlds as W

pytestmark = pytest.mark.gpu

STEPS = 3  # one step from the constructed state, then two more re-synchronised to the oracle


def _gpu(batch, k, agent_params=None):
    import torch
    from collision_avoidance_b200.sim import BatchedRVOSimulator
    E, N = batch["pos"].shape[:2]
    sim = BatchedRVOSimulator(E, N, device="cuda:0", **W.params(k))
    sim.set_obstacles([list(W.WALL)])
    if agent_params is not None:
        sim.set_agent_params(**agent_params)
    sim.pos.copy_(torch.from_numpy(batch["pos"]))
    sim.vel.copy_(torch.from_numpy(batch["vel"]))
    return sim


def _against_oracle(batch, k, agent_params=None):
    """STEPS oracle-synchronised steps under POLICY_EXTERNAL and POLICY_GOAL: ordered neighbor and
    obstacle lists, positions and velocities bit-identical for every agent, the lp3_calls statistic
    equal to the oracle's count of agents whose LP2 failed, no overflow.  Returns the LP3 counts."""
    import torch
    from collision_avoidance_b200 import _lib
    E, N = batch["pos"].shape[:2]
    P = W.params(k)
    ap = agent_params
    sims = [W.oracle_sim(P, batch["pos"][e], batch["vel"][e], None if ap is None else {n: v[e] for n, v in ap.items()})
            for e in range(E)]
    vmax = ap["max_speed"] if ap is not None else np.full((E, N), P["maxSpeed"], np.float32)
    goal = batch["goal"]
    goal_t = torch.from_numpy(goal).cuda()
    gpus = {_lib.POLICY_EXTERNAL: _gpu(batch, k, ap), _lib.POLICY_GOAL: _gpu(batch, k, ap)}
    counts = []
    for t in range(STEPS):
        pos = np.stack([s.positions() for s in sims])
        vel = np.stack([s.velocities() for s in sims])
        pref = W.goal_dir(pos, goal)
        n_lp3 = 0
        for e, s in enumerate(sims):
            s.set_pref_velocities(pref[e])
            s.doStep()
            n_lp3 += int(W.lp3_agents(s, pref[e], vmax[e])[0].sum())
        counts.append(n_lp3)
        o_nbr = [[[j for j, _ in s.agent_neighbors(i)] for i in range(N)] for s in sims]
        o_obs = [[[j for j, _ in s.obstacle_neighbors(i)] for i in range(N)] for s in sims]
        op = np.stack([s.positions() for s in sims])
        ov = np.stack([s.velocities() for s in sims])
        for policy, g in gpus.items():
            g.pos.copy_(torch.from_numpy(pos))
            g.vel.copy_(torch.from_numpy(vel))
            g.pref.copy_(torch.from_numpy(pref))
            before = g.read_stats()["lp3_calls"]
            g.env_step(policy=policy, goal=goal_t if policy == _lib.POLICY_GOAL else None, want_neighbors=True)
            st = g.read_stats()
            assert st["overflow"] == 0
            assert st["lp3_calls"] - before == n_lp3, (policy, t, st["lp3_calls"] - before, n_lp3)
            idx, cnt = g.nbr_idx.cpu().numpy(), g.nbr_cnt.cpu().numpy()
            oidx, ocnt = g.obst_nbr_idx.cpu().numpy(), g.obst_nbr_cnt.cpu().numpy()
            for e in range(E):
                for i in range(N):
                    assert list(idx[e, i, :cnt[e, i]]) == o_nbr[e][i], (policy, t, e, i)
                    assert list(oidx[e, i, :ocnt[e, i]]) == o_obs[e][i], (policy, t, e, i)
            gp, gv = g.pos.cpu().numpy(), g.vel.cpu().numpy()
            bad = np.argwhere((gp.view(np.int32) != op.view(np.int32)).any(-1) | (gv.view(np.int32) != ov.view(np.int32)).any(-1))
            assert len(bad) == 0, (policy, t, len(bad), bad[:5].tolist())
    return counts


# (N, tpb) shapes per kernel variant: together every N in {16, 24, 32, 40, 100, 256} with every block size
# of the tile kernel that holds it, each variant with at least one 256-thread block shape
CASES = [
    ("k5", 5, (16, 256)), ("k5", 5, (16, 128)), ("k5", 5, (24, 64)), ("k5", 5, (32, 32)), ("k5", 5, (40, 128)),
    ("k5", 5, (100, 256)), ("k5", 5, (256, 256)),
    ("k10slim", 10, (16, 256)), ("k10slim", 10, (16, 64)), ("k10slim", 10, (24, 32)), ("k10slim", 10, (32, 128)),
    ("k10full", 10, (16, 256)), ("k10full", 10, (32, 64)), ("k10full", 10, (40, 256)), ("k10full", 10, (100, 128)),
    ("k16", 7, (32, 256)), ("k16", 13, (24, 128)), ("k16", 16, (40, 64)), ("k16", 13, (256, 256)), ("k16", 16, (16, 32)),
    ("k16", 7, (24, 256)),
]


@pytest.mark.parametrize("variant,k,shape", CASES, ids=[f"{v}-k{k}-N{s[0]}-tpb{s[1]}" for v, k, s in CASES])
def test_tile_kernel_lp3_boundaries_match_oracle(variant, k, shape, monkeypatch):
    N, tpb = shape
    monkeypatch.setenv("ORCA_B200_TPB", str(tpb))
    if variant == "k10full":
        monkeypatch.setenv("ORCA_B200_NO_SLIM_KERNEL", "1")
    batch = W.assemble(N, tpb, k)
    counts = _against_oracle(batch, k)
    assert counts[0] == sum(batch["targets"])
    print(variant, k, shape, "block totals", batch["targets"], "LP3 agents per step", counts)


def test_grid_kernel_lp3_matches_oracle(monkeypatch):
    """The uniform-grid step kernel (64-thread blocks over the cell-sorted agents, so whole blocks of
    jammed agents: nstored = 0) on an assembled batch, forced with ORCA_B200_GRID_MIN_AGENTS ..."""
    monkeypatch.setenv("ORCA_B200_GRID_MIN_AGENTS", "2")
    batch = W.assemble(16, 256, 10)
    counts = _against_oracle(batch, 10)
    assert counts[0] == sum(batch["targets"])


def test_grid_kernel_lp3_on_a_700_agent_jam():
    """... and on its natural ground: one 700-agent world with a 400-agent jam."""
    pos, vel, goal, need, _ = W.env(700, 400, "walled", 10, 3)
    batch = dict(pos=pos[None], vel=vel[None], goal=goal[None])
    counts = _against_oracle(batch, 10)
    assert counts[0] == 400


@pytest.mark.parametrize("path", ["tile", "grid"])
def test_hetero_kernels_lp3_use_the_owners_max_speed(path, monkeypatch):
    """Per-agent maxSpeed U(0.3, 3) and radii: block_lp3 compacts the LP3 agents to the first threads,
    so most are solved by another thread than their owner; the solver must use the owner's maxSpeed."""
    if path == "grid":
        monkeypatch.setenv("ORCA_B200_GRID_MIN_AGENTS", "2")
    batch = W.hetero_batch(32, 256, 10)
    counts = _against_oracle(batch, 10, agent_params=batch["agent_params"])
    assert counts[0] == int(batch["need"].sum()) > 500


@pytest.mark.parametrize("N,tpb,k", [(16, 256, 10), (100, 128, 5)])
def test_rl_and_alan_lp3_match_the_host_emulation(N, tpb, k, monkeypatch):
    """POLICY_RL and POLICY_ALAN instantiate their own step kernels; the host emulation solves each
    agent's LP3 alone, in reference order.  action_theta = 0 and zero bandit weights keep the policy
    arithmetic free of sin / cos / exp, whose device and host versions may round differently."""
    import torch
    import _emul
    from collision_avoidance_b200 import _lib
    from _common import snake
    monkeypatch.setenv("ORCA_B200_TPB", str(tpb))
    batch = W.assemble(N, tpb, k)
    E = batch["pos"].shape[0]
    P = snake(W.params(k))
    world = _emul.World([list(W.WALL)])
    goal = np.ascontiguousarray(batch["goal"])
    rng = np.random.default_rng(3)
    A = 8
    acts = rng.normal(size=(A, 2)).astype(np.float32)
    acts /= np.linalg.norm(acts, axis=1, keepdims=True)
    for policy in (_lib.POLICY_RL, _lib.POLICY_ALAN):
        g = _gpu(batch, k)
        hp, hv = batch["pos"].copy(), batch["vel"].copy()
        es = np.zeros(E, np.int32)                  # per-env step counters (ALAN's Philox counter and window)
        for t in range(STEPS):
            theta = np.zeros((E, N), np.float32)
            uni = rng.uniform(0, 1, (E, N)).astype(np.float32)
            w = np.zeros((E, N, A), np.float32)
            g.pos.copy_(torch.from_numpy(hp))
            g.vel.copy_(torch.from_numpy(hv))
            reward = torch.zeros(E, N, dtype=torch.float32, device="cuda")
            if policy == _lib.POLICY_RL:
                g.env_step(policy=policy, goal=torch.from_numpy(goal).cuda(), action_theta=torch.from_numpy(theta).cuda(),
                           reward=reward)
                out = _emul.emul_step(P, hp, hv, policy=policy, goal=goal, world=world, action_theta=theta)
            else:
                w_d = torch.from_numpy(w).cuda()
                act = torch.zeros(E, N, dtype=torch.uint8, device="cuda")
                es_d = torch.from_numpy(es).cuda()
                g.env_step(policy=policy, goal=torch.from_numpy(goal).cuda(), alan_weights=w_d,
                           alan_actions=torch.from_numpy(acts).cuda(), alan_action_out=act,
                           alan_uniform=torch.from_numpy(uni).cuda(), reward=reward, env_step=es_d)
                out = _emul.emul_step(P, hp, hv, policy=policy, goal=goal, world=world, alan_w=w, alan_actions=acts,
                                      alan_uniform=uni, env_step=es)
                assert np.array_equal(act.cpu().numpy(), out["action"]), (policy, t)
                assert w_d.cpu().numpy().tobytes() == w.tobytes(), (policy, t)
                assert np.array_equal(es_d.cpu().numpy(), es) and (es == t + 1).all(), (policy, t)
            assert g.pos.cpu().numpy().tobytes() == hp.tobytes(), (policy, t)
            assert g.vel.cpu().numpy().tobytes() == hv.tobytes(), (policy, t)
            assert reward.cpu().numpy().tobytes() == out["reward"].tobytes(), (policy, t)
        assert g.read_stats()["overflow"] == 0


@pytest.mark.parametrize("N,k", [(16, 10), (32, 10), (40, 13)])
def test_block_size_and_env_order_do_not_change_any_bit(N, k, monkeypatch):
    """Metamorphic: the same batch under every block size the tile kernel allows for N, and with its
    envs permuted (so every env meets other LP3 totals, queue slots and borrowed columns), gives the
    same bits per env."""
    import torch
    from collision_avoidance_b200 import _lib
    batch = W.assemble(N, 256, k)
    E = batch["pos"].shape[0]
    perm = np.random.default_rng(1).permutation(E)
    results = []
    for tpb in [t for t in (32, 64, 128, 256) if t >= N]:
        for order in (np.arange(E), perm):
            monkeypatch.setenv("ORCA_B200_TPB", str(tpb))
            b = dict(pos=batch["pos"][order].copy(), vel=batch["vel"][order].copy())
            g = _gpu(b, k)
            goal = torch.from_numpy(np.ascontiguousarray(batch["goal"][order])).cuda()
            for _ in range(STEPS):
                g.env_step(policy=_lib.POLICY_GOAL, goal=goal)
            inv = np.argsort(order)
            results.append((tpb, g.pos.cpu().numpy()[inv], g.vel.cpu().numpy()[inv], g.read_stats()["lp3_calls"]))
    _, p0, v0, l0 = results[0]
    for tpb, p, v, l in results[1:]:
        assert p.tobytes() == p0.tobytes() and v.tobytes() == v0.tobytes() and l == l0, tpb
