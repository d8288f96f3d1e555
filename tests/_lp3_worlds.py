"""Constructed jam worlds for the LP3 tests, characterised with the oracle, and the block assembler.

Every env is a box of side BOX inside one clockwise enclosing wall (4 processed vertices, so the
slim K + 2 tile kernel stays eligible) holding N agents of radius R:

* jam:     a jittered hexagonal pack at spacing U(1.5 R, 1.9 R) around the box centre, velocities
           toward the centroid, goals outward or at the antipode.  Neighbors overlap, so every
           agent of the pack fails LP2 (RVO2's collision half-planes lie far outside the speed disc).
* walled:  the same pack pressed against the wall x = 0: the obstacle lines stay hard in LP3 and
           LP3's projected programmes become infeasible.
* queue:   rows at exactly y = c with distinct spacings below 2 R and velocities along the row: the
           agent lines of a row are exactly parallel or antiparallel (det = 0, both branches of
           LP3's projection).
* pinch:   one agent between two others closing in on it: exactly one LP3 agent.
* free:    agents on a jittered lattice of side SITE: no LP3.

An env with c LP3 agents is a pack (or queue) of c agents -- or a pinch for c = 1 -- plus N - c free
agents.  ``characterise`` runs the oracle: an agent needs LP3 when LP2 fails on its ORCA lines,
``solve_lp(orca_lines(i), ...)`` returns a fail index below the line count.
"""
from __future__ import annotations

import functools

import numpy as np

from collision_avoidance_b200 import scenarios
from oracle.rvo2_oracle import PyRVOSimulator, solve_lp

R = 0.5
BOX = 80.0
SITE = 4.0
CENTRE = np.array([BOX / 2, BOX / 2])
WALL = [(0.0, 0.0), (0.0, BOX), (BOX, BOX), (BOX, 0.0)]
KINDS = ("jam", "walled", "queue")


def params(k):
    """The ALAN shells' ORCA parameters with maxNeighbors = k."""
    return dict(timeStep=1 / 60., neighborDist=5.0, maxNeighbors=int(k), timeHorizon=1.5, timeHorizonObst=1.5,
                radius=R, maxSpeed=1.0)


def goal_dir(pos, goal):
    """The step kernel's goal-directed preferred velocity (orca_core.cuh goal_direction) in float32:
    unit(goal - pos) with one rounding per operation, (1, 0) at the goal."""
    d = (goal.astype(np.float32) - pos.astype(np.float32)).astype(np.float32)
    n2 = d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]
    with np.errstate(divide="ignore"):
        inv = np.float32(1.0) / np.sqrt(n2)
    out = np.stack([d[..., 0] * inv, d[..., 1] * inv], -1).astype(np.float32)
    out[n2 == 0] = (1.0, 0.0)
    return out


# ---------------------------------------------------------------------------------------- parts
def _hex_pack(m, rng):
    s = rng.uniform(1.5 * R, 1.9 * R)
    M = int(np.sqrt(m)) + 3
    i, j = np.meshgrid(np.arange(-M, M + 1), np.arange(-M, M + 1))
    pts = np.stack([i + 0.5 * j, j * np.sqrt(3) / 2], -1).reshape(-1, 2) * s
    order = np.argsort(np.hypot(pts[:, 0], pts[:, 1]) + rng.uniform(0, 1e-3, len(pts)))
    pts = pts[order[:m]] + rng.uniform(-0.03, 0.03, (m, 2)) * s
    return pts


def _jam(m, rng, walled):
    pts = _hex_pack(m, rng)
    if walled:  # leftmost agents 0.55 .. 0.75 from the wall x = 0
        c = np.array([0.55 + rng.uniform(0, 0.2) - pts[:, 0].min(), BOX / 2])
    else:
        c = CENTRE + rng.uniform(-1, 1, 2)
    pos = pts + c
    cen = pos.mean(0)
    d = cen - pos
    n = np.maximum(np.hypot(d[:, 0], d[:, 1]), 1e-6)[:, None]
    vel = d / n * rng.uniform(0.2, 1.0, (m, 1))
    if rng.random() < 0.5:
        goal = pos + (pos - cen) / n * 10.0        # outward
    else:
        goal = 2 * cen - pos                        # the antipode
    return pos, vel, goal, c, np.abs(pts).max() + 1.0


def _queue(m, rng):
    """Rows of 2 to 16 agents at y = c exactly, spacings distinct and below 2 R, one velocity."""
    rows = (m + 15) // 16
    pos = []
    for r, cnt in enumerate(len(a) for a in np.array_split(np.arange(m), rows)):
        gaps = rng.uniform(1.5 * R, 1.9 * R, cnt - 1)
        xs = BOX / 2 - 7.0 + rng.uniform(0, 0.5) + np.concatenate([[0.0], np.cumsum(gaps)])
        y = np.float32(BOX / 2 - 2.5 * (rows - 1) / 2 + 2.5 * r)
        pos.append(np.stack([xs, np.full(cnt, y)], -1))
    pos = np.concatenate(pos)
    # velocities along the rows (y = 0 exactly): every relative velocity and relative position of two
    # agents of a row has y = 0, so their lines are exactly parallel or antiparallel.  The speeds differ,
    # so that a farther neighbor on one side can be violated more than a nearer one: only then does an
    # LP3 round at its line meet an earlier line of the same direction (skipped).
    vel = np.stack([rng.uniform(-1.0, 1.0, len(pos)), np.zeros(len(pos))], -1)
    goal = pos + np.array([rng.choice([-10.0, 10.0]), 0.0])
    c = np.array([BOX / 2, BOX / 2])
    return pos, vel, goal, c, np.hypot(7.5, 1.25 * rows) + 1.0


def _pinch(rng):
    d = rng.uniform(1.03, 1.12)
    sp = rng.uniform(0.8, 1.0, 2)
    c = CENTRE + rng.uniform(-1, 1, 2)
    pos = np.array([c, c + (d, 0.0), c - (d, 0.0)])
    vel = np.array([(0.0, 0.0), (-sp[0], 0.0), (sp[1], 0.0)])
    goal = pos + rng.uniform(-10, 10, (3, 2))
    return pos, vel, goal, c, 3.0


def _free(m, rng, centre, keep_out):
    g = np.arange(SITE, BOX - SITE + 1e-9, SITE)
    sites = np.stack(np.meshgrid(g, g), -1).reshape(-1, 2)
    far = np.hypot(*(sites - centre).T) > keep_out + 2.5
    sites = sites[far]
    assert len(sites) >= m, (len(sites), m)
    sites = sites[rng.permutation(len(sites))[:m]]
    pos = sites + rng.uniform(-0.4, 0.4, sites.shape)
    ang = rng.uniform(0, 2 * np.pi, m)
    vel = np.stack([np.cos(ang), np.sin(ang)], -1) * rng.uniform(0, 0.5, (m, 1))
    goal = rng.uniform(SITE, BOX - SITE, (m, 2))
    return pos, vel, goal


def compose(N, c, kind, seed):
    """pos, vel, goal (float32 [N, 2]) of an env meant to hold c LP3 agents of the given kind."""
    rng = np.random.default_rng(seed)
    if c == 0:
        parts = [(np.zeros((0, 2)),) * 3]
        centre, keep = CENTRE, 0.0
    else:
        if c == 1:
            p, v, g, centre, keep = _pinch(rng)
        elif kind == "queue":
            p, v, g, centre, keep = _queue(c, rng)
        else:
            p, v, g, centre, keep = _jam(c, rng, kind == "walled")
        parts = [(p, v, g)]
    parts.append(_free(N - len(parts[0][0]), rng, centre, keep))
    pos, vel, goal = (np.concatenate([q[i] for q in parts]).astype(np.float32) for i in range(3))
    perm = rng.permutation(N)                       # LP3 agents scattered over the env's warps
    return pos[perm], vel[perm], goal[perm]


# ---------------------------------------------------------------------------------------- oracle
def oracle_sim(P, pos, vel, agent_params=None):
    """One oracle simulator of an env; agent_params: per-agent dict of [N] arrays (the six names of
    _agent_params.NAMES) or None for the handle's values."""
    s = PyRVOSimulator(P["timeStep"], P["neighborDist"], P["maxNeighbors"], P["timeHorizon"], P["timeHorizonObst"],
                       P["radius"], P["maxSpeed"])
    for i in range(len(pos)):
        if agent_params is None:
            a = (P["neighborDist"], P["maxNeighbors"], P["timeHorizon"], P["timeHorizonObst"], P["radius"], P["maxSpeed"])
        else:
            ap = agent_params
            a = (float(ap["neighbor_dist"][i]), int(ap["max_neighbors"][i]), float(ap["time_horizon"][i]),
                 float(ap["time_horizon_obst"][i]), float(ap["radius"][i]), float(ap["max_speed"][i]))
        s.addAgent(tuple(map(float, pos[i])), *a, tuple(map(float, vel[i])))
    s.addObstacle(WALL)
    s.processObstacles()
    return s


def lp3_agents(sim, pref, vmax):
    """After sim.doStep(): bool [N], which agents' LP2 failed; and their programmes
    [(lines, n_obst, vmax, pref)] for every agent."""
    N = sim.getNumAgents()
    need = np.zeros(N, bool)
    progs = []
    for i in range(N):
        lines, n_obst = sim.orca_lines(i)
        vm = float(np.broadcast_to(vmax, (N,))[i])
        fail, _ = solve_lp(lines, n_obst, vm, pref[i])
        need[i] = fail < len(lines)
        progs.append((lines, int(n_obst), vm, pref[i].copy()))
    return need, progs


def has_tie(pos, nd):
    """Does some agent have two others within neighborDist at bit-equal float32 squared distance?"""
    p = pos.astype(np.float32)
    nd_sq = np.float32(nd) * np.float32(nd)
    for i in range(len(p)):
        d = (p - p[i]).astype(np.float32)
        dsq = d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]
        dsq = np.delete(dsq, i)
        dsq = dsq[dsq < nd_sq]
        if len(np.unique(dsq)) < len(dsq):
            return True
    return False


@functools.lru_cache(maxsize=None)
def env(N, c, kind, k, seed):
    """A tie-free env with exactly c LP3 agents at its first step (the oracle's count), for
    maxNeighbors k.  Returns (pos, vel, goal, need[N], programmes)."""
    P = params(k)
    for attempt in range(40):
        pos, vel, goal = compose(N, c, kind, seed * 1000 + attempt)
        if has_tie(pos, P["neighborDist"]):
            continue
        sim = oracle_sim(P, pos, vel)
        pref = goal_dir(pos, goal)
        sim.set_pref_velocities(pref)
        sim.doStep()
        need, progs = lp3_agents(sim, pref, P["maxSpeed"])
        if need.sum() == c:
            return pos, vel, goal, need, progs
    raise AssertionError(f"no tie-free {kind} env of {N} agents with {c} LP3 agents (k={k})")


# ---------------------------------------------------------------------------------------- blocks
def block_targets(N, tpb):
    """Per-block LP3 totals at the boundaries of block_lp3 for blocks of tpb threads holding
    epb = tpb // N envs: nfree = tpb - total columns are dead, nstored = min(total, nfree) solvers
    store their programme, cut to whole warps when total > nfree.  0, 1 (a lone solver), 31/32/33
    (one warp, and one lane past it), tpb/2 - 1 .. tpb/2 + 1 (dead columns run out), 5/8 and 7/8 of
    tpb (stored and recomputing warps side by side), tpb - 1 (nstored = 0) and epb * N (every agent of
    the block; = tpb, every column busy, when whole envs fill the block) -- those a block of epb * N
    agents can hold."""
    cap = (tpb // N) * N
    h = tpb // 2
    t = {0, 1, 31, 32, 33, h - 1, h, h + 1, 5 * tpb // 8, 7 * tpb // 8, tpb - 1, cap}
    return sorted(x for x in t if 0 <= x <= cap)


def split_total(total, epb, N, rng):
    """epb per-env LP3 counts (each 0..N) summing to total, in shuffled order."""
    counts = [min(N, max(0, total - N * j)) for j in range(epb)]
    assert sum(counts) == total
    return [counts[j] for j in rng.permutation(epb)]


def nstored(total, tpb):
    """The number of block_lp3 solvers that store their projected programme (the rest recompute)."""
    nfree = tpb - total
    ns = min(total, nfree)
    return ns & ~31 if ns < total else ns


@functools.lru_cache(maxsize=None)
def assemble(N, tpb, k, seed=0, kinds=KINDS):
    """A batch whose tile-kernel blocks (tpb threads, epb = tpb // N whole envs each, envs
    [b * epb, (b + 1) * epb) in block b) have the LP3 totals of block_targets, one block per
    target.  Returns dict(pos, vel, goal [E, N, 2] float32, need [E, N], totals [blocks],
    targets, epb, progs: per env the oracle programmes of the first step).  The totals are the
    oracle's counts, asserted here."""
    epb = tpb // N
    rng = np.random.default_rng(seed + 7919 * N + 31 * tpb + k)
    targets = block_targets(N, tpb)
    pos, vel, goal, need, progs = [], [], [], [], []
    e = 0
    for t in targets:
        for c in split_total(t, epb, N, rng):
            kind = kinds[e % len(kinds)]
            p, v, g, nd, pr = env(N, c, kind, k, int(rng.integers(1 << 30)) if c else e % 7)
            pos.append(p)
            vel.append(v)
            goal.append(g)
            need.append(nd)
            progs.append(pr)
            e += 1
    need = np.stack(need)
    totals = need.reshape(len(targets), epb * N).sum(1)
    assert list(totals) == targets, (N, tpb, k, list(totals), targets)
    return dict(pos=np.stack(pos), vel=np.stack(vel), goal=np.stack(goal), need=need, totals=totals,
                targets=targets, epb=epb, progs=progs)


def scenario(batch, k):
    """The batch as a scenarios.Scenario (shared 4-vertex wall)."""
    return scenarios.Scenario("lp3_jam", batch["pos"].copy(), batch["vel"].copy(), batch["goal"].copy(),
                              batch["goal"].copy(), BOX, [list(WALL)], params=params(k))


# ---------------------------------------------------------------------------------------- programmes
KEPS = np.float32(1e-5)  # RVO_EPSILON, the parallel test of LP1 and of LP3's projection


def _unit(a):
    return np.array([np.cos(a), np.sin(a)], np.float32)


def _prog(lines, n_obst, vmax, pref):
    return (np.ascontiguousarray(lines, np.float32).reshape(-1, 4), int(n_obst), float(np.float32(vmax)),
            np.asarray(pref, np.float32))


def synthetic_programmes(seed=0):
    """LP programmes (lines [n, 4], n_obst, vmax, pref) at LP3's edges:
    * near-parallel partners of an axis-aligned line, so that det is exactly 0, +-kEps, or one ulp on
      either side of kEps, pointing the same way (skipped) or the opposite way (midpoint);
    * exact duplicates of lines;
    * obstacle lines that are infeasible among themselves (every LP3 round fails, and LP2 may
      fail on an obstacle line);
    * random programmes of n = 1 .. 22 lines (K = 16 agent lines + 6 obstacle lines), preferred
      velocities inside and outside the speed circle."""
    rng = np.random.default_rng(seed)
    out = []
    up = np.nextafter(KEPS, np.float32(1))
    dn = np.nextafter(KEPS, np.float32(0))
    axes = [np.array(a, np.float32) for a in ((1, 0), (0, 1), (-1, 0), (0, -1))]
    for y in (np.float32(0), KEPS, -KEPS, up, -up, dn, -dn):
        for ax in axes:
            perp = np.array([-ax[1], ax[0]], np.float32)         # det(ax, s * ax + y * perp) = y exactly
            for s in (np.float32(1), np.float32(-1)):
                for trial in range(3):
                    vmax = rng.uniform(0.5, 2.0)
                    # line i: wants the velocity well to its left (outside the disc) ...
                    pi = perp * np.float32(rng.uniform(1.2, 3.0) * vmax) + ax * np.float32(rng.uniform(-1, 1))
                    dj = (s * ax + y * perp).astype(np.float32)
                    pj = (perp * np.float32(rng.uniform(-2, 2) * vmax) + ax * np.float32(rng.uniform(-1, 1))).astype(np.float32)
                    # ... behind a random line or two, then the near-parallel partner j, then line i
                    pre = []
                    for q in range(rng.integers(0, 3)):
                        d = _unit(rng.uniform(0, 2 * np.pi))
                        pre.append([*(rng.uniform(-1, 1, 2) * vmax), *d])
                    lines = pre + [[*pj, *dj], [*(pi.astype(np.float32)), *ax]]
                    if trial == 2:                               # and a later copy of line i
                        lines.append(list(lines[-1]))
                    n_obst = int(rng.integers(0, len(pre) + 1))
                    pref = _unit(rng.uniform(0, 2 * np.pi)) * np.float32(rng.choice([0.5, 1.5]) * vmax)
                    out.append(_prog(lines, n_obst, vmax, pref))
    for t in range(60):                                          # obstacle lines infeasible among themselves
        vmax = rng.uniform(0.5, 2.0)
        a = rng.uniform(0, 2 * np.pi)
        d = _unit(a)
        nrm = np.array([-d[1], d[0]], np.float32)
        gap = np.float32(rng.uniform(0.1, 1.0) * vmax)
        obst = [[*(nrm * gap), *d], [*(-nrm * gap), *(-d)]]    # y' >= gap and y' <= -gap
        if t % 3 == 0:
            obst.append([*(rng.uniform(-1, 1, 2) * vmax), *_unit(rng.uniform(0, 2 * np.pi))])
        agents = []
        for q in range(rng.integers(1, 8)):
            agents.append([*(_unit(rng.uniform(0, 2 * np.pi)) * np.float32(rng.uniform(0.5, 3) * vmax)),
                           *_unit(rng.uniform(0, 2 * np.pi))])
        lines = obst + agents if t % 2 == 0 else agents[:1] + obst + agents[1:]
        n_obst = len(obst) if t % 2 == 0 else len(obst) + 1
        out.append(_prog(lines, n_obst, vmax, _unit(rng.uniform(0, 2 * np.pi)) * np.float32(vmax * 0.8)))
    for n in range(1, 23):                                       # random programmes, every length
        for t in range(40):
            vmax = rng.uniform(0.3, 3.0)
            n_obst = int(rng.integers(0, min(n, 6) + 1))
            ang = rng.uniform(0, 2 * np.pi, n)
            lines = np.concatenate([rng.uniform(-2, 2, (n, 2)) * vmax, np.stack([np.cos(ang), np.sin(ang)], -1)], 1)
            if n > 2 and t % 4 == 0:
                lines[rng.integers(1, n)] = lines[rng.integers(0, n - 1)]   # a duplicate
            pref = _unit(rng.uniform(0, 2 * np.pi)) * np.float32(vmax * rng.choice([0.3, 0.99, 1.0, 2.0]))
            out.append(_prog(lines, n_obst, vmax, pref))
    return out


def library_programmes(k_values=(5, 10, 16)):
    """Every agent's programme of the first step of assembled batches and of a batch with per-agent
    parameters: (lines, n_obst, vmax, pref), LP3 agents and others."""
    out = []
    for k in k_values:
        for N, tpb in ((16, 256), (32, 128), (100, 256), (256, 256)):
            for progs in assemble(N, tpb, k)["progs"]:
                out.extend(_prog(*p) for p in progs)
    for progs in hetero_batch(32, 256, 10)["progs"]:
        out.extend(_prog(*p) for p in progs)
    return out


# ---------------------------------------------------------------------------------------- per-agent parameters
def hetero_batch(N, tpb, k, seed=0):
    """An assembled batch with per-agent maxSpeed U(0.3, 3) and radius U(0.45, 0.6), and in every env
    with three free agents to spare a parallel trio instead of them: A, then B 0.8 to its right with
    radius 0.2 (apart from A, on its cut-off circle), then C 1.0 to its right with radius 0.6
    (overlapping A), all at one y and moving along x.  A's lines of B and C are exactly parallel and
    point the same way, and C's is violated more: LP3's round at C skips B's line, which a world of
    one radius never produces (there the nearer neighbor's line is always the more violated one).
    Returns the batch dict of ``assemble`` with ``agent_params`` ([E, N] arrays, _agent_params.NAMES)
    and the oracle's ``need`` and ``progs`` of the first step recomputed with them."""
    b = dict(assemble(N, tpb, k, seed))
    rng = np.random.default_rng(seed + 17)
    E = b["pos"].shape[0]
    pos, vel, goal = b["pos"].copy(), b["vel"].copy(), b["goal"].copy()
    radius = rng.uniform(0.45, 0.6, (E, N)).astype(np.float32)
    vmax = rng.uniform(0.3, 3.0, (E, N)).astype(np.float32)
    for e in range(E):
        free = np.flatnonzero(~b["need"][e])
        if len(free) < 4:
            continue
        a, bb, c = free[:3]
        y = np.float32(pos[e, a, 1])
        pos[e, [a, bb, c]] = [(pos[e, a, 0], y), (pos[e, a, 0] + 0.8, y), (pos[e, a, 0] + 1.0, y)]
        vel[e, [a, bb, c]] = [(0.0, 0.0), (rng.uniform(-0.3, 0.3), 0.0), (rng.uniform(-1, 1), 0.0)]
        radius[e, [a, bb, c]] = (0.5, 0.2, 0.6)
    ap = dict(neighbor_dist=np.full((E, N), 5.0, np.float32), max_neighbors=np.full((E, N), k, np.int32),
              time_horizon=np.full((E, N), 1.5, np.float32), time_horizon_obst=np.full((E, N), 1.5, np.float32),
              radius=radius, max_speed=vmax)
    P = params(k)
    need, progs = [], []
    for e in range(E):
        assert not has_tie(pos[e], P["neighborDist"]), e
        sim = oracle_sim(P, pos[e], vel[e], {n: v[e] for n, v in ap.items()})
        pref = goal_dir(pos[e], goal[e])
        sim.set_pref_velocities(pref)
        sim.doStep()
        nd, pr = lp3_agents(sim, pref, vmax[e])
        need.append(nd)
        progs.append(pr)
    b.update(pos=pos, vel=vel, goal=goal, agent_params=ap, need=np.stack(need), progs=progs)
    return b
