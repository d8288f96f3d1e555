"""Scenario generators: initial positions, initial velocities, two-stage goals and obstacle
polygons for a batch of worlds.

Each generator follows the geometry of the reference's ``_init_world_*`` method (file:line in
the docstrings) in float64 and returns float32 arrays ``[E, N, 2]``; the reference's unseeded
``random.uniform`` calls (SURVEY Q11) are replaced by a seeded ``numpy`` generator.  Obstacle
polygons keep the reference's vertex order (clockwise enclosing wall, SURVEY Q6).

``reference_rng=True`` draws from Python's ``random.Random(seed + env)`` in exactly the order the
reference's generator calls ``random.uniform``: world ``e`` of the batch then equals, bit for
bit, what the reference builds after ``random.seed(seed + e)`` (pinned against the unmodified
reference in tests/golden/shell_scenarios.json, tests/test_shell_golden.py).
"""
from __future__ import annotations

import random as _pyrandom
from dataclasses import dataclass, field
from math import cos, pi, sin, sqrt
from typing import List, Optional

import numpy as np

# ORCA constants shared by every ALAN scenario (ALAN_true.py:15-20, addAgent :461-468)
ALAN_PARAMS = dict(timeStep=1 / 60., neighborDist=5.0, maxNeighbors=10, timeHorizon=1.5, timeHorizonObst=1.5,
                   radius=0.5, maxSpeed=1.0)
# ... and by the gym env (collision_avoidence_env.py:27-33, addAgent :126-133)
ENV_PARAMS = dict(timeStep=1 / 60., neighborDist=1.5, maxNeighbors=5, timeHorizon=1.5, timeHorizonObst=1.5,
                  radius=0.5, maxSpeed=1.0)


@dataclass
class Scenario:
    name: str
    pos: np.ndarray          # [E, N, 2] float32
    vel: np.ndarray          # [E, N, 2] float32 initial velocity = random unit vector (SURVEY Q2)
    goal: np.ndarray         # [E, N, 2] float32 first goal
    goal2: np.ndarray        # [E, N, 2] float32 goal taken after arrival
    envsize: float
    obstacles: List = field(default_factory=list)   # shared polygons, or per-env lists when per_env
    per_env_obstacles: bool = False
    params: dict = field(default_factory=lambda: dict(ALAN_PARAMS))

    @property
    def num_envs(self):
        return self.pos.shape[0]

    @property
    def agents_per_env(self):
        return self.pos.shape[1]


def _unit_vels(rng, E, N):
    ang = rng.uniform(0.0, 2 * pi, size=(E, N))
    return np.stack([np.cos(ang), np.sin(ang)], -1)


def _reference_draws(seed, num_envs, num_agents, agent_spec, tail_spec=()):
    """Per-world draws in the reference's call order: for every agent the ``agent_spec`` fields
    (each a (lo, hi) of one ``random.uniform`` call), then the ``tail_spec`` fields once.
    ``seed`` may also be a list of ``random.Random`` objects (one per world) to continue their
    streams.  Returns (agents[E, N, F], tail[E, T]) float64."""
    agents = np.zeros((num_envs, num_agents, len(agent_spec)))
    tail = np.zeros((num_envs, len(tail_spec)))
    for e in range(num_envs):
        r = seed[e] if isinstance(seed, (list, tuple)) else _pyrandom.Random(seed + e)
        for i in range(num_agents):
            for f, (lo, hi) in enumerate(agent_spec):
                agents[e, i, f] = r.uniform(lo, hi)
        for t, (lo, hi) in enumerate(tail_spec):
            tail[e, t] = r.uniform(lo, hi)
    return agents, tail


def _vels_from_angles(ang):
    """(cos, sin) with math.cos / math.sin, as the reference computes them (ALAN_true.py:182-183)."""
    out = np.zeros(ang.shape + (2,))
    it = np.nditer(ang, flags=["multi_index"])
    for a in it:
        out[it.multi_index] = (cos(float(a)), sin(float(a)))
    return out


def _wall(lo, hi_x, hi_y=None):
    """Enclosing wall in the reference's clockwise order: (x0,0) (x0,S) (x1,S) (x1,0)."""
    hi_y = hi_x if hi_y is None else hi_y
    return [(lo, 0.0), (lo, hi_y), (hi_x, hi_y), (hi_x, 0.0)]


def _f32(*arrs):
    return [np.ascontiguousarray(a, dtype=np.float32) for a in arrs]


def circle(num_envs: int, num_agents: int, seed: int = 0, radius: float = 0.5, rotate: bool = True,
           reference_rng: bool = False) -> Scenario:
    """ALAN_true.py:297-330 ``_init_world_circle``: agents evenly on a circle, antipodal goals.

    ``rotate`` adds a per-env random rotation of the whole ring so that the envs of a batch are
    not copies of each other (SURVEY 8d, config 2)."""
    rng = np.random.default_rng(seed)
    circumference = radius * 3 * num_agents
    R = circumference / (2 * pi)
    envsize = 2 * R + 4 * radius
    c = envsize / 2
    if reference_rng:  # theta accumulates (:322), math.cos / math.sin
        ang, _ = _reference_draws(seed, num_envs, num_agents, [(0, 2 * pi)])
        vel = _vels_from_angles(ang[..., 0])
        theta, th = np.zeros(num_agents), 0
        for i in range(num_agents):
            theta[i] = th
            th += (2 * pi) / num_agents
        pos = np.broadcast_to(c + R * _vels_from_angles(theta), (num_envs, num_agents, 2))
        goal = np.broadcast_to(c + R * _vels_from_angles(theta + pi), (num_envs, num_agents, 2))
        pos, vel, goal = _f32(pos, vel, goal)
        return Scenario("circle", pos, vel, goal, goal.copy(), envsize, [_wall(0.0, envsize)])
    theta = np.arange(num_agents) * ((2 * pi) / num_agents)
    theta = theta[None, :] + (rng.uniform(0, 2 * pi, size=(num_envs, 1)) if rotate else np.zeros((num_envs, 1)))
    pos = np.stack([c + R * np.cos(theta), c + R * np.sin(theta)], -1)
    goal = np.stack([c + R * np.cos(theta + pi), c + R * np.sin(theta + pi)], -1)
    vel = _unit_vels(rng, num_envs, num_agents)
    pos, vel, goal = _f32(pos, vel, goal)
    return Scenario("circle", pos, vel, goal, goal.copy(), envsize, [_wall(0.0, envsize)])


def crowd(num_envs: int, num_agents: int, seed: int = 0, radius: float = 0.5, blocks: int = 0,
          reference_rng: bool = False) -> Scenario:
    """ALAN_true.py:270-294 ``_init_world_crowd``: uniform random starts and goals in a square of
    side 2*sqrt(2 r N).  ``blocks`` > 0 adds that many square blocks per env placed with the
    ``_init_world_blocks`` recipe (ALAN_true.py:363-372) -- BASELINE config 4."""
    rng = np.random.default_rng(seed)
    envsize = sqrt(2 * radius * num_agents) * 2
    if reference_rng:  # per agent: x, y, angle, target x, target y (:275-282)
        if blocks:
            raise ValueError("the reference's crowd has no blocks; reference_rng needs blocks=0")
        d, _ = _reference_draws(seed, num_envs, num_agents, [(0, envsize), (0, envsize), (0, 2 * pi), (0, envsize),
                                                             (0, envsize)])
        pos, vel, goal = d[..., 0:2], _vels_from_angles(d[..., 2]), d[..., 3:5]
    else:
        pos = rng.uniform(0, envsize, size=(num_envs, num_agents, 2))
        goal = rng.uniform(0, envsize, size=(num_envs, num_agents, 2))
        vel = _unit_vels(rng, num_envs, num_agents)
    pos, vel, goal = _f32(pos, vel, goal)
    wall = _wall(0.0, envsize)
    if blocks <= 0:
        return Scenario("crowd", pos, vel, goal, goal.copy(), envsize, [wall])
    bs = envsize / (blocks * 2)
    worlds = []
    for _ in range(num_envs):
        polys = [wall]
        for _b in range(blocks):
            cx, cy = rng.uniform(bs, envsize - bs), rng.uniform(0, envsize)
            polys.append([(cx - bs / 2, cy - bs / 2), (cx + bs / 2, cy - bs / 2),
                          (cx + bs / 2, cy + bs / 2), (cx - bs / 2, cy + bs / 2)])
        worlds.append(polys)
    return Scenario("crowd_blocks", pos, vel, goal, goal.copy(), envsize, worlds, per_env_obstacles=True)


def blocks(num_envs: int, num_agents: int, seed: int = 0, radius: float = 0.5, reference_rng: bool = False) -> Scenario:
    """ALAN_true.py:332-374 ``_init_world_blocks``: a column of agents crossing a field of 4 blocks."""
    rng = np.random.default_rng(seed)
    envsize = 3 * radius * num_agents
    y = np.cumsum([1.5 * radius] + [3 * radius] * (num_agents - 1))  # y_pos += y_inc (:354)
    pos = np.broadcast_to(np.stack([np.full(num_agents, 1.5 * radius), y], -1), (num_envs, num_agents, 2))
    goal = np.broadcast_to(np.stack([np.full(num_agents, envsize - 1.5 * radius), y], -1), (num_envs, num_agents, 2))
    wall = _wall(0.0, envsize)
    nb = 4
    bs = envsize / (nb * 2)
    if reference_rng:  # per agent: angle; then per block: centre x, centre y (:341-367)
        ang, centres = _reference_draws(seed, num_envs, num_agents, [(0, 2 * pi)], [(bs, envsize - bs), (0, envsize)] * nb)
        vel = _vels_from_angles(ang[..., 0])
    else:
        vel = _unit_vels(rng, num_envs, num_agents)
    worlds = []
    for e in range(num_envs):
        polys = [wall]
        for _b in range(nb):
            if reference_rng:
                cx, cy = centres[e, 2 * _b], centres[e, 2 * _b + 1]
            else:
                cx, cy = rng.uniform(bs, envsize - bs), rng.uniform(0, envsize)
            polys.append([(cx - bs / 2, cy - bs / 2), (cx + bs / 2, cy - bs / 2),
                          (cx + bs / 2, cy + bs / 2), (cx - bs / 2, cy + bs / 2)])
        worlds.append(polys)
    pos, vel, goal = _f32(pos, vel, goal)
    return Scenario("blocks", pos, vel, goal, goal.copy(), envsize, worlds, per_env_obstacles=True)


def congested(num_envs: int, num_agents: int, seed: int = 0, radius: float = 0.5, reference_rng: bool = False) -> Scenario:
    """ALAN_true.py:175-210 ``_init_world_congested``: a crowd squeezing through a 2.5 r doorway."""
    rng = np.random.default_rng(seed)
    S = sqrt(2 * radius * num_agents) * 3
    if reference_rng:  # per agent: x, y, angle (:180-182)
        d, _ = _reference_draws(seed, num_envs, num_agents, [(S * 0.2, S), (0, S), (0, 2 * pi)])
        pos, vel = d[..., 0:2], _vels_from_angles(d[..., 2])
    else:
        pos = np.stack([rng.uniform(S * 0.2, S, size=(num_envs, num_agents)),
                        rng.uniform(0, S, size=(num_envs, num_agents))], -1)
        vel = _unit_vels(rng, num_envs, num_agents)
    goal = np.broadcast_to(np.array([0.1 * S - 1.0, S / 2]), (num_envs, num_agents, 2))
    goal2 = np.broadcast_to(np.array([0.1 * S - S, S / 2]), (num_envs, num_agents, 2))
    polys = [
        [(-S, 0.0), (-S, S), (S, S), (S, 0.0)],
        [(0.1 * S, 0.0), (0.1 * S + 0.5, 0.0), (0.1 * S + 0.5, S / 2 - 1.25 * radius), (0.1 * S, S / 2 - 1.25 * radius)],
        [(0.1 * S, S / 2 + 1.25 * radius), (0.1 * S + 0.5, S / 2 + 1.25 * radius), (0.1 * S + 0.5, S), (0.1 * S, S)],
    ]
    pos, vel, goal, goal2 = _f32(pos, vel, goal, goal2)
    return Scenario("congested", pos, vel, goal, goal2, S, polys)


def incoming(num_envs: int, num_agents: int, seed: int = 0, radius: float = 0.5, reference_rng: bool = False) -> Scenario:
    """ALAN_true.py:212-267 ``_init_world_incoming``: one agent against an oncoming block."""
    rng = np.random.default_rng(seed)
    S = sqrt(2 * radius * num_agents) * 10
    p = [(0.1 * S, S / 2)]
    g = [(0.9 * S, S / 2)]
    n_in = num_agents - 1
    block_len = sqrt(n_in)
    x_inc, y_inc = 3 * radius, 2.1 * radius
    y_start = S / 2 - ((y_inc * block_len) / 2)
    x_pos, y_pos = 0.8 * S, y_start
    for _ in range(n_in):
        p.append((x_pos, y_pos))
        g.append((x_pos - 0.7 * S, y_pos))
        y_pos += y_inc
        if y_pos > y_start + y_inc * block_len:
            x_pos += x_inc
            y_pos = y_start
    pos = np.broadcast_to(np.asarray(p), (num_envs, num_agents, 2))
    goal = np.broadcast_to(np.asarray(g), (num_envs, num_agents, 2))
    if reference_rng:  # one angle per agent, in agent order (:220,243)
        vel = _vels_from_angles(_reference_draws(seed, num_envs, num_agents, [(0, 2 * pi)])[0][..., 0])
    else:
        vel = _unit_vels(rng, num_envs, num_agents)
    pos, vel, goal = _f32(pos, vel, goal)
    return Scenario("incoming", pos, vel, goal, goal.copy(), S, [_wall(0.0, S)])


def deadlock(num_envs: int, num_agents: int, seed: int = 0, radius: float = 0.5, reference_rng: bool = False) -> Scenario:
    """ALAN_true.py:376-457 ``_init_world_deadlock``: two queues meeting in a one-lane tube."""
    rng = np.random.default_rng(seed)
    S = sqrt(2 * radius * num_agents) * 10
    half = int(num_agents / 2)
    p, g, g2 = [], [], []
    x = 0.2 * S
    for _ in range(half):
        p.append((x, S / 2))
        g.append((0.9 * S, S / 2))
        g2.append((0.9 * S + S, S / 2))
        x += -3 * radius
    x = 0.8 * S
    for _ in range(half, num_agents):
        p.append((x, S / 2))
        g.append((0.1 * S, S / 2))
        g2.append((0.1 * S - S, S / 2))
        x += 3 * radius
    lo, hi = S / 2 - 1.25 * radius, S / 2 + 1.25 * radius
    polys = [
        [(-S, 0.0), (-S, S), (2 * S, S), (2 * S, 0.0)],
        [(0.0, 0.0), (0.5, 0.0), (0.2 * S + 0.5, lo), (0.2 * S, lo)],
        [(0.0, S), (0.2 * S, hi), (0.2 * S + 0.5, hi), (0.5, S)],
        [(S - 0.5, 0.0), (S, 0.0), (0.8 * S, lo), (0.8 * S - 0.5, lo)],
        [(S - 0.5, S), (0.8 * S - 0.5, hi), (0.8 * S, hi), (S, S)],
        [(0.2 * S, lo - 0.5), (0.8 * S, lo - 0.5), (0.8 * S, lo), (0.2 * S, lo)],
        [(0.2 * S, hi + 0.5), (0.2 * S, hi), (0.8 * S, hi), (0.8 * S, hi + 0.5)],
    ]
    pos = np.broadcast_to(np.asarray(p), (num_envs, num_agents, 2))
    goal = np.broadcast_to(np.asarray(g), (num_envs, num_agents, 2))
    goal2 = np.broadcast_to(np.asarray(g2), (num_envs, num_agents, 2))
    if reference_rng:  # one angle per agent, in agent order (:386,403)
        vel = _vels_from_angles(_reference_draws(seed, num_envs, num_agents, [(0, 2 * pi)])[0][..., 0])
    else:
        vel = _unit_vels(rng, num_envs, num_agents)
    pos, vel, goal, goal2 = _f32(pos, vel, goal, goal2)
    return Scenario("deadlock", pos, vel, goal, goal2, S, polys)


# ORCA constants of the roadmap world below (the scale of RVO2's Blocks / Roadmap examples)
ROADMAP_PARAMS = dict(timeStep=0.25, neighborDist=15.0, maxNeighbors=10, timeHorizon=5.0, timeHorizonObst=5.0,
                      radius=2.0, maxSpeed=2.0)


def roadmap_blocks(num_envs: int, agents_per_group: int = 25, jitter: float = 0.0, seed: int = 0):
    """Four square blocks around the origin, four groups of agents in the corners crossing to the
    opposite corner, and a roadmap around the blocks -- the layout of RVO2's Blocks / Roadmap examples,
    with numbers defined here.  Roadmap vertices: the four goals first (corner targets), then one
    vertex off each block corner.  ``jitter`` > 0 moves every block, with its four roadmap vertices, by
    a uniform offset in [-jitter, jitter]^2 per env: per-env obstacles and roadmaps.

    Returns (Scenario, roadmap vertices float32 [R, 2] or [E, R, 2], goal vertex ids int32 [E, N])."""
    rng = np.random.default_rng(seed)
    goals = np.array([(-75.0, -75.0), (75.0, -75.0), (-75.0, 75.0), (75.0, 75.0)])
    # counter-clockwise squares (RVO2's obstacle orientation) and the roadmap vertices 2 units off their corners
    blocks_ = [np.array([(-10.0, 40.0), (-40.0, 40.0), (-40.0, 10.0), (-10.0, 10.0)]),
               np.array([(10.0, 40.0), (10.0, 10.0), (40.0, 10.0), (40.0, 40.0)]),
               np.array([(10.0, -40.0), (40.0, -40.0), (40.0, -10.0), (10.0, -10.0)]),
               np.array([(-10.0, -40.0), (-10.0, -10.0), (-40.0, -10.0), (-40.0, -40.0)])]
    corners = [b + 2.0 * np.sign(b - b.mean(0)) for b in blocks_]
    side = int(np.ceil(np.sqrt(agents_per_group)))
    k = np.arange(agents_per_group)
    offs = np.stack([55.0 + 10.0 * (k % side), 55.0 + 10.0 * (k // side)], -1)
    # group g starts in the corner opposite to goal g
    starts = [offs * (1, 1), offs * (-1, 1), offs * (1, -1), offs * (-1, -1)]
    pos = np.concatenate(starts)
    goal_id = np.repeat(np.arange(4, dtype=np.int32), agents_per_group)
    N = pos.shape[0]
    pos = np.broadcast_to(pos, (num_envs, N, 2))
    goal = np.broadcast_to(goals[goal_id], (num_envs, N, 2))
    vel = np.zeros((num_envs, N, 2))
    goal_vertex = np.ascontiguousarray(np.broadcast_to(goal_id, (num_envs, N)), np.int32)
    if jitter > 0.0:
        shift = rng.uniform(-jitter, jitter, size=(num_envs, 4, 1, 2))
        worlds = [[(blocks_[b] + shift[e, b]).tolist() for b in range(4)] for e in range(num_envs)]
        rm = np.concatenate([np.broadcast_to(goals, (num_envs, 4, 2))]
                            + [np.asarray(corners[b]) + shift[:, b] for b in range(4)], axis=1)
        per_env = True
    else:
        worlds = [b.tolist() for b in blocks_]
        rm = np.concatenate([goals] + corners)
        per_env = False
    pos, vel, goal = _f32(pos, vel, goal)
    scn = Scenario("roadmap_blocks", pos, vel, goal, goal.copy(), 150.0, worlds, per_env_obstacles=per_env,
                   params=dict(ROADMAP_PARAMS))
    return scn, np.ascontiguousarray(rm, np.float32), goal_vertex


def reference_streams(seed: int, num_envs: int):
    """One ``random.Random(seed + e)`` per world: the stream the reference's module-level
    ``random.uniform`` would follow after ``random.seed(seed + e)``."""
    return [_pyrandom.Random(seed + e) for e in range(num_envs)]


def default_env_reset_positions(streams, num_agents: int, envsize: float = 10.0) -> np.ndarray:
    """collision_avoidence_env.py:476-479: per agent x~U(S/2, S), y~U(0, S), continuing ``streams``."""
    d, _ = _reference_draws(streams, len(streams), num_agents, [(envsize * 0.5, envsize), (0, envsize)])
    return d.astype(np.float32)


def default_env(num_envs: int, num_agents: int = 10, seed: int = 0, reference_rng=False) -> Scenario:
    """collision_avoidence_env.py:77-123 ``_init_world``: the gym env's built-in world
    (BASELINE config 1): spawn x~U(5,10), y~U(0,10), goal (1,5), wall + two gate blocks."""
    rng = np.random.default_rng(seed)
    S = 10.0
    if reference_rng:  # per agent: x, y, angle (:88-90); a list of random.Random continues those streams
        d, _ = _reference_draws(reference_rng if isinstance(reference_rng, (list, tuple)) else seed, num_envs,
                                num_agents, [(S * 0.5, S), (0, S), (0, 2 * pi)])
        pos, vel = d[..., 0:2], _vels_from_angles(d[..., 2])
    else:
        pos = np.stack([rng.uniform(S * 0.5, S, size=(num_envs, num_agents)),
                        rng.uniform(0, S, size=(num_envs, num_agents))], -1)
        vel = _unit_vels(rng, num_envs, num_agents)
    goal = np.broadcast_to(np.array([1.0, 5.0]), (num_envs, num_agents, 2))
    goal2 = np.broadcast_to(np.array([-10.0, 5.0]), (num_envs, num_agents, 2))
    polys = [
        [(-15.0, 0.0), (-15.0, S), (S, S), (S, 0.0)],
        [(2.0, 0.0), (2.5, 0.0), (2.5, 4.4), (2.0, 4.4)],
        [(2.0, 5.6), (2.5, 5.6), (2.5, 10.0), (2.0, 10.0)],
    ]
    pos, vel, goal, goal2 = _f32(pos, vel, goal, goal2)
    return Scenario("default_env", pos, vel, goal, goal2, S, polys, params=dict(ENV_PARAMS))


GENERATORS = {"circle": circle, "crowd": crowd, "blocks": blocks, "congested": congested, "incoming": incoming,
              "deadlock": deadlock, "default_env": default_env}


def make(name: str, num_envs: int, num_agents: int, seed: int = 0, **kw) -> Scenario:
    if name not in GENERATORS:
        raise ValueError(f"{name} is not a valid scenario")  # ALAN_true.py:158
    return GENERATORS[name](num_envs, num_agents, seed=seed, **kw)
