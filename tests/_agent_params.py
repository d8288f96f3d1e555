"""Shared helpers of the per-agent parameter tests: seeded mixed parameter draws and oracle
simulators built with one addAgent(pos, nd, k, th, tho, r, vmax, vel) per agent."""
from __future__ import annotations

import numpy as np

from _common import OraclePyRVO

NAMES = ("neighbor_dist", "max_neighbors", "time_horizon", "time_horizon_obst", "radius", "max_speed")


def mixed_params(E, N, K, seed):
    """radius U(0.2, 0.8), maxSpeed U(0.5, 2), neighborDist U(1.5, 6), maxNeighbors in {0..K},
    timeHorizon and timeHorizonObst U(0.5, 3), float32 / int32 [E, N]."""
    rng = np.random.default_rng(seed)
    f = lambda lo, hi: rng.uniform(lo, hi, (E, N)).astype(np.float32)
    return dict(radius=f(0.2, 0.8), max_speed=f(0.5, 2.0), neighbor_dist=f(1.5, 6.0),
                max_neighbors=rng.integers(0, K + 1, (E, N)).astype(np.int32),
                time_horizon=f(0.5, 3.0), time_horizon_obst=f(0.5, 3.0))


def full_params(scn, ap):
    """Every one of the six arrays, the scenario's value where ap has none."""
    P = scn.params
    dflt = dict(neighbor_dist=P["neighborDist"], max_neighbors=P["maxNeighbors"], time_horizon=P["timeHorizon"],
                time_horizon_obst=P["timeHorizonObst"], radius=P["radius"], max_speed=P["maxSpeed"])
    shape = (scn.num_envs, scn.agents_per_env)
    out = {}
    for n in NAMES:
        dt = np.int32 if n == "max_neighbors" else np.float32
        out[n] = np.full(shape, dflt[n], dt) if ap.get(n) is None else np.asarray(ap[n], dt).reshape(shape)
    return out


def oracle_sims_per_agent(scn, ap, pos=None, vel=None):
    """One oracle simulator per env, every agent added with its own parameters."""
    P = scn.params
    full = full_params(scn, ap)
    pos = scn.pos if pos is None else pos
    vel = scn.vel if vel is None else vel
    sims = []
    for e in range(scn.num_envs):
        s = OraclePyRVO(P["timeStep"], P["neighborDist"], P["maxNeighbors"], P["timeHorizon"], P["timeHorizonObst"],
                        P["radius"], P["maxSpeed"])
        for i in range(scn.agents_per_env):
            s.addAgent(tuple(map(float, pos[e, i])), float(full["neighbor_dist"][e, i]), int(full["max_neighbors"][e, i]),
                       float(full["time_horizon"][e, i]), float(full["time_horizon_obst"][e, i]),
                       float(full["radius"][e, i]), float(full["max_speed"][e, i]), tuple(map(float, vel[e, i])))
        polys = scn.obstacles[e] if scn.per_env_obstacles else scn.obstacles
        for poly in polys:
            s.addObstacle([tuple(map(float, v)) for v in poly])
        s.processObstacles()
        sims.append(s)
    return sims


def max_obstacle_range(scn, ap):
    """The largest timeHorizonObst * maxSpeed + radius (float32) among the agents."""
    full = full_params(scn, ap)
    return float((full["time_horizon_obst"] * full["max_speed"] + full["radius"]).max())
