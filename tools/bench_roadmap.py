#!/usr/bin/env python
"""Device-timed cost of line-of-sight queries and roadmap navigation on one GPU.

  visibility   orca_query_visibility: 16,777,216 random queries in the roadmap_blocks world (one
               shared world) and in the deadlock world held per env (4,096 envs x 4,096 queries),
               radius 2; queries per second from CUDA events around 5 launches after 2 warm-up
               launches, arms alternated, 3 repeats.
  set_roadmap  host clock around orca_set_roadmap (it synchronises): roadmap_blocks x 4,096 envs,
               shared world and per-env jitter 5.
  pref         roadmap_pref_kernel next to the step kernel it feeds, roadmap_blocks x 4,096 envs x 100
               agents (shared and jitter 5), mid-episode (after 150 roadmap-navigation steps): CUDA
               events around 50 launches of each, alternated, 3 repeats.  BSP walks per agent of
               Roadmap.cpp's index-order loop, and of a search in (cost, index) order that stops at the
               first visible candidate, are counted from the device's visibility answers at that state.
Prints the device name, power limit and max SM clock and one JSON line per measurement; writes them
to --out."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from bench_agent_params import device_info  # noqa: E402
from collision_avoidance_b200 import _lib, scenarios  # noqa: E402
from collision_avoidance_b200.sim import BatchedRVOSimulator  # noqa: E402


def events_us(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1000.0 / reps


def visibility_arms():
    rng = np.random.default_rng(0)
    dev = "cuda:0"
    arms = []
    scn, _, _ = scenarios.roadmap_blocks(1)
    sim = BatchedRVOSimulator(1, 1, device=dev, **scn.params)
    sim.set_obstacles(scn.obstacles)
    Q = 1 << 24
    q = torch.from_numpy(rng.uniform(-100, 100, (2, 1, Q, 2)).astype(np.float32)).to(dev)
    arms.append(("roadmap_blocks_shared", sim, q[0], q[1], Q))
    E, Qe = 4096, 4096
    dl = scenarios.deadlock(1, 10)
    sim2 = BatchedRVOSimulator(E, 1, device=dev, **dl.params)
    sim2.set_obstacles([dl.obstacles] * E, per_env=True)
    S = dl.envsize
    q2 = torch.from_numpy(rng.uniform((-S, 0), (2 * S, S), (2, E, Qe, 2)).astype(np.float32)).to(dev)
    arms.append(("deadlock_per_env", sim2, q2[0], q2[1], E * Qe))
    return arms


def walks_per_agent(sim, xy, dist, pos, goal_vertex, vertex, radius):
    """BSP walks per agent of Roadmap.cpp's index-order loop (the kernel's) and of a search in (cost,
    index) order, from the device's visibility answers (numpy float32 costs: the kernel's expressions,
    one rounding per operation)."""
    E, N = goal_vertex.shape
    R = xy.shape[-2]
    xy_e = np.broadcast_to(xy, (E, R, 2)) if xy.ndim == 2 else xy
    q1 = np.repeat(pos[:, :, None, :], R, axis=2).reshape(E, N * R, 2)
    q2 = np.repeat(xy_e[:, None, :, :], N, axis=1).reshape(E, N * R, 2)
    vis = sim.query_visibility(torch.from_numpy(np.ascontiguousarray(q1)).cuda(),
                               torch.from_numpy(np.ascontiguousarray(q2)).cuda(), radius).cpu().numpy().reshape(E, N, R)
    d = xy_e[:, None, :, :] - pos[:, :, None, :]
    cost = np.sqrt(d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + dist[np.arange(E)[:, None], goal_vertex]
    inf = np.float32(9e9)
    # Roadmap.cpp's loop: a walk for every vertex that would lower the running minimum
    run = np.full((E, N), inf, np.float32)
    idx_walks = np.zeros((E, N), np.int64)
    for j in range(R):
        c = cost[..., j]
        w = c < run
        idx_walks += w
        run = np.where(w & vis[..., j], c, run)
    # cost order: every candidate before the answer in (cost, index) order, and the answer
    j = np.arange(R)
    ans_cost = np.where(vertex >= 0, np.take_along_axis(cost, np.maximum(vertex, 0)[..., None], -1)[..., 0], inf)
    before = (cost < inf) & ((cost < ans_cost[..., None]) | ((cost == ans_cost[..., None]) & (j < vertex[..., None])))
    cost_walks = before.sum(-1) + (vertex >= 0)
    return float(idx_walks.mean()), float(cost_walks.mean())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "profiles",
                                                  "r04_roadmap.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_roadmap needs a CUDA device")
    gpu, power = device_info()
    print(f"device: {gpu}; power.limit, clocks.max.sm: {power}", flush=True)
    lines = []

    def emit(rec):
        rec.update(gpu=gpu, power_limit_and_max_sm_clock=power)
        print(json.dumps(rec), flush=True)
        lines.append(rec)

    arms = visibility_arms()
    for rep in range(args.repeats):
        for name, sim, q1, q2, total in arms:
            us = events_us(lambda: sim.query_visibility(q1, q2, 2.0), 2, 5)
            emit(dict(bench="visibility", arm=name, repeat=rep, queries=total, us_per_launch=round(us, 1),
                      queries_per_s=round(total / us * 1e6)))
    for _, sim, *_ in arms:
        sim.close()
    del arms
    torch.cuda.empty_cache()

    E = 4096
    for jitter in (0.0, 5.0):
        scn, xy, goal_vertex = scenarios.roadmap_blocks(E, jitter=jitter, seed=1)
        label = "per_env_jitter5" if jitter else "shared"
        sim = BatchedRVOSimulator(E, scn.agents_per_env, device="cuda:0", **scn.params)
        sim.set_obstacles(scn.obstacles, per_env=scn.per_env_obstacles)
        for rep in range(args.repeats):
            t0 = time.perf_counter()
            sim.set_roadmap(xy, 4)
            ms = (time.perf_counter() - t0) * 1e3
            emit(dict(bench="set_roadmap", arm=label, repeat=rep, envs=E, vertices=int(xy.shape[-2]), goals=4,
                      ms=round(ms, 2)))
        gv = torch.from_numpy(goal_vertex).cuda()
        sim.pos.copy_(torch.from_numpy(scn.pos))
        sim.vel.copy_(torch.from_numpy(scn.vel))
        for _ in range(150):  # mid-episode
            sim.roadmap_pref_velocity(gv)
            sim.env_step(policy=_lib.POLICY_EXTERNAL, collect_stats=False)
        pos0, vel0 = sim.pos.clone(), sim.vel.clone()
        sim.roadmap_pref_velocity(gv)
        pref0 = sim.pref.clone()

        def step():
            sim.env_step(policy=_lib.POLICY_EXTERNAL, collect_stats=False)

        for rep in range(args.repeats):
            res = {}
            for arm in ("step", "pref"):  # alternated
                sim.pos.copy_(pos0)
                sim.vel.copy_(vel0)
                sim.pref.copy_(pref0)
                out = torch.empty_like(sim.pref)
                fn = step if arm == "step" else (lambda: sim.roadmap_pref_velocity(gv, out=out))
                res[arm] = events_us(fn, 5, 50)
            for arm, us in res.items():
                emit(dict(bench="pref_vs_step", world=label, arm=arm, repeat=rep, envs=E, agents_per_env=scn.agents_per_env,
                          roadmap_vertices=int(xy.shape[-2]), us_per_launch=round(us, 1),
                          pref_over_step=round(us / res["step"], 3)))
        sim.pos.copy_(pos0)
        _, vertex = sim.roadmap_pref_velocity(gv, out=torch.empty_like(sim.pref), return_vertex=True)
        torch.cuda.synchronize()
        _, dist0 = sim.roadmap(0)
        dist = np.stack([sim.roadmap(e)[1] for e in range(E)]) if jitter else np.broadcast_to(dist0, (E,) + dist0.shape)
        idx_w, cost_w = walks_per_agent(sim, xy, dist, pos0.cpu().numpy(), goal_vertex, vertex.cpu().numpy(),
                                        scn.params["radius"])
        emit(dict(bench="bsp_walks", world=label, envs=E, agents_per_env=scn.agents_per_env,
                  walks_per_agent_index_order=round(idx_w, 3), walks_per_agent_cost_order=round(cost_w, 3)))
        sim.close()
        torch.cuda.empty_cache()

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
