#!/usr/bin/env python
"""Device-timed cost of orca_agent_lines (BatchedRVOSimulator.orca_lines) against the step it mirrors.

Shapes: cfg2 (circle 16 agents x 65,536 envs), cfg4 (crowd 256 + blocks x 2,048 envs), cfg5 (one world
of 1,000,000 agents) and the gym shape (10 envs x 100,000 agents, maxNeighbors 5, per-env blocks).
Each shape is advanced 60 goal-directed steps into its episode; then the two arms -- the lines call
(default max_lines = maxNeighbors + 6) and orca_env_step(POLICY_GOAL) -- are timed with CUDA events
around 200 calls after 10 warm-up calls, alternated, 3 repeats.  The step arm moves the state on, so
the lines arm of the next repeat sees a later state.  Bytes written per agent by the lines call, from
the counts of the last call: min(count, max_lines) rows of 16 B plus two int32 counts.  Then, in a
separate pass under torch.profiler (CUDA activity only), 20 calls of each arm: device time per call of
every kernel, so the lines call's grid prep (G1-G4) and lines kernel can be told apart.  Prints the
device name and power limit, read in the same run, and one JSON line per shape; writes them to --out."""
import argparse
import json
import os
import sys

import torch
from torch.profiler import ProfilerActivity, profile

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


def kernel_split_us(fn, calls):
    """{kernel name: device us per call} of `calls` calls of fn, from torch.profiler."""
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            name = e.key.split("<")[0].split("(")[0].replace("void ", "").replace("orca::", "")
            out[name] = round(out.get(name, 0.0) + t / calls, 2)
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def shapes(small):
    s = 64 if small else 1
    gym = scenarios.crowd(10, 100_000 // s, seed=4, blocks=4)
    gym.params = dict(gym.params, maxNeighbors=5)
    return [("cfg2", scenarios.make("circle", 65_536 // s, 16, seed=1)),
            ("cfg4", scenarios.crowd(2_048 // s, 256, seed=2, blocks=4)),
            ("cfg5", scenarios.crowd(1, 1_000_000 // s, seed=3)),
            ("gym_10x100k_k5", gym)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "profiles",
                                                  "r05_agent_lines.jsonl"))
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--small", action="store_true", help="1/64 of every shape (a rehearsal, not a measurement)")
    args = ap.parse_args()
    gpu, power = device_info()
    print(f"device: {gpu}; power.limit, clocks.max.sm: {power}", flush=True)
    records = []
    for name, scn in shapes(args.small):
        E, N = scn.num_envs, scn.agents_per_env
        sim = BatchedRVOSimulator(E, N, device="cuda:0", **scn.params)
        sim.set_obstacles(scn.obstacles, per_env=scn.per_env_obstacles)
        sim.pos.copy_(torch.from_numpy(scn.pos))
        sim.vel.copy_(torch.from_numpy(scn.vel))
        goal = torch.from_numpy(scn.goal).cuda()
        for _ in range(60):
            sim.env_step(policy=_lib.POLICY_GOAL, goal=goal, collect_stats=False)
        L = sim.max_neighbors + _lib.MAX_OBST_LINES
        lines = torch.zeros(E, N, L, 4, dtype=torch.float32, device="cuda:0")
        cnt = torch.zeros(E, N, dtype=torch.int32, device="cuda:0")
        n_obst = torch.zeros(E, N, dtype=torch.int32, device="cuda:0")
        stream = sim._stream()

        def lines_call():  # the C call itself: no output allocation inside the timed window
            _lib.check(sim._L.orca_agent_lines(sim._h, sim._p(sim.pos), sim._p(sim.vel), L, sim._p(lines), sim._p(cnt),
                                               sim._p(n_obst), stream))

        def step_call():
            sim.env_step(policy=_lib.POLICY_GOAL, goal=goal, collect_stats=False)

        t_lines, t_step = [], []
        for _ in range(args.repeats):
            t_lines.append(events_us(lines_call, 10, args.reps))
            t_step.append(events_us(step_call, 10, args.reps))
        c = cnt.cpu().long()
        rows = torch.clamp(c, 0, L)
        split_lines = kernel_split_us(lines_call, 20)
        split_step = kernel_split_us(step_call, 20)
        rec = dict(shape=name, envs=E, agents_per_env=N, max_neighbors=sim.max_neighbors, max_lines=L,
                   lines_us=[round(x, 2) for x in t_lines], step_us=[round(x, 2) for x in t_step],
                   ratio_median=round(sorted(t_lines)[len(t_lines) // 2] / sorted(t_step)[len(t_step) // 2], 3),
                   bytes_written_per_agent=round(float(rows.float().mean()) * 16 + 8, 2),
                   bytes_written_per_agent_bound=L * 16 + 8, mean_lines_per_agent=round(float(c.float().mean()), 3),
                   lines_call_kernels_us=split_lines, step_kernels_us=split_step,
                   agents_beyond_max_lines=int((c > L).sum()), path="grid" if N >= 257 else "tile",
                   reps=args.reps, repeats=args.repeats, small=args.small, gpu=gpu, power_limit_and_max_sm_clock=power)
        print(json.dumps(rec), flush=True)
        records.append(rec)
        sim.close()
        del lines, cnt, n_obst
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for r in records:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
