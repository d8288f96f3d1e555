#!/usr/bin/env python
"""Device-timed cost of per-agent ORCA parameters (orca_set_agent_params) on one GPU.

Three arms per shape, from the same reset state:
  uniform       no table: the uniform kernels
  hetero-equal  a table holding the handle's own values: the same work through the HETERO kernels
  hetero-mixed  radius U(0.2, 0.8), maxSpeed U(0.5, 2), neighborDist U(1.5, 6), maxNeighbors in
                {0..K}, timeHorizon and timeHorizonObst U(0.5, 3), seeded (other work: other neighbor
                counts, more LP3 -- reported as measured)
Shapes: cfg2 circle 16 x 65,536 (GOAL policy), cfg4 crowd 256 + 4 blocks x 2,048 (GOAL), cfg5 one
crowd of 1,000,000 (uniform grid, GOAL), gym default world 10 x 100,000 (K = 5, RL policy + done test).
Method: CUDA events around 200 steps after 20 warm-up steps, every arm restarted from the reset
state, arms alternated, 3 repeats.  Prints the device name and power limit and one JSON line per
(shape, arm, repeat); writes them to --out."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from collision_avoidance_b200 import _lib, scenarios  # noqa: E402
from collision_avoidance_b200.sim import BatchedRVOSimulator  # noqa: E402

SHAPES = {
    "cfg2": lambda: scenarios.circle(65536, 16, seed=0),
    "cfg4": lambda: scenarios.crowd(2048, 256, seed=0, blocks=4),
    "cfg5": lambda: scenarios.crowd(1, 1_000_000, seed=0),
    "gym": lambda: scenarios.default_env(100_000, 10, seed=0),
}


def mixed(E, N, K, seed=1):
    rng = np.random.default_rng(seed)
    f = lambda lo, hi: rng.uniform(lo, hi, (E, N)).astype(np.float32)
    return dict(radius=f(0.2, 0.8), max_speed=f(0.5, 2.0), neighbor_dist=f(1.5, 6.0),
                max_neighbors=rng.integers(0, K + 1, (E, N)).astype(np.int32),
                time_horizon=f(0.5, 3.0), time_horizon_obst=f(0.5, 3.0))


def equal(scn):
    P, shape = scn.params, (scn.num_envs, scn.agents_per_env)
    return dict(neighbor_dist=np.full(shape, P["neighborDist"], np.float32),
                max_neighbors=np.full(shape, P["maxNeighbors"], np.int32),
                time_horizon=np.full(shape, P["timeHorizon"], np.float32),
                time_horizon_obst=np.full(shape, P["timeHorizonObst"], np.float32),
                radius=np.full(shape, P["radius"], np.float32), max_speed=np.full(shape, P["maxSpeed"], np.float32))


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


class Arm:
    def __init__(self, scn, name, ap, gym):
        self.scn, self.name, self.gym = scn, name, gym
        E, N = scn.num_envs, scn.agents_per_env
        self.sim = BatchedRVOSimulator(E, N, device="cuda:0", **scn.params)
        self.sim.set_obstacles(scn.obstacles, per_env=scn.per_env_obstacles)
        if ap is not None:
            self.sim.set_agent_params(**ap)
        dev = self.sim.pos.device
        self.pos0, self.vel0 = torch.from_numpy(scn.pos).to(dev), torch.from_numpy(scn.vel).to(dev)
        self.goal0 = torch.from_numpy(scn.goal).to(dev)
        self.goal2 = torch.from_numpy(scn.goal2).to(dev)
        self.goal = self.goal0.clone()
        self.theta = (torch.rand(E, N, generator=torch.Generator().manual_seed(2)) - 0.5).to(dev)
        self.reward = torch.zeros(E, N, device=dev)
        self.done = torch.zeros(E, N, dtype=torch.uint8, device=dev)
        self.env_step = torch.zeros(E, dtype=torch.int32, device=dev)
        self.env_done = torch.zeros(E, dtype=torch.int32, device=dev)

    def reset(self):
        self.sim.pos.copy_(self.pos0)
        self.sim.vel.copy_(self.vel0)
        self.goal.copy_(self.goal0)
        for t in (self.reward, self.done, self.env_step, self.env_done):
            t.zero_()

    def step(self):
        if self.gym:
            self.sim.env_step(policy=_lib.POLICY_RL, goal=self.goal, goal2=self.goal2, action_theta=self.theta,
                              reward=self.reward, done_mode=_lib.DONE_X_BELOW, agent_done=self.done,
                              env_step=self.env_step, env_done_cnt=self.env_done, collect_stats=False)
        else:
            self.sim.env_step(policy=_lib.POLICY_GOAL, goal=self.goal, collect_stats=False)

    def time(self, warmup, steps):
        self.reset()
        for _ in range(warmup):
            self.step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            self.step()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1000.0 / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="cfg2,cfg4,cfg5,gym")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "profiles",
                                                  "r03_agent_params.jsonl"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_agent_params needs a CUDA device")
    gpu, power = device_info()
    print(f"device: {gpu}; power.limit, clocks.max.sm: {power}", flush=True)
    lines = []
    for shape in args.shapes.split(","):
        scn = SHAPES[shape]()
        E, N = scn.num_envs, scn.agents_per_env
        arms = [Arm(scn, "uniform", None, shape == "gym"), Arm(scn, "hetero-equal", equal(scn), shape == "gym"),
                Arm(scn, "hetero-mixed", mixed(E, N, scn.params["maxNeighbors"]), shape == "gym")]
        for rep in range(args.repeats):
            for arm in arms:  # alternated
                us = arm.time(args.warmup, args.steps)
                rec = dict(shape=shape, arm=arm.name, repeat=rep, envs=E, agents_per_env=N, us_per_step=round(us, 2),
                           agent_steps_per_s=round(E * N / us * 1e6), warmup=args.warmup, steps=args.steps, gpu=gpu,
                           power_limit_and_max_sm_clock=power)
                print(json.dumps(rec), flush=True)
                lines.append(rec)
        for arm in arms:
            arm.sim.close()
        del arms
        torch.cuda.empty_cache()
    with open(args.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
