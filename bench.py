#!/usr/bin/env python
"""Headline benchmark: ORCA agent-steps/sec (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config cfg2|cfg3|cfg4|cfg5]
                  [--dump-outputs DIR]

Workloads = BASELINE.json configs, one GPU's share each (env instances are independent, so N GPUs
each own one share: weak scaling, no data-path collective; episode statistics are all-reduced
once after the timed region):
  cfg2 (default, configs[1])  circle-crossing 16 agents x 65,536 envs, ORCA policy = the reference's
                              run_sim(mode=0) loop: doStep + goal-directed preferred velocity + done
                              test (ALAN_true.py:106-131,631-636,547-566)
  cfg3 (configs[2])           circle 32 agents x 32,768 envs per GPU (262,144 over 8), ALAN online
                              action selection, 8 candidate actions (ALAN_true.py:569-628)
  cfg4 (configs[3])           dense crowd 256 agents + wall + 4 obstacle blocks x 2,048 envs per GPU
  cfg5 (configs[4])           one world of 1,000,000 agents, uniform-grid neighbor search (1 GPU; N
                              ranks run N replicas)

A "step" is one fused environment step over every env of the rank.  The cost of a step depends
on the phase of the episode (for cfg2: 184 us in the first steps, ~270 us when the ring meets in
the middle, less again once it has dissolved), so the timed window does not start at the reset
state: the state is first advanced, untimed, to episode step `--episode-step` (default per
config: the expensive mid-episode phase), then W warm-up steps, then exactly K timed steps.
`ms_per_step_by_phase` / `episode_mean_ms_per_step` report the whole profile next to it.

  value         device-timed throughput, state resident in HBM (CUDA events around each launch,
                L2 flushed between launches), max over ranks
  e2e           same metric through the host-buffer C-ABI call (orca_step_host): inputs go
                host->device and the new state comes device->host inside the timed region
  roofline      algorithmic HBM bytes / kernel time vs. the measured copy bandwidth
  cpu_baseline  the CPU oracle (restatement of RVO2, oracle/) on this box's host cores

--dump-outputs DIR writes what the last timed step left for its caller (rank 0's share: positions,
velocities and the per-agent / per-env results of the step) as DIR/<name>.npy, so that two builds
can be compared output for output on identical seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from

METRIC = "orca_agent_steps_per_sec"
UNIT = "agent-steps/s"
E2E_REPEATS = 3  # end-to-end regions per run (see run_ours)
SEED = 1234

# name -> workload description.  bytes = algorithmic HBM bytes per agent-step (DESIGN.md section 5,
# SURVEY 8d); episode_step = where the timed window starts (see module docstring)
CONFIGS = {
    "cfg2": dict(workload="circle-crossing 16 agents/env x 65,536 envs, ORCA policy, per B200", scenario="circle",
                 envs=65536, agents=16, policy="orca_step + done_test", bytes=41, kernel="step_small_kernel<10,GOAL>",
                 episode_step=130),
    "cfg3": dict(workload="circle 32 agents/env x 32,768 envs per B200 (262,144 over 8), ALAN online action selection, "
                          "8 candidate actions", scenario="circle", envs=32768, agents=32, policy="online_step (ALAN) + done_test",
                 bytes=82, kernel="step_small_kernel<10,ALAN>", episode_step=130),
    "cfg4": dict(workload="dense crowd 256 agents/env + wall + 4 obstacle blocks x 2,048 envs per B200 (16,384 over 8), "
                          "ORCA policy", scenario="crowd_blocks", envs=2048, agents=256, policy="orca_step + done_test",
                 bytes=48, kernel="step_small_kernel<10,GOAL> (in-block grid)", episode_step=60),
    "cfg5": dict(workload="single-env crowd of 1,000,000 agents, maxNeighbors 10, uniform-grid neighbor search, 1 B200",
                 scenario="crowd", envs=1, agents=1_000_000, policy="orca_step + done_test", bytes=150,
                 kernel="grid pipeline + step_grid_kernel<10,GOAL>", episode_step=60),
}
PHASE_STEPS = {"cfg2": (10, 60, 130, 250, 500, 900), "cfg3": (10, 60, 130, 250, 500, 900), "cfg4": (10, 60, 150, 400),
               "cfg5": (10, 60, 150)}


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst)"
    return 6650.0, "fallback (B200_PROFILING.md)"


_RESULT_OUT = sys.stdout  # replaced in main() by a private duplicate of the real stdout


def _static_profile(cfg_name):
    """ncu figures of the dominant kernel from the COMMITTED capture (profiles/traffic.json): they
    are not measured in this run and say which capture / episode step they come from."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(path):
        return None, None
    with open(path) as f:
        t = json.load(f).get(cfg_name)
    if not t:
        return None, None
    prof = {k: t[k] for k in ("issue_slots_busy_frac", "warp_instructions_per_launch", "active_lanes_per_instruction")
            if k in t}
    prof.update(static=True, source=t.get("source"), episode_step=t.get("episode_step"))
    return t.get("dram_bytes_per_launch"), prof


class ClockSampler:
    """Samples SM clocks + throttle reasons (NVML, every few ms) while the timed region runs."""

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.samples = []  # (sm_mhz, reasons bitmask)
        self.max_mhz = None
        self._stop = threading.Event()
        self._t = None
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices; honour CUDA_VISIBLE_DEVICES remapping
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = gpu_index
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if gpu_index < len(ids) and ids[gpu_index].isdigit():
                    phys = int(ids[gpu_index])
            self._h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self._nvml = pynvml
        except Exception:
            self._nvml = None

    def _run(self):
        nv = self._nvml
        while not self._stop.is_set():
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                reasons = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                self.samples.append((mhz, reasons))
            except Exception:
                pass
            self._stop.wait(0.002)

    def __enter__(self):
        if self._nvml is not None:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._t is not None:
            self._t.join(timeout=2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        nv = self._nvml
        sm = sorted(s[0] for s in self.samples)
        bits = 0
        for s in self.samples:
            bits |= s[1]
        names = [("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"),
                 ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
                 ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"),
                 ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap")]
        alt = {"nvmlClocksEventReasonHwSlowdown": 0x8, "nvmlClocksEventReasonHwThermalSlowdown": 0x40,
               "nvmlClocksEventReasonSwThermalSlowdown": 0x20, "nvmlClocksEventReasonSwPowerCap": 0x4}
        reasons = [n for n, attr in names if bits & int(getattr(nv, attr, alt[attr]))]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(self.samples)}


def _scenario(cfg, envs, seed):
    from collision_avoidance_b200 import scenarios
    if cfg["scenario"] == "crowd_blocks":
        return scenarios.crowd(envs, cfg["agents"], seed=seed, blocks=4)
    return scenarios.make(cfg["scenario"], envs, cfg["agents"], seed=seed)


def _config_dict(cfg_name, cfg, args):
    """Identical for both arms (the driver compares them)."""
    return {"workload": cfg["workload"], "name": cfg_name, "envs_per_gpu": cfg["envs"], "agents_per_env": cfg["agents"],
            "policy": cfg["policy"], "episode_window": [args.episode_step + args.warmup, args.episode_step + args.warmup + args.steps]}


# ------------------------------------------------------------------------------------------
def cpu_orca_throughput(cfg, envs, episode_step, warmup, steps, threads):
    """The CPU oracle (C++ restatement of RVO2 behind the reference's shell loop: doStep + float64
    goal-directed preferred velocity) on `envs` envs of the workload, `threads` host threads, over
    the same episode window as the GPU arm.  Returns (agent-steps/s, seconds timed)."""
    from oracle import rvo2_oracle
    from oracle.helpers import oracle_sims
    scn = _scenario(cfg, envs, SEED)
    sims = oracle_sims(scn)
    goals = scn.goal.astype("float64")
    if episode_step + warmup > 0:
        rvo2_oracle.batch_orca_steps(sims, goals, episode_step + warmup, threads)
    t0 = time.perf_counter()
    rvo2_oracle.batch_orca_steps(sims, goals, steps, threads)
    dt = time.perf_counter() - t0
    return envs * cfg["agents"] * steps / dt, dt


def cpu_baseline(cfg, args, target_seconds: float = 15.0, threads: int | None = None):
    """Bounded sample for the in-line `cpu_baseline` object of the GPU arm: as many envs of the
    workload as ~target_seconds of host work cover (fast-forward included)."""
    threads = min(threads or (os.cpu_count() or 1), cfg["envs"])
    total_steps = args.episode_step + args.warmup + args.steps
    # calibrate on a few envs over a short window
    cal_envs = max(1, min(cfg["envs"], 2 * threads))
    v, _ = cpu_orca_throughput(cfg, cal_envs, 0, 2, 8, threads)
    envs = int(target_seconds * v / (cfg["agents"] * total_steps))
    envs = max(1 if cfg["envs"] == 1 else threads, min(cfg["envs"], envs))
    value, dt = cpu_orca_throughput(cfg, envs, args.episode_step, args.warmup, args.steps, threads)
    return {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{envs} of {cfg['envs']} envs x {cfg['agents']} agents x {args.steps} steps of the same episode window "
                      f"(steps {args.episode_step + args.warmup}..{args.episode_step + args.warmup + args.steps}), C++ oracle: kd-tree + ORCA + LP, "
                      f"float64 preferred-velocity update, {dt:.2f} s timed"}


def cpu_python_driver_baseline(cfg, steps: int = 30, envs: int = 8):
    """The reference's own call pattern on one core: per agent setAgentPrefVelocity, one doStep,
    per agent getAgentPosition/getAgentVelocity, all through Python (collision_avoidence_env.py
    :371-400), with the oracle standing in for rvo2.  This is what "Python-RVO2 as the reference
    uses it" costs; reported next to the C++-driver figure."""
    from collision_avoidance_b200 import scenarios
    from oracle.shell_oracle import AlanShellOracle
    n = min(cfg["agents"], 64)
    scn = scenarios.circle(envs, n, seed=SEED)
    shells = [AlanShellOracle(scn, e) for e in range(envs)]
    for sh in shells:
        sh.orca_step()
    t0 = time.perf_counter()
    for _ in range(steps):
        for sh in shells:
            sh.orca_step()
            sh.step_count += 1
            sh.done_test()
    dt = time.perf_counter() - t0
    return {"value": envs * n * steps / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"{envs} envs x {n} agents x {steps} steps, Python per-agent call pattern over the oracle"}


def run_reference(args, cfg_name, cfg):
    """--impl reference: the reference's own CPU implementation of the path.  rvo2 (Python-RVO2)
    is not available offline, so this times the oracle port of it (oracle/) with all host threads
    on the SAME config and episode window; each step covers the full per-GPU batch for cfg2 and a
    bounded sample of it where the full batch would not finish within minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = min(os.cpu_count() or 1, cfg["envs"])   # the oracle driver parallelises over envs
    total_steps = args.episode_step + args.warmup + args.steps
    # full batch when it costs < ~90 s of host work at ~3e6 agent-steps/s/thread, else a bounded sample
    budget = 90.0 * 3.0e6 * threads
    envs = cfg["envs"]
    if cfg["envs"] * cfg["agents"] * total_steps > budget and cfg["envs"] > 1:
        envs = max(threads, int(budget / (cfg["agents"] * total_steps)))
    value, dt = cpu_orca_throughput(cfg, envs, args.episode_step, args.warmup, args.steps, threads)
    note = "ORCA policy" if "ALAN" not in cfg["policy"] else \
        "doStep + goal-directed preferred velocity only: the ALAN bandit (Python in the reference) is NOT included, which favours this arm"
    sample = (f"{envs} of {cfg['envs']} envs x {cfg['agents']} agents per step, {threads} threads, {dt:.2f} s timed; {note}")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3 * (cfg["envs"] / envs), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _config_dict(cfg_name, cfg, args),
        "notes": "rvo2 (Python-RVO2) unavailable offline; oracle port of RVO2 (oracle/rvo2_oracle.cpp) timed on host cores; "
                 "ms_per_step is scaled to the full per-GPU batch",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=_RESULT_OUT, flush=True)


# ------------------------------------------------------------------------------------------
class GpuWorkload:
    """One GPU's share of a BASELINE config: state on the device + the fused step."""

    def __init__(self, cfg_name, cfg, dev, rank):
        import torch
        from collision_avoidance_b200 import _lib, alan
        from collision_avoidance_b200.sim import BatchedRVOSimulator
        self.torch, self._lib, self.cfg, self.name, self.dev = torch, _lib, cfg, cfg_name, dev
        E, N = cfg["envs"], cfg["agents"]
        self.E, self.N = E, N
        self.alan = None
        if cfg_name == "cfg3":
            self.alan = alan.Collision_Avoidance_Sim(numAgents=N, scenario="circle", num_envs=E, seed=SEED + rank, device=dev)
            self.sim = self.alan.sim
            self.scn = self.alan.scn
        else:
            self.scn = _scenario(cfg, E, SEED + rank)
            self.sim = BatchedRVOSimulator(E, N, device=dev, **self.scn.params)
            self.sim.set_obstacles(self.scn.obstacles, per_env=self.scn.per_env_obstacles)
        self.reset()

    def reset(self):
        torch, dev, E, N = self.torch, self.dev, self.E, self.N
        if self.alan is not None:
            self.alan.reset()
            self.alan.sim.stats.zero_()
            return
        self.sim.pos.copy_(torch.from_numpy(self.scn.pos))
        self.sim.vel.copy_(torch.from_numpy(self.scn.vel))
        self.st = dict(goal=torch.from_numpy(self.scn.goal).to(dev), goal2=torch.from_numpy(self.scn.goal2).to(dev),
                       agent_done=torch.zeros(E, N, dtype=torch.uint8, device=dev),
                       arrival_time=torch.full((E, N), 0.0, device=dev),
                       env_step=torch.zeros(E, dtype=torch.int32, device=dev),
                       env_done_cnt=torch.zeros(E, dtype=torch.int32, device=dev))
        self.sim.stats.zero_()

    def step(self, steps=1):
        if self.alan is not None:
            self.alan.online_step(steps=steps)
        else:
            self.sim.env_step(policy=self._lib.POLICY_GOAL, done_mode=self._lib.DONE_GOAL_RADIUS_DEFERRED, steps=steps, **self.st)

    def goal_tensor(self):
        return self.alan.goal if self.alan is not None else self.st["goal"]

    def outputs(self):
        """What a caller holds after a step: the new state and the results the step wrote."""
        out = {"pos": self.sim.pos, "vel": self.sim.vel}
        if self.alan is not None:
            a = self.alan
            out.update(reward=a.reward, action_ids=a.action_ids, agent_done=a.agents_done, arrival_time=a.agents_time,
                       env_step=a.env_step, env_done_cnt=a.env_done_cnt)
        else:
            out.update({k: self.st[k] for k in ("agent_done", "arrival_time", "env_step", "env_done_cnt")})
        return out


DUMP_LIMIT_BYTES = 64_000_000


def dump_outputs(wl, out_dir):
    """DIR/<name>.npy of wl.outputs(): float32 as computed, flags as float32 and counters as float64
    (both exact)."""
    import numpy as np
    arrays = {}
    for name, t in wl.outputs().items():
        a = t.cpu().numpy()
        arrays[name] = a.astype(np.float32 if a.dtype in (np.float32, np.uint8) else np.float64)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args, cfg_name, cfg):
    import torch
    import torch.distributed as dist
    from collision_avoidance_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # one process per GPU: run on (and pin host buffers from) the cores next to that GPU
    from collision_avoidance_b200.dist import bind_to_gpu_numa
    # (only with several ranks: at N=1 the CPU baseline below wants every host core)
    cores = bind_to_gpu_numa(local_rank) if world > 1 and not os.environ.get("BENCH_NO_AFFINITY") else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    wl = GpuWorkload(cfg_name, cfg, dev, rank)
    sim, E, N = wl.sim, wl.E, wl.N
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-timed region: fast-forward (untimed) -> W warm-up -> K timed steps -----------
    if args.episode_step > 0:
        wl.step(steps=args.episode_step)
    for _ in range(args.warmup):
        wl.step()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    launches0 = sim.launch_count()
    barrier()
    with ClockSampler(local_rank) as clocks:
        wall0 = time.perf_counter()
        for i in range(args.steps):
            flush_buf.zero_()  # evict the state from L2 between timed launches
            starts[i].record()
            wl.step()
            ends[i].record()
        barrier()
        wall = time.perf_counter() - wall0
    launches = sim.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(wl, args.dump_outputs)
    kernel_ms = [s.elapsed_time(e) for s, e in zip(starts, ends)]
    total_ms = sum(kernel_ms)
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    value = world * E * N * args.steps / (total_ms_max * 1e-3)

    # episode statistics: the only collective of the path (one packed all-reduce, after timing)
    stats = sim.stats.clone()
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
    stats_d = {"agent_steps": int(stats[_lib.STAT_AGENT_STEPS]), "finished": int(stats[_lib.STAT_FINISHED]),
               "collisions": int(stats[_lib.STAT_COLLISIONS]), "lp3_calls": int(stats[_lib.STAT_LP3_CALLS]),
               "overflow": int(stats[_lib.STAT_OVERFLOW])}

    # ---- end-to-end region: host buffers through the C ABI, same episode phase ----------------
    e2e_steps = max(3, args.steps)
    bytes_state = E * N * 8
    e2e_min = None
    if wl.alan is None:
        # (huge-page-backed, cudaHostRegister'ed buffers measured the same as pin_memory(): tools/e2e_hostmem.py)
        pos_h = sim.pos.cpu().pin_memory()
        vel_h = sim.vel.cpu().pin_memory()
        goal_h = wl.goal_tensor().cpu().pin_memory()

        def host_region(vel_out, aux_unchanged):
            sim.step_host(pos_h, vel_h, goal_h, policy=_lib.POLICY_GOAL, upload_state=True, steps=1, aux_unchanged=aux_unchanged)
            for _ in range(24):  # untimed: the library times both of its routes (direct / staged) on its first ten steady calls and keeps the faster
                sim.step_host(pos_h, vel_out, goal_h, policy=_lib.POLICY_GOAL, upload_state=False, steps=1, aux_unchanged=aux_unchanged)
            barrier()
            per_call = []
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                tc = time.perf_counter()
                sim.step_host(pos_h, vel_out, goal_h, policy=_lib.POLICY_GOAL, upload_state=False, steps=1, aux_unchanged=aux_unchanged)
                per_call.append(time.perf_counter() - tc)
            barrier()
            dt = time.perf_counter() - t0
            if os.environ.get("BENCH_E2E_TRACE"):
                pc = sorted(per_call)
                print(f"e2e per call: min {pc[0] * 1e3:.3f} median {pc[len(pc) // 2] * 1e3:.3f} p90 {pc[int(len(pc) * 0.9)] * 1e3:.3f} "
                      f"max {pc[-1] * 1e3:.3f} ms; region {dt / e2e_steps * 1e3:.3f} ms/step", file=sys.stderr)
            return dt

        # headline e2e: per step the goals go host->device (the setAgentPrefVelocity traffic), doStep,
        # then positions + velocities come device->host (the getAgentPosition/Velocity traffic)
        # The host link of a shared box is not ours alone: the same loop measures 0.40 ms per step in one region
        # and 0.43-0.6 ms in the next (per-call minimum 0.393 ms throughout, profiles/README.md).  Three
        # regions of K steps each, all reported; the headline is the fastest one (max over ranks per region).
        e2e_regions = [host_region(vel_h, False) for _ in range(E2E_REPEATS)]
        h2d, d2h = bytes_state, 2 * bytes_state
        e2e_api = ("BatchedRVOSimulator.step_host -> orca_step_host_ex (pinned host buffers; the library keeps the faster of its "
                   "two routes: kernel reads/writes the mapped host buffers directly, or chunked upload | step | download over streams)")
        # the least a host-side run_sim(mode=0) loop needs per step: the new positions (the goals are
        # static, velocities are never read by that loop: ALAN_true.py:483-495,547-566,631-633)
        min_dt = host_region(None, True)
        tm = torch.tensor([min_dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        e2e_min = {"value": world * E * N * e2e_steps / float(tm.item()), "unit": UNIT, "h2d_bytes_per_step": 0,
                   "d2h_bytes_per_step": bytes_state,
                   "api": "orca_step_host_ex(vel_host = NULL, ORCA_HOST_AUX_UNCHANGED): positions-only write-back, goal buffer not re-read"}
    else:
        # ALAN has no per-step host INPUT (actions are drawn on the device); what a host-side caller
        # reads back every step is the reward, the chosen action and the done flags
        rew_h = torch.empty(E, N, dtype=torch.float32).pin_memory()
        act_h = torch.empty(E, N, dtype=torch.uint8).pin_memory()
        done_h = torch.empty(E, N, dtype=torch.uint8).pin_memory()
        e2e_regions = []
        for _ in range(E2E_REPEATS):
            barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                wl.alan.online_step()
                rew_h.copy_(wl.alan.reward, non_blocking=True)
                act_h.copy_(wl.alan.action_ids, non_blocking=True)
                done_h.copy_(wl.alan.agents_done, non_blocking=True)
                torch.cuda.synchronize()
            barrier()
            e2e_regions.append(time.perf_counter() - t0)
        h2d, d2h = 0, E * N * 6
        e2e_api = ("alan.Collision_Avoidance_Sim.online_step + per-step device->host read of rewards, action ids and done flags "
                   "(pinned buffers); the ALAN step has no per-step host input")
    te = torch.tensor(e2e_regions, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_regions_ms = [float(x) / e2e_steps * 1e3 for x in te.tolist()]
    e2e_value = world * E * N * e2e_steps / float(te.min().item())

    # ---- host-link probe: what the box's host memory / PCIe complex carries when every rank moves
    # the e2e byte pattern (8 B in + 16 B out per agent) with NO compute: the ceiling of `e2e` -----
    probe_in = torch.empty(E * N * 2, dtype=torch.float32).pin_memory()
    probe_out = torch.empty(E * N * 4, dtype=torch.float32).pin_memory()
    d_in, d_out = torch.empty(E * N * 2, device=dev), torch.empty(E * N * 4, device=dev)
    s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    probe_iters = 20

    def probe_once():
        with torch.cuda.stream(s_in):
            d_in.copy_(probe_in, non_blocking=True)
        with torch.cuda.stream(s_out):
            probe_out.copy_(d_out, non_blocking=True)
    for _ in range(3):
        probe_once()
    barrier()
    t0 = time.perf_counter()
    for _ in range(probe_iters):
        probe_once()
    barrier()
    tp = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tp, op=dist.ReduceOp.MAX)
    probe_gbs = world * (probe_in.numel() + probe_out.numel()) * 4 * probe_iters / float(tp.item()) / 1e9

    # ---- cost profile over the episode (rank 0, untimed in the headline) -----------------------
    by_phase, trace_mean = None, None
    if rank == 0 and not args.no_phase_profile:
        wl.reset()
        by_phase, at, chunk_ms, chunk_steps = {}, 0, [], []
        for target in PHASE_STEPS[cfg_name]:
            if target > at:      # fast-forward, itself timed as one chunk (no L2 flush) for the episode mean
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                wl.step(steps=target - at)
                e1.record()
                torch.cuda.synchronize()
                chunk_ms.append(e0.elapsed_time(e1))
                chunk_steps.append(target - at)
                at = target
            ms = []
            for _ in range(5):
                flush_buf.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                wl.step()
                e1.record()
                torch.cuda.synchronize()
                ms.append(e0.elapsed_time(e1))
                at += 1
            by_phase[str(target)] = sum(ms) / len(ms)
        trace_mean = sum(chunk_ms) / max(1, sum(chunk_steps))

    if rank == 0:
        peak, peak_src = _peaks()
        avg_kernel_s = (total_ms / args.steps) * 1e-3  # rank 0's own launches
        achieved = cfg["bytes"] * E * N / avg_kernel_s / 1e9
        traffic, issue_profile = _static_profile(cfg_name)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": _config_dict(cfg_name, cfg, args),
            "notes": {"sharding": f"envs x{world}, no data-path collective" if cfg["envs"] > 1 else f"{world} independent replicas",
                      "l2": "flushed between timed launches (256 MiB memset; per-GPU state is smaller than L2)",
                      "timing": "CUDA events per launch, summed; max over ranks",
                      "window": f"state advanced untimed to episode step {args.episode_step}, then {args.warmup} warm-up and "
                                f"{args.steps} timed steps"},
            "ms_per_step_by_phase": by_phase, "episode_mean_ms_per_step": trace_mean,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_static": True, "peak_source": peak_src,
                         "bytes_per_agent_step": cfg["bytes"], "kernel": cfg["kernel"],
                         "note": "kernel is instruction-issue / latency bound, not HBM bound; see DESIGN.md section 5; "
                                 "traffic and issue_profile come from the committed ncu capture, not from this run",
                         "issue_profile": issue_profile},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "regions": E2E_REPEATS, "ms_per_step_by_region": e2e_regions_ms,
                    "region_rule": "fastest of the regions (each K steps, max over ranks): the host link of a shared box carries other tenants' traffic",
                    "api": e2e_api},
            "e2e_min_traffic": e2e_min,
            "host_link_probe": {"aggregate_GBps": probe_gbs, "bytes_per_agent_step": 24,
                                "e2e_ceiling": probe_gbs * 1e9 / 24.0,
                                "how": "every rank copies 8 B/agent host->device and 16 B/agent device->host (pinned, two streams, "
                                       "no kernel) at the same time; e2e cannot exceed this on this host"},
            "gpu_launches": launches,
            "clocks": clocks.summary(),
            "host_affinity": {"rank0_cores": len(cores) if cores else None,
                              "note": "each rank runs on the cores NVML lists next to its GPU" if cores else "not bound"},
            "wall_s_timed_region": wall,
            "episode_stats": stats_d,
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(cfg, args)
            line["cpu_baseline_python_driver"] = cpu_python_driver_baseline(cfg)
        print(json.dumps(line), file=_RESULT_OUT, flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--episode-step", type=int, default=None,
                    help="episode step the (untimed) fast-forward stops at before warm-up; default per config")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-phase-profile", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    cfg = CONFIGS[args.config]
    if args.episode_step is None:
        args.episode_step = cfg["episode_step"]
    # The contract is ONE JSON line on stdout.  Libraries may write there too (NCCL prints its
    # version banner to stdout when NCCL_DEBUG is set, as on the GPU boxes): keep a private handle on
    # the real stdout for the line and point fd 1 at stderr for everything else.
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args, args.config, cfg)
    else:
        run_ours(args, args.config, cfg)


if __name__ == "__main__":
    main()
