#!/usr/bin/env python
"""Golden fixtures recorded from the UNMODIFIED reference shells (run with
COLLISION_AVOIDANCE_REFERENCE naming a checkout of the reference; the fixtures are committed, the
reference is not).

What runs: collision_avoidance/ALAN/ALAN_true.py (``Collision_Avoidance_Sim``: ``_init_world_*``
:175-457, ``run_sim`` :106-131, ``online_step`` :569-628, ``orca_step`` :631-636, ``done_test``
:547-566), collision_avoidance/envs/collision_avoidence_env.py (``Collision_Avoidance_Env``:
``reset`` :461-488, ``step`` :367-416, ``orca_step`` :447-458, ``_get_obs`` :231-318) and
collision_avoidance/ALAN/Train_ALAN_action_space.py (``MCMC_trainer``: moves :86-126, accept
rule :41, ``train`` :27-47) -- imported as they lie, with ``tkinter`` / ``gym`` / ``ray`` stubbed
and ``time.clock`` patched (tests/_ref_stubs.py) and with ``rvo2.PyRVOSimulator`` bound to the
CPU oracle (oracle/rvo2_oracle.py; upstream rvo2 is not available, SURVEY F2).  The global RNGs
the reference draws from (``random``, ``np.random``; SURVEY Q11) are seeded, and
``np.random.choice`` is wrapped so that the uniform behind every softmax draw is recorded too.

Writes (tests/golden/):
  shell_scenarios.json     geometry of the six ``_init_world_*`` + the gym env's ``_init_world``
  shell_alan_<name>.npz    per-step states of ``run_sim`` (mode 1 = ALAN, mode 0 = ORCA only)
  shell_env[_small].npz    reset / step / orca_step of the gym env: obs, rewards, dones, states
  shell_calltrace.json.gz  every call the shells make at the rvo2 boundary, with its result
  shell_mcmc.json          MCMC moves, accept probabilities and a full ``train()`` on a fake cost
"""
from __future__ import annotations

import ast
import contextlib
import gzip
import io
import json
import os
import random
import sys
from math import cos, pi, sin

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import _ref_stubs  # noqa: E402
from oracle import rvo2_oracle  # noqa: E402

ACT_DIR = os.path.join(_ref_stubs.REFERENCE_ROOT, "collision_avoidance", "ALAN")

# (scenario, numAgents, action file or None = the default 8 actions, seed, recorded steps)
ALAN_RUNS = [
    ("circle", 32, None, 101, 160),          # BASELINE config 3's world shape
    ("circle", 16, "circle", 102, 160),
    ("blocks", 8, "blocks", 103, 160),
    ("deadlock", 10, "deadlock", 104, 200),
    ("congested", 12, "congested", 105, 200),
    ("incoming", 10, "incoming", 106, 160),
    ("crowd", 12, "crowd", 107, 160),
]
ORCA_RUNS = [("circle", 16, 201, 200), ("crowd", 24, 202, 200), ("congested", 12, 203, 300)]
SCENARIO_SHAPES = [("circle", 16, 11), ("circle", 7, 12), ("crowd", 20, 13), ("blocks", 9, 14), ("congested", 15, 15),
                   ("incoming", 10, 16), ("incoming", 17, 17), ("deadlock", 11, 18), ("deadlock", 8, 19)]


def read_act(name):
    with open(os.path.join(ACT_DIR, name + "_actions.act")) as f:
        return [tuple(a) for a in ast.literal_eval(f.read())]


# ---------------------------------------------------------------------------------- recording
class ChoiceRecorder:
    """Wraps ``np.random.choice``: numpy's legacy sampler takes ONE ``random_sample`` per draw with
    ``p`` given, so peeking it (draw, restore the state) gives the uniform behind the choice."""

    def __init__(self):
        self.uniforms, self.ids = [], []
        self._orig = np.random.choice

    def __enter__(self):
        def choice(a, size=None, replace=True, p=None):
            if p is not None and size == 1:
                st = np.random.get_state()
                u = float(np.random.random_sample())
                np.random.set_state(st)
                r = self._orig(a, size, replace, p)
                self.uniforms.append(u)
                self.ids.append(int(r[0]))
                return r
            return self._orig(a, size, replace, p)
        np.random.choice = choice
        return self

    def __exit__(self, *exc):
        np.random.choice = self._orig


def snapshot_sim(CA):
    sim, n = CA.sim, CA.numAgents
    return dict(pos=[sim.getAgentPosition(i) for i in range(n)], vel=[sim.getAgentVelocity(i) for i in range(n)],
                pref=[sim.getAgentPrefVelocity(i) for i in range(n)])


def polygons_of(CA):
    return [[CA.sim.getObstacleVertex(v) for v in ids] for ids in CA.world["obstacles_vertex_ids"]]


# ---------------------------------------------------------------------------------- scenarios
def gen_scenarios(alan_mod, env_mod):
    out = {"alan": [], "env": []}
    for name, n, seed in SCENARIO_SHAPES:
        random.seed(seed)
        CA = alan_mod.Collision_Avoidance_Sim(numAgents=n, scenario=name, visualize=False)
        min_ttime_ctor = CA.min_TTime            # 0: __init__ overwrites it after _init_world (ALAN_true.py:71)
        s = snapshot_sim(CA)
        rec = dict(name=name, numAgents=n, seed=seed, envsize=CA.envsize, max_step=CA.max_step,
                   pos=s["pos"], vel=s["vel"], pref=s["pref"],
                   targets=[[list(t[0]), list(t[1])] for t in CA.world["targets_pos"]],
                   polygons=polygons_of(CA), min_TTime_after_ctor=min_ttime_ctor)
        random.seed(seed)
        CA.reset()
        rec["min_TTime_after_reset"] = float(CA.min_TTime)     # :161-172, kept by reset() (:79-103)
        rec["pos_after_reset"] = snapshot_sim(CA)["pos"]
        out["alan"].append(rec)
    for n, seed in ((10, 21), (6, 22)):
        random.seed(seed)
        env = env_mod.Collision_Avoidance_Env(numAgents=n)
        s = snapshot_sim(env)
        out["env"].append(dict(numAgents=n, seed=seed, envsize=env.envsize, pos=s["pos"], vel=s["vel"], pref=s["pref"],
                               targets=[list(t) for t in env.world["targets_pos"]], polygons=polygons_of(env),
                               action_space=[env.action_space.low, env.action_space.high, list(env.action_space.shape)],
                               observation_space=[env.observation_space.low, env.observation_space.high,
                                                  list(env.observation_space.shape)],
                               ray_lines=env.ray_lines, approx_lines=env.approx_lines,
                               registry=dict(_ref_stubs.REGISTRY)))
    return out


# ---------------------------------------------------------------------------------- ALAN runs
def gen_alan_run(alan_mod, name, n, actions, seed, rec_steps, mode):
    random.seed(seed)
    np.random.seed(seed)
    CA = alan_mod.Collision_Avoidance_Sim(numAgents=n, scenario=name, online_actions=actions, visualize=False)
    A = len(CA.online_actions)
    frames = []

    def frame():
        s = snapshot_sim(CA)
        s.update(w=[list(w) for w in CA.world["action_weights"]], done=list(CA.agents_done),
                 atime=list(CA.agents_time), tgt=[list(t[0]) for t in CA.world["targets_pos"]])
        return s

    init = frame()
    init["tgt2"] = [list(t[1]) for t in CA.world["targets_pos"]]
    frames.append(init)
    orig_done_test = CA.done_test

    def recording_done_test():          # run_sim calls it once per step, after the step (:120)
        r = orig_done_test()
        if len(frames) <= rec_steps:
            frames.append(frame())
        return r

    CA.done_test = recording_done_test
    with ChoiceRecorder() as rec:
        success, total_time, ttime, min_ttime = CA.run_sim(mode)
    T = CA.step_count
    f32 = lambda k: np.asarray([f[k] for f in frames], np.float32)        # noqa: E731
    f64 = lambda k: np.asarray([f[k] for f in frames], np.float64)        # noqa: E731
    out = dict(scenario=name, numAgents=n, seed=seed, mode=mode, steps=T, actions=np.asarray(CA.online_actions, np.float64),
               pos=f32("pos"), vel=f32("vel"), pref=f32("pref"), w=f64("w"), done=np.asarray([f["done"] for f in frames], np.uint8),
               atime=f64("atime"), tgt=f64("tgt"), tgt2=np.asarray(init["tgt2"], np.float64),
               polygons=np.asarray(polygons_of(CA), np.float64), envsize=CA.envsize,
               final_atime=np.asarray(CA.agents_time, np.float64), final_done=np.asarray(CA.agents_done, np.uint8),
               result=np.asarray([float(success), total_time, ttime, min_ttime], np.float64))
    if mode == 1:
        out["u"] = np.asarray(rec.uniforms, np.float64).reshape(T, n)
        out["aid"] = np.asarray(rec.ids, np.uint8).reshape(T, n)
        assert A <= 16
    return out


# ---------------------------------------------------------------------------------- gym env
def neighbor_lists(sim, n, k_agents, k_obst):
    na = np.zeros(n, np.int32)
    ia = np.full((n, k_agents), -1, np.int32)
    no = np.zeros(n, np.int32)
    io = np.full((n, k_obst), -1, np.int32)
    for i in range(n):
        na[i] = sim.getAgentNumAgentNeighbors(i)
        for j in range(na[i]):
            ia[i, j] = sim.getAgentAgentNeighbor(i, j)
        no[i] = sim.getAgentNumObstacleNeighbors(i)
        for j in range(no[i]):
            io[i, j] = sim.getAgentObstacleNeighbor(i, j)
    return na, ia, no, io


def gen_env_run(env_mod, seed=301, n=10, steps_a=260, steps_b=60, steps_orca=120, stop_on_done=False):
    random.seed(seed)
    env = env_mod.Collision_Avoidance_Env(numAgents=n)      # __init__ ends with reset() (:74)
    rng = np.random.RandomState(seed)
    keys = ["agent_%d" % i for i in range(n)]
    rows = []

    def row(kind, obs, rew=None, done=None, theta=None):
        s = snapshot_sim(env)
        na, ia, no, io = neighbor_lists(env.sim, n, env.maxNeighbors, 16)
        rows.append(dict(kind=kind, pos=s["pos"], vel=s["vel"], pref=s["pref"],
                         obs=[list(map(float, obs[k])) for k in keys],
                         rew=[0.0] * n if rew is None else [float(rew[k]) for k in keys],
                         done=False if done is None else bool(done["__all__"]),
                         theta=[0.0] * n if theta is None else theta, agents_done=list(env.agents_done),
                         tgt=[list(t) for t in env.world["targets_pos"]], na=na, ia=ia, no=no, io=io,
                         step_count=env.step_count))

    row(0, env.gym_obs)                                      # state after the constructor's reset
    # episode A: small steering angles so that agents pass the gate and finish (x < 2, :359)
    for t in range(steps_a):
        theta = [float(x) for x in rng.normal(0.0, 0.35, n)]
        obs, rew, done, info = env.step({k: theta[i] for i, k in enumerate(keys)})
        row(1, obs, rew, done, theta)
        if stop_on_done and done["__all__"]:
            break
    random.seed(seed + 1)
    row(2, env.reset())                                      # Q4: positions only; velocities, targets, lists kept
    for t in range(steps_b):
        theta = [float(x) for x in rng.uniform(-pi, pi, n)]
        obs, rew, done, info = env.step({k: theta[i] for i, k in enumerate(keys)})
        row(1, obs, rew, done, theta)
    random.seed(seed + 2)
    row(2, env.reset())
    for t in range(steps_orca):                              # the reference's __main__ loop (:570-573), config 1
        env.orca_step((0, 0))
        row(3, env.gym_obs)
    arr = lambda k, dt: np.asarray([r[k] for r in rows], dt)  # noqa: E731
    return dict(numAgents=n, seed=seed, kind=arr("kind", np.int8), pos=arr("pos", np.float32), vel=arr("vel", np.float32),
                pref=arr("pref", np.float32), obs=arr("obs", np.float64), rew=arr("rew", np.float64), done=arr("done", np.uint8),
                theta=arr("theta", np.float64), agents_done=arr("agents_done", np.uint8), tgt=arr("tgt", np.float64),
                na=arr("na", np.int32), ia=arr("ia", np.int32), no=arr("no", np.int32), io=arr("io", np.int32),
                step_count=arr("step_count", np.int32), polygons=np.asarray(polygons_of(env), np.float64),
                max_step=env.max_step)


# ---------------------------------------------------------------------------------- boundary call trace
class RecordingSimulator:
    """PyRVOSimulator proxy that logs every boundary call: [method, args, kwargs, result]."""
    LOG = []

    def __init__(self, *a, **k):
        self._s = rvo2_oracle.PyRVOSimulator(*a, **k)
        RecordingSimulator.LOG.append(["__init__", _plain(a), _plain(k), None])

    def __getattr__(self, name):
        fn = getattr(self._s, name)

        def call(*a, **k):
            r = fn(*a, **k)
            RecordingSimulator.LOG.append([name, _plain(a), _plain(k), _plain(r)])
            return r
        return call


def _plain(x):
    if isinstance(x, dict):
        return {k: _plain(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [_plain(v) for v in x]
    if isinstance(x, (np.floating, float)):
        return float(x)
    if isinstance(x, (np.integer, int)):
        return int(x)
    return x


def gen_calltrace(alan_mod, env_mod):
    traces = {}
    _ref_stubs.bind_simulator(RecordingSimulator)
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            RecordingSimulator.LOG = []
            random.seed(401)
            np.random.seed(401)
            CA = alan_mod.Collision_Avoidance_Sim(numAgents=8, scenario="blocks", online_actions=read_act("blocks"),
                                                  visualize=False)
            for t in range(90):                     # run_sim's loop body (:113-121), cut short
                CA.online_step()
                CA.step_count += 1
                CA.done_test()
            traces["alan_blocks_online"] = RecordingSimulator.LOG
            RecordingSimulator.LOG = []
            random.seed(402)
            CA = alan_mod.Collision_Avoidance_Sim(numAgents=12, scenario="congested", visualize=False)
            for t in range(90):
                CA.orca_step()
                CA.step_count += 1
                CA.done_test()
            traces["alan_congested_orca"] = RecordingSimulator.LOG
            RecordingSimulator.LOG = []
            random.seed(403)
            env = env_mod.Collision_Avoidance_Env(numAgents=10)
            rng = np.random.RandomState(403)
            for t in range(50):
                env.step({"agent_%d" % i: float(a) for i, a in enumerate(rng.normal(0, 0.4, 10))})
            random.seed(404)
            env.reset()
            for t in range(20):
                env.orca_step((0, 0))
            traces["env_step_reset_orca"] = RecordingSimulator.LOG
            RecordingSimulator.LOG = []
    finally:
        _ref_stubs.bind_simulator(rvo2_oracle.PyRVOSimulator)
    return traces


# ---------------------------------------------------------------------------------- MCMC trainer
def fake_cost(actions):
    """Deterministic stand-in for ``evaluate_action`` (3 simulations in the reference, :55-67):
    smooth in the action angles, so that the accept rule sees both better and worse proposals."""
    ang = np.arctan2([a[1] for a in actions], [a[0] for a in actions])
    return float(10.0 + np.sum(np.cos(3.0 * ang)) + 0.25 * len(actions))


def gen_mcmc(train_mod):
    T = train_mod.MCMC_trainer
    bare = T.__new__(T)                                    # the moves need no simulator
    out = {"moves": [], "train": []}
    np.random.seed(501)
    random.seed(501)
    actions = [(1, 0), bare.random_action()]
    for k in range(120):
        before = [list(a) for a in actions]
        st_before = len(actions)
        modification = int(bare.select_modification(actions, k))
        if modification == 1 and st_before <= 2:
            modification = 0                               # keep >= 2 actions so that every move stays legal
        d, actions = bare.apply_modification(actions, modification)
        out["moves"].append(dict(before=before, modification=modification, dist=float(d),
                                 after=[list(a) for a in actions], likelihood=float(bare.symmetric_likelihood(d))))
    for seed, rounds in ((502, 25), (503, 40)):
        np.random.seed(seed)
        random.seed(seed)
        tr = T.__new__(T)
        tr.numRounds = rounds
        tr.evaluate_action = lambda actions, i=0: fake_cost(actions)
        # __init__ body (:16-25) without the simulator
        tr.actions = [(1, 0), tr.random_action()]
        tr.actions_opt = tr.actions
        tr.eval = tr.evaluate_action(tr.actions)
        tr.eval_opt = tr.eval
        tr.init_temp, tr.final_temp = 0.9, 0.1
        tr.temp = tr.init_temp
        tr.delta_temp = (tr.final_temp - tr.init_temp) / (tr.numRounds - 1)
        hist = []
        orig_eval = tr.evaluate_action

        def logging_eval(actions, i=0, _tr=tr, _h=hist, _e=orig_eval):
            v = _e(actions, i)
            _h.append(dict(round=i, temp=_tr.temp, proposal=[list(a) for a in actions], new_eval=v))
            return v
        tr.evaluate_action = logging_eval
        best = tr.train()
        out["train"].append(dict(seed=seed, numRounds=rounds, history=hist, actions_opt=[list(a) for a in best],
                                 eval_opt=tr.eval_opt, final_actions=[list(a) for a in tr.actions], final_eval=tr.eval,
                                 final_temp=tr.temp))
    return out


def main():
    alan_mod, env_mod, train_mod = _ref_stubs.load_reference(rvo2_oracle.PyRVOSimulator)
    with open(os.path.join(HERE, "shell_scenarios.json"), "w") as f:
        json.dump(_plain(gen_scenarios(alan_mod, env_mod)), f)
    for name, n, act, seed, rec in ALAN_RUNS:
        actions = None if act is None else read_act(act)
        r = gen_alan_run(alan_mod, name, n, actions, seed, rec, mode=1)
        np.savez_compressed(os.path.join(HERE, "shell_alan_%s%d.npz" % (name, n)), **r)
        print("alan", name, n, "steps", r["steps"], "result", r["result"])
    for name, n, seed, rec in ORCA_RUNS:
        r = gen_alan_run(alan_mod, name, n, None, seed, rec, mode=0)
        np.savez_compressed(os.path.join(HERE, "shell_orca_%s%d.npz" % (name, n)), **r)
        print("orca", name, n, "steps", r["steps"], "result", r["result"])
    with contextlib.redirect_stdout(io.StringIO()):      # the env prints episode_time once done (:413-414)
        np.savez_compressed(os.path.join(HERE, "shell_env.npz"), **gen_env_run(env_mod))
        # a small world that runs to done['__all__'] (all agents behind x < 2, :352-365,404)
        np.savez_compressed(os.path.join(HERE, "shell_env_small.npz"),
                            **gen_env_run(env_mod, seed=303, n=2, steps_a=1000, steps_b=30, steps_orca=0,
                                          stop_on_done=True))
    with gzip.open(os.path.join(HERE, "shell_calltrace.json.gz"), "wt") as f:
        json.dump(gen_calltrace(alan_mod, env_mod), f)
    with open(os.path.join(HERE, "shell_mcmc.json"), "w") as f:
        json.dump(gen_mcmc(train_mod), f)


if __name__ == "__main__":
    main()
