"""Batched RVO2-style simulator: the tensor API over the C ABI.

``BatchedRVOSimulator`` owns the state of ``num_envs`` independent worlds of
``agents_per_env`` agents as torch CUDA tensors (structure of arrays, ``[E, N, 2]`` float32)
and steps all of them with one kernel launch.  Its method names follow the
``rvo2.PyRVOSimulator`` calls the reference uses (SURVEY.md 8b) -- ``doStep``,
``setAgentPrefVelocity`` ... -- but operate on whole batches; the scalar, tuple-in/tuple-out
drop-in for a single world is ``rvo2_compat.PyRVOSimulator``.

torch is plumbing here (device memory + streams); all arithmetic happens in
``liborca_b200.so``.  There is no fallback path.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib


def _dev_index(device) -> int:
    device = torch.device(device)
    if device.type != "cuda":
        raise ValueError("BatchedRVOSimulator needs a CUDA device (there is no CPU path)")
    return torch.cuda.current_device() if device.index is None else device.index


class BatchedRVOSimulator:
    """Batch of ORCA worlds on one GPU.

    Constructor arguments are those of ``rvo2.PyRVOSimulator`` (ALAN_true.py:22-28) plus the
    batch shape.  They are every agent's parameters, as everywhere in the reference
    (collision_avoidence_env.py:126-133, ALAN_true.py:461-468), until ``set_agent_params`` gives
    agents their own neighborDist, maxNeighbors, timeHorizon, timeHorizonObst, radius and maxSpeed
    (RVO2's per-agent addAgent arguments).  The time step, the done test's 2 * radius and
    ``observe`` stay those of the constructor.
    """

    def __init__(self, num_envs: int, agents_per_env: int, timeStep: float, neighborDist: float, maxNeighbors: int,
                 timeHorizon: float, timeHorizonObst: float, radius: float, maxSpeed: float, device="cuda:0"):
        self._L = _lib.load()
        self.device = torch.device(device)
        self.device_index = _dev_index(device)
        self.num_envs = int(num_envs)
        self.agents_per_env = int(agents_per_env)
        self.params = _lib.OrcaParams(float(timeStep), float(neighborDist), int(maxNeighbors), float(timeHorizon),
                                      float(timeHorizonObst), float(radius), float(maxSpeed))
        h = ctypes.c_void_p()
        _lib.check(self._L.orca_create(ctypes.byref(self.params), self.device_index, self.num_envs,
                                       self.agents_per_env, ctypes.byref(h)))
        self._h = h
        E, N = self.num_envs, self.agents_per_env
        dev = torch.device("cuda", self.device_index)
        self.pos = torch.zeros(E, N, 2, dtype=torch.float32, device=dev)
        self.vel = torch.zeros(E, N, 2, dtype=torch.float32, device=dev)
        self.pref = torch.zeros(E, N, 2, dtype=torch.float32, device=dev)
        self.stats = torch.zeros(_lib.STAT_COUNT, dtype=torch.int64, device=dev)
        # neighbor lists of the last step that asked for them (SURVEY Q3 semantics)
        self.nbr_idx: Optional[torch.Tensor] = None
        self.nbr_cnt: Optional[torch.Tensor] = None
        self.obst_nbr_idx: Optional[torch.Tensor] = None
        self.obst_nbr_cnt: Optional[torch.Tensor] = None
        self._obst_vertex_cache = {}
        self._roadmap_shape = None  # (R, G) of the roadmap set by set_roadmap

    # ------------------------------------------------------------------ lifecycle
    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._L.orca_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def max_neighbors(self) -> int:
        return self.params.max_neighbors

    @property
    def time_step(self) -> float:
        return self.params.time_step

    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device_index).cuda_stream)

    @staticmethod
    def _p(t: Optional[torch.Tensor]):
        return None if t is None else ctypes.c_void_p(t.data_ptr())

    def _check_state(self, t: torch.Tensor, shape, dtype, name):
        if t.dtype != dtype or tuple(t.shape) != tuple(shape) or not t.is_contiguous() or not t.is_cuda:
            raise ValueError(f"{name} must be a contiguous CUDA {dtype} tensor of shape {tuple(shape)}, "
                             f"got {t.dtype} {tuple(t.shape)}")

    # ------------------------------------------------------------------ per-agent parameters
    _AGENT_PARAMS = (("neighbor_dist", np.float32), ("max_neighbors", np.int32), ("time_horizon", np.float32),
                     ("time_horizon_obst", np.float32), ("radius", np.float32), ("max_speed", np.float32))

    def set_agent_params(self, neighbor_dist=None, max_neighbors=None, time_horizon=None, time_horizon_obst=None,
                         radius=None, max_speed=None):
        """Per-agent ORCA parameters (RVO2's addAgent / setAgent{NeighborDist,MaxNeighbors,TimeHorizon,
        TimeHorizonObst,Radius,MaxSpeed}).  Each argument is an ``[E, N]`` array or tensor (CPU or CUDA),
        copied to the host once; ``None`` = the constructor's value for every agent.  All ``None``
        returns to uniform parameters.  ``max_neighbors`` must lie in [0, maxNeighbors of the
        constructor]; time horizons must be > 0, the others >= 0, all finite (``ValueError``).
        Synchronises with the device, like ``set_obstacles``."""
        given = dict(neighbor_dist=neighbor_dist, max_neighbors=max_neighbors, time_horizon=time_horizon,
                     time_horizon_obst=time_horizon_obst, radius=radius, max_speed=max_speed)
        shape = (self.num_envs, self.agents_per_env)
        arrays = {}
        for name, dtype in self._AGENT_PARAMS:
            v = given[name]
            if v is None:
                arrays[name] = None
                continue
            if isinstance(v, torch.Tensor):
                v = v.detach().cpu().numpy()
            v = np.asarray(v)
            if tuple(v.shape) != shape:
                raise ValueError(f"{name} must have shape {shape}, got {tuple(v.shape)}")
            if dtype is np.int32 and not np.issubdtype(v.dtype, np.integer):
                raise ValueError(f"{name} must be integral, got {v.dtype}")
            arrays[name] = np.ascontiguousarray(v, dtype)
        ptr = lambda a: None if a is None else a.ctypes.data
        _lib.check(self._L.orca_set_agent_params(self._h, *(ptr(arrays[n]) for n, _ in self._AGENT_PARAMS)))

    # ------------------------------------------------------------------ obstacles
    def set_obstacles(self, polygons: Sequence, per_env: bool = False):
        """addObstacle(...) for every polygon, then processObstacles().

        ``polygons``: list of polygons (each a list of (x, y)), shared by all envs; or, with
        ``per_env=True``, a list of ``num_envs`` such lists.  Vertex order follows RVO2: the
        visible side of an edge is its right side (collision_avoidence_env.py:139-141)."""
        worlds = polygons if per_env else [polygons]
        if per_env and len(worlds) != self.num_envs:
            raise ValueError("per_env=True needs one polygon list per env")
        flat, sizes, counts = [], [], []
        for w in worlds:
            counts.append(len(w))
            for poly in w:
                arr = np.asarray(poly, dtype=np.float32).reshape(-1, 2)
                flat.append(arr)
                sizes.append(arr.shape[0])
        xy = np.ascontiguousarray(np.concatenate(flat) if flat else np.zeros((0, 2), np.float32))
        sizes_a = np.asarray(sizes, np.int32)
        counts_a = np.asarray(counts, np.int32)
        _lib.check(self._L.orca_set_obstacles(self._h, xy.ctypes.data, sizes_a.ctypes.data, len(sizes),
                                              counts_a.ctypes.data if per_env else None))
        self._obst_vertex_cache = {}

    def obstacle_vertices(self, env: int = 0):
        """Processed vertex table of one world: (points[V,2], next[V], prev[V], convex[V])."""
        if env in self._obst_vertex_cache:
            return self._obst_vertex_cache[env]
        n = _lib.check(self._L.orca_obstacle_vertex_count(self._h, int(env)))
        xy = np.zeros((n, 2), np.float32)
        nxt = np.zeros(n, np.int32)
        prv = np.zeros(n, np.int32)
        cvx = np.zeros(n, np.int32)
        if n:
            _lib.check(self._L.orca_get_obstacle_vertices(self._h, int(env), xy.ctypes.data, nxt.ctypes.data,
                                                          prv.ctypes.data, cvx.ctypes.data))
        self._obst_vertex_cache[env] = (xy, nxt, prv, cvx)
        return self._obst_vertex_cache[env]

    # ------------------------------------------------------------------ line of sight and roadmaps
    def query_visibility(self, p1: torch.Tensor, p2: torch.Tensor, radius=0.0) -> torch.Tensor:
        """RVO2's queryVisibility for a batch: ``p1``, ``p2`` are ``[E, Q, 2]`` CUDA float32, ``radius`` a
        float or an ``[E, Q]`` CUDA float32 tensor.  Returns a bool tensor ``[E, Q]``: whether a disc of
        the radius moves from p1 to p2 without crossing an obstacle edge of the env's world."""
        E = self.num_envs
        if p1.dim() != 3 or p1.shape[0] != E or p1.shape[2] != 2:
            raise ValueError(f"p1 must have shape [{E}, Q, 2], got {tuple(p1.shape)}")
        Q = p1.shape[1]
        self._check_state(p1, (E, Q, 2), torch.float32, "p1")
        self._check_state(p2, (E, Q, 2), torch.float32, "p2")
        r_dev, r = None, 0.0
        if isinstance(radius, torch.Tensor):
            self._check_state(radius, (E, Q), torch.float32, "radius")
            r_dev = radius
        else:
            r = float(radius)
        out = torch.empty(E, Q, dtype=torch.uint8, device=self.pos.device)
        _lib.check(self._L.orca_query_visibility(self._h, self._p(p1), self._p(p2), self._p(r_dev), r, int(Q),
                                                 self._p(out), self._stream()))
        return out.view(torch.bool)

    def set_roadmap(self, vertices, num_goals: int, radius: Optional[float] = None):
        """Roadmap of RVO2's obstacle example (Roadmap.cpp buildRoadmap): ``vertices`` is ``[R, 2]``
        (shared by every env) or ``[E, R, 2]`` (one roadmap per env), array or tensor; its first
        ``num_goals`` vertices are the goals.  Edges join vertices that see each other for a disc of
        ``radius`` (default: the constructor's radius); distances to every goal are computed on the
        device, and again after every ``set_obstacles``.  ``R = 0`` removes the roadmap.  At most 512
        vertices and 1 <= num_goals <= R (``NotImplementedError``).  Synchronises."""
        if isinstance(vertices, torch.Tensor):
            vertices = vertices.detach().cpu().numpy()
        v = np.ascontiguousarray(np.asarray(vertices, np.float32))
        if v.ndim == 3:
            if v.shape[0] != self.num_envs or v.shape[2] != 2:
                raise ValueError(f"per-env roadmap vertices must have shape [{self.num_envs}, R, 2], got {v.shape}")
            per_env, R = True, v.shape[1]
        elif v.ndim == 2 and v.shape[1] == 2:
            per_env, R = False, v.shape[0]
        else:
            raise ValueError(f"roadmap vertices must have shape [R, 2] or [E, R, 2], got {v.shape}")
        r = self.params.radius if radius is None else float(radius)
        _lib.check(self._L.orca_set_roadmap(self._h, v.ctypes.data if R else None, int(R), int(num_goals),
                                            1 if per_env else 0, r))
        self._roadmap_shape = (R, int(num_goals)) if R else None

    def roadmap(self, env: int = 0):
        """The roadmap tables of one env: (adjacency bool [R, R], row u column v = edge u -> v;
        distances float32 [G, R], 9e9 when unreachable)."""
        if self._roadmap_shape is None:
            raise RuntimeError("no roadmap is set")
        R, G = self._roadmap_shape
        words = (R + 31) // 32
        adj = np.zeros((R, words), np.uint32)
        dist = np.zeros((G, R), np.float32)
        _lib.check(self._L.orca_get_roadmap(self._h, int(env), adj.ctypes.data, dist.ctypes.data))
        bits = np.unpackbits(adj.view(np.uint8).reshape(R, words * 4), axis=1, bitorder="little")[:, :R]
        return bits.astype(bool), dist

    def roadmap_pref_velocity(self, goal_vertex: torch.Tensor, pos: Optional[torch.Tensor] = None,
                              out: Optional[torch.Tensor] = None, return_vertex: bool = False):
        """Roadmap.cpp's preferred velocities (without the perturbation) toward each agent's goal vertex
        (``goal_vertex``: ``[E, N]`` CUDA int32, ids in [0, num_goals); others give (0, 0) and vertex -1),
        from ``pos`` (default: the current positions).  Writes ``self.pref`` unless ``out`` is given, so
        that ``env_step(policy=POLICY_EXTERNAL)`` / ``doStep()`` steps with it.  Returns the preferred
        velocities, and the chosen vertex ids ``[E, N]`` int32 with ``return_vertex``."""
        E, N = self.num_envs, self.agents_per_env
        pos = self.pos if pos is None else pos
        out = self.pref if out is None else out
        self._check_state(goal_vertex, (E, N), torch.int32, "goal_vertex")
        self._check_state(pos, (E, N, 2), torch.float32, "pos")
        self._check_state(out, (E, N, 2), torch.float32, "out")
        vertex = torch.empty(E, N, dtype=torch.int32, device=self.pos.device) if return_vertex else None
        _lib.check(self._L.orca_roadmap_pref_velocity(self._h, self._p(pos), self._p(goal_vertex), self._p(out),
                                                      self._p(vertex), self._stream()))
        return (out, vertex) if return_vertex else out

    # ------------------------------------------------------------------ batched rvo2 calls
    def setAgentPosition(self, pos):
        self.pos.copy_(torch.as_tensor(pos, dtype=torch.float32).reshape(self.pos.shape))

    def setAgentVelocity(self, vel):
        self.vel.copy_(torch.as_tensor(vel, dtype=torch.float32).reshape(self.vel.shape))

    def setAgentPrefVelocity(self, pref):
        self.pref.copy_(torch.as_tensor(pref, dtype=torch.float32).reshape(self.pref.shape))

    def getAgentPosition(self) -> torch.Tensor:
        return self.pos

    def getAgentVelocity(self) -> torch.Tensor:
        return self.vel

    def getAgentPrefVelocity(self) -> torch.Tensor:
        return self.pref

    def doStep(self):
        """One RVO2 doStep for every env, in place on ``self.pos`` / ``self.vel``."""
        _lib.check(self._L.orca_step(self._h, self._p(self.pos), self._p(self.vel), self._p(self.pref),
                                     self._stream()))

    def _alloc_neighbor_outputs(self):
        if self.nbr_idx is None:
            E, N, k = self.num_envs, self.agents_per_env, max(1, self.max_neighbors)
            dev = self.pos.device
            self.nbr_idx = torch.full((E, N, k), -1, dtype=torch.int32, device=dev)
            self.nbr_cnt = torch.zeros(E, N, dtype=torch.int32, device=dev)
            self.obst_nbr_idx = torch.full((E, N, _lib.MAX_OBST_NEIGHBORS), -1, dtype=torch.int32, device=dev)
            self.obst_nbr_cnt = torch.zeros(E, N, dtype=torch.int32, device=dev)

    def neighbors(self, pos: Optional[torch.Tensor] = None, with_distsq: bool = False):
        """Neighbor search only (parity hook).  Returns (nbr_idx, nbr_cnt, obst_nbr_idx, obst_nbr_cnt[, distsq])."""
        self._alloc_neighbor_outputs()
        pos = self.pos if pos is None else pos
        self._check_state(pos, self.pos.shape, torch.float32, "pos")
        dsq = torch.zeros_like(self.nbr_idx, dtype=torch.float32) if with_distsq else None
        _lib.check(self._L.orca_neighbors(self._h, self._p(pos), self._p(self.nbr_idx), self._p(dsq),
                                          self._p(self.nbr_cnt), self._p(self.obst_nbr_idx),
                                          self._p(self.obst_nbr_cnt), self._stream()))
        out = (self.nbr_idx, self.nbr_cnt, self.obst_nbr_idx, self.obst_nbr_cnt)
        return out + (dsq,) if with_distsq else out

    def orca_lines(self, pos: Optional[torch.Tensor] = None, vel: Optional[torch.Tensor] = None,
                   max_lines: Optional[int] = None):
        """The ORCA half-planes every agent solves in the NEXT step from the state ``(pos, vel)``
        (default: the current ``self.pos`` / ``self.vel``) -- RVO2's getAgentNumORCALines /
        getAgentORCALine for the whole batch.  To record what a step solves, call this before stepping.

        Returns device tensors ``(lines [E, N, L, 4] float32, count [E, N] int32, n_obst [E, N] int32)``.
        Row ``j`` of an agent is ``(point.x, point.y, direction.x, direction.y)``: its ``n_obst`` obstacle
        lines first, then one line per agent neighbor in ascending (distSq, id) order, bit for bit the
        programme of the step.  ``L = max_lines`` (default ``maxNeighbors + 6``, the obstacle lines of the
        step's fast path); rows past ``L`` are absent, which ``count > L`` shows, and rows at and past
        ``count`` are zero.  ``count = -1``: more than 64 obstacle lines (the step's overflow statistic).
        The lines do not depend on the preferred velocity.  Writes nothing a step reads."""
        E, N = self.num_envs, self.agents_per_env
        pos = self.pos if pos is None else pos
        vel = self.vel if vel is None else vel
        self._check_state(pos, (E, N, 2), torch.float32, "pos")
        self._check_state(vel, (E, N, 2), torch.float32, "vel")
        if pos.device != self.pos.device or vel.device != self.pos.device:
            raise ValueError(f"pos and vel must live on {self.pos.device}")
        L = self.max_neighbors + _lib.MAX_OBST_LINES if max_lines is None else int(max_lines)
        if L < 0:
            raise ValueError(f"max_lines must be >= 0, got {L}")
        dev = self.pos.device
        lines = torch.zeros(E, N, L, 4, dtype=torch.float32, device=dev)
        count = torch.empty(E, N, dtype=torch.int32, device=dev)
        n_obst = torch.empty(E, N, dtype=torch.int32, device=dev)
        _lib.check(self._L.orca_agent_lines(self._h, self._p(pos), self._p(vel), L, self._p(lines) if L else None,
                                            self._p(count), self._p(n_obst), self._stream()))
        return lines, count, n_obst

    # ------------------------------------------------------------------ fused env step
    def env_step(self, *, policy: int, goal: Optional[torch.Tensor] = None, goal2: Optional[torch.Tensor] = None,
                 done_mode: int = _lib.DONE_NONE, action_theta: Optional[torch.Tensor] = None,
                 rl_reward_scale: float = 0.3, done_x_threshold: float = 2.0,
                 alan_weights: Optional[torch.Tensor] = None, alan_actions: Optional[torch.Tensor] = None,
                 alan_action_out: Optional[torch.Tensor] = None, alan_uniform: Optional[torch.Tensor] = None,
                 alan_num_actions_env: Optional[torch.Tensor] = None,
                 alan_window_steps: int = 121, alan_gamma: float = 0.6, alan_temp: float = 0.2, rng_seed: int = 0,
                 reward: Optional[torch.Tensor] = None, agent_done: Optional[torch.Tensor] = None,
                 arrival_time: Optional[torch.Tensor] = None, env_step: Optional[torch.Tensor] = None,
                 env_done_cnt: Optional[torch.Tensor] = None, want_neighbors: bool = False,
                 collect_stats: bool = True, steps: int = 1):
        """One fused step: policy -> doStep -> reward -> done test -> bandit update (orca_env_step)."""
        E, N = self.num_envs, self.agents_per_env
        a = _lib.OrcaEnvStepArgs()
        a.struct_size = ctypes.sizeof(_lib.OrcaEnvStepArgs)
        a.policy, a.done_mode = int(policy), int(done_mode)
        a.pos_dev, a.vel_dev = self.pos.data_ptr(), self.vel.data_ptr()
        if policy == _lib.POLICY_EXTERNAL:
            a.pref_dev = self.pref.data_ptr()
        if goal is not None:
            self._check_state(goal, (E, N, 2), torch.float32, "goal")
            a.goal_dev = goal.data_ptr()
        if goal2 is not None:
            self._check_state(goal2, (E, N, 2), torch.float32, "goal2")
            a.goal2_dev = goal2.data_ptr()
        if action_theta is not None:
            self._check_state(action_theta, (E, N), torch.float32, "action_theta")
            a.action_theta_dev = action_theta.data_ptr()
        a.rl_reward_scale, a.done_x_threshold = float(rl_reward_scale), float(done_x_threshold)
        if alan_weights is not None:
            # alan_actions: [A, 2] shared by all envs, or [E, A, 2] one table per env
            A = alan_actions.shape[-2]
            self._check_state(alan_weights, (E, N, A), torch.float32, "alan_weights")
            if alan_actions.dim() == 3:
                self._check_state(alan_actions, (E, A, 2), torch.float32, "alan_actions")
                a.alan_actions_env_stride = A
                if alan_num_actions_env is not None:
                    self._check_state(alan_num_actions_env, (E,), torch.int32, "alan_num_actions_env")
                    a.alan_num_actions_env_dev = alan_num_actions_env.data_ptr()
            else:
                self._check_state(alan_actions, (A, 2), torch.float32, "alan_actions")
            a.alan_weights_dev, a.alan_actions_dev, a.alan_num_actions = alan_weights.data_ptr(), alan_actions.data_ptr(), A
            if alan_action_out is not None:
                self._check_state(alan_action_out, (E, N), torch.uint8, "alan_action_out")
                a.alan_action_out_dev = alan_action_out.data_ptr()
            if alan_uniform is not None:
                self._check_state(alan_uniform, (E, N), torch.float32, "alan_uniform")
                a.alan_uniform_in_dev = alan_uniform.data_ptr()
        a.alan_window_steps, a.alan_gamma, a.alan_temp = int(alan_window_steps), float(alan_gamma), float(alan_temp)
        a.rng_seed = int(rng_seed) & 0xFFFFFFFFFFFFFFFF
        if reward is not None:
            self._check_state(reward, (E, N), torch.float32, "reward")
            a.reward_dev = reward.data_ptr()
        if agent_done is not None:
            self._check_state(agent_done, (E, N), torch.uint8, "agent_done")
            a.agent_done_dev = agent_done.data_ptr()
        if arrival_time is not None:
            self._check_state(arrival_time, (E, N), torch.float32, "arrival_time")
            a.arrival_time_dev = arrival_time.data_ptr()
        if env_step is not None:
            self._check_state(env_step, (E,), torch.int32, "env_step")
            a.env_step_dev = env_step.data_ptr()
        if env_done_cnt is not None:
            self._check_state(env_done_cnt, (E,), torch.int32, "env_done_cnt")
            a.env_done_cnt_dev = env_done_cnt.data_ptr()
        if want_neighbors:
            self._alloc_neighbor_outputs()
            a.nbr_idx_dev, a.nbr_cnt_dev = self.nbr_idx.data_ptr(), self.nbr_cnt.data_ptr()
            a.obst_nbr_idx_dev, a.obst_nbr_cnt_dev = self.obst_nbr_idx.data_ptr(), self.obst_nbr_cnt.data_ptr()
        if collect_stats:
            a.stats_dev = self.stats.data_ptr()
        if steps == 1:
            _lib.check(self._L.orca_env_step(self._h, ctypes.byref(a), self._stream()))
        else:  # back-to-back launches issued from C (orca_env_step_many): no Python in between
            _lib.check(self._L.orca_env_step_many(self._h, ctypes.byref(a), int(steps), self._stream()))

    # ------------------------------------------------------------------ observation
    def observe(self, goal: torch.Tensor, obs: Optional[torch.Tensor] = None, laser_num: int = 16,
                circle_approx_num: int = 8) -> torch.Tensor:
        """Laser-scan observation of every agent ([E, N, laser_num * 4] float32), from the current
        positions / velocities and the neighbor lists of the last step that recorded them
        (``env_step(want_neighbors=True)`` or ``neighbors()``) -- collision_avoidence_env.py:231-318."""
        E, N = self.num_envs, self.agents_per_env
        self._alloc_neighbor_outputs()
        self._check_state(goal, (E, N, 2), torch.float32, "goal")
        if obs is None:
            obs = torch.empty(E, N, laser_num * 4, dtype=torch.float32, device=self.pos.device)
        self._check_state(obs, (E, N, laser_num * 4), torch.float32, "obs")
        _lib.check(self._L.orca_observe(self._h, self._p(self.pos), self._p(self.vel), self._p(goal),
                                        self._p(self.nbr_idx), self._p(self.nbr_cnt), self._p(self.obst_nbr_idx),
                                        self._p(self.obst_nbr_cnt), int(laser_num), int(circle_approx_num),
                                        self._p(obs), self._stream()))
        return obs

    # ------------------------------------------------------------------ host-buffer (e2e) path
    def step_host(self, pos_host: torch.Tensor, vel_host: Optional[torch.Tensor], pref_or_goal_host: torch.Tensor,
                  policy: int = _lib.POLICY_EXTERNAL, upload_state: bool = True, steps: int = 1,
                  aux_unchanged: bool = False):
        """orca_step_host_ex: host buffers in, host buffers out, copies inside the call.
        ``vel_host=None`` writes only the positions back; ``aux_unchanged`` promises that the goal /
        pref buffer still holds what it held at the previous call (nothing is read from the host)."""
        for t, name in ((pos_host, "pos_host"), (vel_host, "vel_host"), (pref_or_goal_host, "pref_or_goal_host")):
            if t is None and name == "vel_host":
                continue
            if t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous() or t.numel() != self.pos.numel():
                raise ValueError(f"{name} must be a contiguous CPU float32 tensor with {self.pos.numel()} elements")
        flags = (_lib.HOST_UPLOAD_STATE if upload_state else 0) | (_lib.HOST_AUX_UNCHANGED if aux_unchanged else 0)
        _lib.check(self._L.orca_step_host_ex(self._h, pos_host.data_ptr(), None if vel_host is None else vel_host.data_ptr(),
                                             pref_or_goal_host.data_ptr(), int(policy), int(flags), int(steps)))

    def launch_count(self) -> int:
        return int(self._L.orca_launch_count(self._h))

    def check_overflow(self):
        """Raises if any agent exceeded even the uncapped path's capacity (ORCA_SLOW_MAX_OBST = 64
        obstacle edges in range / obstacle lines): from then on an obstacle constraint is missing from
        that agent's linear program, which RVO2 never allows.  Cannot happen for obstacle worlds of at
        most 64 processed vertices (every world of the reference has fewer)."""
        n = int(self.stats[_lib.STAT_OVERFLOW].item())
        if n:
            raise RuntimeError(f"{n} agent-steps exceeded the obstacle capacity of the step kernel (64 edges / lines per "
                               "agent): results are no longer RVO2's; simplify the obstacle world")

    def read_stats(self, allow_overflow: bool = False) -> dict:
        if not allow_overflow:
            self.check_overflow()
        s = self.stats.cpu()
        f = s.view(torch.float64)
        return {
            "agent_steps": int(s[_lib.STAT_AGENT_STEPS]), "sum_reward": float(f[_lib.STAT_SUM_REWARD]),
            "finished": int(s[_lib.STAT_FINISHED]), "collisions": int(s[_lib.STAT_COLLISIONS]),
            "lp3_calls": int(s[_lib.STAT_LP3_CALLS]), "overflow": int(s[_lib.STAT_OVERFLOW]),
            "sum_arrival": float(f[_lib.STAT_SUM_ARRIVAL]), "sum_arrival2": float(f[_lib.STAT_SUM_ARRIVAL2]),
        }
