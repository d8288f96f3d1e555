"""Scalar drop-in for ``rvo2.PyRVOSimulator`` (one world) on top of the batched CUDA simulator.

The reference shells talk to RVO2 through 16 methods with Python tuples in and out
(SURVEY.md 8b: collision_avoidence_env.py:62-68,123-148,154-157,237-252,283-312,385,479 and
ALAN_true.py:22-28,461-479,490,553,598-613).  This class offers exactly those, so
``sys.modules['rvo2'] = collision_avoidance_b200.rvo2_compat`` lets the reference's shell logic
run unmodified against the CUDA path (tests/test_gpu_compat.py replays the recorded call trace of the unmodified shells against it).  It is a
compatibility shim, not the fast path: every ``doStep`` is one kernel launch for one world plus
host<->device mirrors; throughput comes from ``BatchedRVOSimulator`` / ``envs`` / ``alan``.

Agents may have parameters of their own, as in RVO2: ``addAgent`` takes all six per agent, and
``getAgent``/``setAgent`` ``NeighborDist``, ``MaxNeighbors``, ``TimeHorizon``, ``TimeHorizonObst``,
``Radius`` and ``MaxSpeed`` read and change them between steps.  A world whose agents all share one
set runs the uniform kernels; a mixed one uploads its per-agent table before the next ``doStep``.

``getAgentNumORCALines(i)`` / ``getAgentORCALine(i, j)`` return the ORCA half-planes agent i solved in
the last ``doStep``, as in RVO2.  They are computed on the first query after a step (from the pre-step
state the shim keeps), so ``doStep`` costs nothing more for callers that never ask; a call that would
change what the device computes (``addAgent``, ``addObstacle``, ``processObstacles``, a ``setAgent*``
parameter setter) computes them first.

``queryVisibility(point1, point2, radius)`` answers RVO2's line-of-sight query on the processed
obstacles (True before ``processObstacles``, as in RVO2); roadmap navigation for whole batches is
``BatchedRVOSimulator.set_roadmap`` / ``roadmap_pref_velocity``.

Restrictions (checked, never silent): ``maxNeighbors <= 16``.
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import numpy as np
import torch

from . import _lib
from .sim import BatchedRVOSimulator


class PyRVOSimulator:
    def __init__(self, timeStep, neighborDist, maxNeighbors, timeHorizon, timeHorizonObst, radius, maxSpeed,
                 velocity=(0.0, 0.0), device="cuda:0"):
        self._time_step = float(timeStep)
        self._defaults = (float(neighborDist), int(maxNeighbors), float(timeHorizon), float(timeHorizonObst),
                          float(radius), float(maxSpeed))
        self._default_velocity = (float(velocity[0]), float(velocity[1]))
        self._device = device
        self._params: List[Tuple] = []     # per agent: (neighborDist, maxNeighbors, timeHorizon, timeHorizonObst, radius, maxSpeed)
        self._params_dirty = True          # the table on the device (if any) is older than self._params
        self._sim_params: Optional[Tuple] = None  # the OrcaParams the current simulator was built with
        self._table_set = False
        self._pos: List[Tuple[float, float]] = []
        self._vel: List[Tuple[float, float]] = []
        self._pref: List[Tuple[float, float]] = []
        self._polygons: List[np.ndarray] = []
        self._processed = False
        self._sim: Optional[BatchedRVOSimulator] = None
        self._dirty = True            # host state newer than device state
        self._nbr_host = None         # (nbr_idx, nbr_cnt, obst_idx, obst_cnt) of the last doStep
        # ORCA lines of the last doStep: its pre-step (pos, vel) until the first query or mutation, then
        # the host copy (lines [n, L, 4], count [n], n_obst [n]) for the n agents the step had
        self._lines_pending = None
        self._lines_host = None
        self._global_time = 0.0
        self._vertex_table = None

    # ------------------------------------------------------------------ construction
    def addAgent(self, pos, neighborDist=None, maxNeighbors=None, timeHorizon=None, timeHorizonObst=None,
                 radius=None, maxSpeed=None, velocity=None):
        opt = (neighborDist, maxNeighbors, timeHorizon, timeHorizonObst, radius, maxSpeed, velocity)
        if all(o is None for o in opt):
            params, vel = self._defaults, self._default_velocity
        elif any(o is None for o in opt):
            raise ValueError("Either pass only 'pos', or pass all parameters.")
        else:
            params = (float(neighborDist), int(maxNeighbors), float(timeHorizon), float(timeHorizonObst),
                      float(radius), float(maxSpeed))
            vel = (float(velocity[0]), float(velocity[1]))
        self._materialize_lines()
        self._params.append(tuple(self._f32(x) if i != 1 else x for i, x in enumerate(params)))
        self._params_dirty = True
        self._pos.append((float(np.float32(pos[0])), float(np.float32(pos[1]))))
        self._vel.append((float(np.float32(vel[0])), float(np.float32(vel[1]))))
        self._pref.append((0.0, 0.0))
        self._sim = None  # shape changed: rebuild lazily
        self._dirty = True
        return len(self._pos) - 1

    def addObstacle(self, vertices):
        arr = np.asarray(vertices, dtype=np.float32).reshape(-1, 2)
        if arr.shape[0] < 2:
            raise RuntimeError("Error adding obstacle to RVO simulation")
        self._materialize_lines()
        first = sum(p.shape[0] for p in self._polygons)
        self._polygons.append(arr)
        self._processed = False
        self._vertex_table = None
        return first

    def processObstacles(self):
        self._materialize_lines()
        self._processed = True
        self._vertex_table = None
        if self._sim is not None:
            self._sim.set_obstacles([p for p in self._polygons])

    # ------------------------------------------------------------------ device plumbing
    @staticmethod
    def _f32(x) -> float:
        return float(np.float32(x))

    def _handle_params(self):
        """(OrcaParams of the simulator, whether the agents need a per-agent table).  Shared
        parameters are the simulator's own; otherwise the first agent's, with the largest maxNeighbors."""
        first = self._params[0]
        if all(p == first for p in self._params):
            return first, False
        return (first[0], max(p[1] for p in self._params)) + first[2:], True

    def _ensure_sim(self) -> BatchedRVOSimulator:
        if not self._pos:
            raise RuntimeError("no agents in the simulation")
        if self._params_dirty:
            self._materialize_lines()  # the last step's lines come from the parameters it ran with
        hp, hetero = self._handle_params()
        if self._sim is not None and hp != self._sim_params:
            self._sim = None  # another maxNeighbors bound (or another shared set): rebuild
        if self._sim is None:
            nd, k, th, tho, r, vmax = hp
            self._sim = BatchedRVOSimulator(1, len(self._pos), self._time_step, nd, k, th, tho, r, vmax,
                                            device=self._device)
            self._sim_params = hp
            self._table_set = False
            self._params_dirty = True
            if self._processed:
                self._sim.set_obstacles([p for p in self._polygons])
            self._dirty = True
        if self._params_dirty:
            if hetero:
                cols = list(zip(*self._params))
                self._sim.set_agent_params(
                    *(np.asarray(c, np.int32 if j == 1 else np.float32).reshape(1, -1) for j, c in enumerate(cols)))
                self._table_set = True
            elif self._table_set:
                self._sim.set_agent_params()
                self._table_set = False
            self._params_dirty = False
        return self._sim

    def _obstacle_sim(self):
        """(simulator holding the processed obstacles, whether it is a throw-away one): with no agents
        yet, a 1-agent world built just to run the BSP."""
        if self._pos:
            return self._ensure_sim(), False
        tmp = BatchedRVOSimulator(1, 1, self._time_step, *self._defaults, device=self._device)
        tmp.set_obstacles([p for p in self._polygons])
        return tmp, True

    def _vertices(self):
        """Vertex table after processObstacles (BSP splits may have appended vertices)."""
        if self._vertex_table is None:
            if self._processed:
                sim, temporary = self._obstacle_sim()
                self._vertex_table = sim.obstacle_vertices(0)
                if temporary:
                    sim.close()
            else:
                pts = np.concatenate(self._polygons) if self._polygons else np.zeros((0, 2), np.float32)
                nxt, prv, off = [], [], 0
                for p in self._polygons:
                    n = p.shape[0]
                    nxt += [off + (i + 1) % n for i in range(n)]
                    prv += [off + (i - 1) % n for i in range(n)]
                    off += n
                self._vertex_table = (pts, np.asarray(nxt, np.int32), np.asarray(prv, np.int32),
                                      np.ones(len(nxt), np.int32))
        return self._vertex_table

    def doStep(self):
        sim = self._ensure_sim()
        if self._dirty:
            sim.pos.copy_(torch.tensor(self._pos, dtype=torch.float32).reshape(1, -1, 2))
            sim.vel.copy_(torch.tensor(self._vel, dtype=torch.float32).reshape(1, -1, 2))
        sim.pref.copy_(torch.tensor(self._pref, dtype=torch.float32).reshape(1, -1, 2))
        sim.env_step(policy=_lib.POLICY_EXTERNAL, want_neighbors=True, collect_stats=False)
        # the host lists are replaced below, never changed in place: they stay this step's input
        self._lines_pending = (self._pos, self._vel)
        self._lines_host = None
        pos = sim.pos[0].cpu().numpy()
        vel = sim.vel[0].cpu().numpy()
        self._pos = [(float(p[0]), float(p[1])) for p in pos]
        self._vel = [(float(v[0]), float(v[1])) for v in vel]
        self._nbr_host = (sim.nbr_idx[0].cpu().numpy(), sim.nbr_cnt[0].cpu().numpy(),
                          sim.obst_nbr_idx[0].cpu().numpy(), sim.obst_nbr_cnt[0].cpu().numpy())
        self._dirty = False
        self._global_time += self._time_step

    # ------------------------------------------------------------------ getters / setters
    def getAgentPosition(self, i):
        return self._pos[i]

    def getAgentVelocity(self, i):
        return self._vel[i]

    def getAgentPrefVelocity(self, i):
        return self._pref[i]

    def setAgentPrefVelocity(self, i, v):
        self._pref[i] = (float(np.float32(v[0])), float(np.float32(v[1])))

    def setAgentPosition(self, i, p):
        self._pos[i] = (float(np.float32(p[0])), float(np.float32(p[1])))
        self._dirty = True

    def setAgentVelocity(self, i, v):
        self._vel[i] = (float(np.float32(v[0])), float(np.float32(v[1])))
        self._dirty = True

    def getAgentNumAgentNeighbors(self, i):
        return 0 if self._nbr_host is None else int(self._nbr_host[1][i])

    def getAgentAgentNeighbor(self, i, j):
        if self._nbr_host is None or j >= int(self._nbr_host[1][i]):
            raise IndexError("neighbor index out of range")
        return int(self._nbr_host[0][i, j])

    def getAgentNumObstacleNeighbors(self, i):
        return 0 if self._nbr_host is None else int(self._nbr_host[3][i])

    def getAgentObstacleNeighbor(self, i, j):
        if self._nbr_host is None or j >= int(self._nbr_host[3][i]):
            raise IndexError("neighbor index out of range")
        return int(self._nbr_host[2][i, j])

    def _materialize_lines(self):
        """Compute the ORCA lines of the last doStep from its kept pre-step state, on the simulator
        (parameters, obstacles) it ran with."""
        if self._lines_pending is None:
            return
        pos, vel = self._lines_pending
        self._lines_pending = None
        sim = self._sim
        dev = sim.pos.device
        p = torch.tensor(pos, dtype=torch.float32, device=dev).reshape(1, -1, 2)
        v = torch.tensor(vel, dtype=torch.float32, device=dev).reshape(1, -1, 2)
        lines, count, n_obst = sim.orca_lines(p, v, max_lines=sim.max_neighbors + _lib.SLOW_MAX_OBST)
        self._lines_host = (lines[0].cpu().numpy(), count[0].cpu().numpy(), n_obst[0].cpu().numpy())

    def _num_lines(self, i):
        self._materialize_lines()
        if self._lines_host is None or i >= self._lines_host[1].shape[0]:
            return 0  # before the first doStep, or an agent added after it
        n = int(self._lines_host[1][i])
        if n < 0:
            raise RuntimeError(f"agent {i} has more than {_lib.SLOW_MAX_OBST} obstacle lines")
        return n

    def getAgentNumORCALines(self, i):
        """Number of ORCA half-planes agent i solved in the last doStep (0 before the first one)."""
        if not 0 <= i < len(self._pos):
            raise IndexError("agent index out of range")
        return self._num_lines(i)

    def getAgentORCALine(self, i, j):
        """Half-plane j of agent i in the last doStep as (point.x, point.y, direction.x, direction.y):
        obstacle lines first, then agent lines by ascending distance.  The flat tuple follows
        Python-RVO2's rvo2.pyx as far as it is known without its source at hand; the test suite pins it."""
        if not 0 <= i < len(self._pos) or not 0 <= j < self._num_lines(i):
            raise IndexError("ORCA line index out of range")
        ln = self._lines_host[0][i, j]
        return (float(ln[0]), float(ln[1]), float(ln[2]), float(ln[3]))

    def getNextObstacleVertexNo(self, v):
        return int(self._vertices()[1][v])

    def getPrevObstacleVertexNo(self, v):
        return int(self._vertices()[2][v])

    def getObstacleVertex(self, v):
        p = self._vertices()[0][v]
        return (float(p[0]), float(p[1]))

    # per-agent parameters (RVO2's getAgent* / setAgent*); a change takes effect at the next doStep
    def _set_param(self, i, j, value):
        self._materialize_lines()
        p = list(self._params[i])
        p[j] = int(value) if j == 1 else self._f32(value)
        self._params[i] = tuple(p)
        self._params_dirty = True

    def getAgentNeighborDist(self, i):
        return self._params[i][0]

    def getAgentMaxNeighbors(self, i):
        return self._params[i][1]

    def getAgentTimeHorizon(self, i):
        return self._params[i][2]

    def getAgentTimeHorizonObst(self, i):
        return self._params[i][3]

    def getAgentRadius(self, i):
        return self._params[i][4]

    def getAgentMaxSpeed(self, i):
        return self._params[i][5]

    def setAgentNeighborDist(self, i, neighborDist):
        self._set_param(i, 0, neighborDist)

    def setAgentMaxNeighbors(self, i, maxNeighbors):
        self._set_param(i, 1, maxNeighbors)

    def setAgentTimeHorizon(self, i, timeHorizon):
        self._set_param(i, 2, timeHorizon)

    def setAgentTimeHorizonObst(self, i, timeHorizonObst):
        self._set_param(i, 3, timeHorizonObst)

    def setAgentRadius(self, i, radius):
        self._set_param(i, 4, radius)

    def setAgentMaxSpeed(self, i, maxSpeed):
        self._set_param(i, 5, maxSpeed)

    def queryVisibility(self, point1, point2, radius=0.0):
        """Whether a disc of ``radius`` can move from point1 to point2 without crossing an obstacle edge
        (RVO2's queryVisibility).  True before processObstacles: RVO2 has no obstacle tree then."""
        if not self._processed:
            return True
        sim, temporary = self._obstacle_sim()
        dev = sim.pos.device
        q1 = torch.tensor([[[self._f32(point1[0]), self._f32(point1[1])]]], dtype=torch.float32, device=dev)
        q2 = torch.tensor([[[self._f32(point2[0]), self._f32(point2[1])]]], dtype=torch.float32, device=dev)
        visible = bool(sim.query_visibility(q1, q2, self._f32(radius)).item())
        if temporary:
            sim.close()
        return visible

    def getNumAgents(self):
        return len(self._pos)

    def getNumObstacleVertices(self):
        return int(self._vertices()[0].shape[0])

    def getGlobalTime(self):
        return self._global_time

    def getTimeStep(self):
        return self._time_step
