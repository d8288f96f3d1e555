"""Float64 restatement of the reference's per-step SHELL arithmetic (TEST INFRASTRUCTURE).

Restates, line for line in meaning (not in text), what the two Python shells of the reference
do around ``sim.doStep()``; every function cites the lines it follows.  The simulator behind
it is the CPU oracle (``oracle.rvo2_oracle.PyRVOSimulator``), reached through the same scalar
per-agent calls the reference makes.

  env  = collision_avoidance/envs/collision_avoidence_env.py   (paths in the reference project)
  ALAN = collision_avoidance/ALAN/ALAN_true.py
  util = collision_avoidance/envs/utils.py

Pinning: ``line_intersection`` / ``comp_laser`` below are checked against golden vectors
produced by importing the reference's own ``utils.py`` (tests/golden/make_laser_golden.py).
The rest of the shell has no runnable reference here (gym / ray / tkinter / rvo2 absent,
``time.clock`` removed): it is pinned by the known-answer tests in tests/ (Q7 period 121,
reward formulas, done rules).  Randomness: the reference draws from unseeded global RNGs
(SURVEY Q11); here every draw is an explicit input.
"""
from __future__ import annotations

from math import atan2, cos, pi, sin, sqrt

import numpy as np

from .rvo2_oracle import PyRVOSimulator


# ------------------------------------------------------------------------------------- util.py
def line_intersection(L1, L2):
    """util:5-40.  Ray/segment intersection; returns (distance from origin, hit point)."""
    p0, p1 = L1
    p2, p3 = L2
    ax, ay = p1[0] - p0[0], p1[1] - p0[1]
    bx, by = p3[0] - p2[0], p3[1] - p2[1]
    denom = ax * by - bx * ay
    if denom == 0:
        return float("inf"), (0, 0)
    pos = denom > 0
    cx, cy = p0[0] - p2[0], p0[1] - p2[1]
    s_num = ax * cy - ay * cx
    if (s_num < 0) == pos:
        return float("inf"), (0, 0)
    t_num = bx * cy - by * cx
    if (t_num < 0) == pos:
        return float("inf"), (0, 0)
    if (s_num > denom) == pos or (t_num > denom) == pos:
        return float("inf"), (0, 0)
    t = t_num / denom
    hx, hy = p0[0] + t * ax, p0[1] + t * ay
    return sqrt(hx * hx + hy * hy), (hx, hy)


def comp_laser(laser_lines, lines_with_vel, orientation):
    """util:42-113.  Rotate every segment (and its velocity) into the frame whose x axis is
    ``orientation``, then take the nearest hit of each ray."""
    theta = -np.arctan2(orientation[1], orientation[0])
    # the same numpy 2x2 @ 2 products as util:48-64, so that results agree to the last bit
    rot = np.array([[np.cos(theta), -np.sin(theta)], [np.sin(theta), np.cos(theta)]])

    rotated = []
    for (a, b), vel in lines_with_vel:
        a_r = rot @ np.array(a)
        b_r = rot @ np.array(b)
        tip = rot @ (np.array(a) + np.array(vel))
        rotated.append(((a_r, b_r), tip - a_r))
    out = []
    for ray in laser_lines:
        best_d, best_hit, best_vel = float("inf"), (0, 0), (0, 0)
        for seg, vel in rotated:
            d, hit = line_intersection(ray, seg)
            if d < best_d:
                best_d, best_hit, best_vel = d, hit, vel
        if best_hit == (0, 0):
            best_vel = (0, 0)
        out.append((best_hit, best_vel))
    return out


def laser_rays(num=16, length=1.5):
    """env:321-332."""
    return [((0, 0), (length * cos(i * 2 * pi / num), -length * sin(i * 2 * pi / num))) for i in range(num)]


def circle_approx(num=8, radius=0.5):
    """env:335-350: octagon whose vertices are (r cos t, -r sin t)."""
    pts = [(radius * cos(i * 2 * pi / num), -radius * sin(i * 2 * pi / num)) for i in range(num)]
    return [(pts[i], pts[(i + 1) % num]) for i in range(num)]


# ------------------------------------------------------------------------------------ shells
def _goal_dir(pos, target):
    """env:156-162 / ALAN:489-495: (cos, sin) of atan2(target - pos)."""
    ang = np.arctan2(target[1] - pos[1], target[0] - pos[0])
    return (cos(ang), sin(ang))


def _make_sim(scn, env_index, sim_cls=None):
    """Build the world like the shells do (env:62-68,126-148 ; ALAN:22-28,461-479).  ``sim_cls``
    lets a test put another PyRVOSimulator-compatible class behind the same shell logic."""
    P = scn.params
    sim = (sim_cls or PyRVOSimulator)(P["timeStep"], P["neighborDist"], P["maxNeighbors"], P["timeHorizon"], P["timeHorizonObst"],
                         P["radius"], P["maxSpeed"])
    for i in range(scn.agents_per_env):
        a = sim.addAgent(tuple(map(float, scn.pos[env_index, i])), P["neighborDist"], P["maxNeighbors"],
                         P["timeHorizon"], P["timeHorizonObst"], P["radius"], P["maxSpeed"],
                         tuple(map(float, scn.vel[env_index, i])))
        sim.setAgentPrefVelocity(a, tuple(map(float, scn.vel[env_index, i])))  # env:137, ALAN:471
    polys = scn.obstacles[env_index] if scn.per_env_obstacles else scn.obstacles
    for poly in polys:
        sim.addObstacle([tuple(map(float, v)) for v in poly])
    sim.processObstacles()
    return sim


class AlanShellOracle:
    """ALAN:10-172,483-495,547-636 for ONE world built from env ``env_index`` of a Scenario."""

    def __init__(self, scn, env_index=0, online_actions=None, gamma=0.6, timewindow=2, online_temp=0.2,
                 sim_cls=None):
        self.P = scn.params
        self.N = scn.agents_per_env
        self.timeStep = self.P["timeStep"]
        self.radius = self.P["radius"]
        self.maxSpeed = self.P["maxSpeed"]
        self.online_actions = list(online_actions) if online_actions is not None else [
            (1, 0), (0.70711, 0.70711), (0, 1), (-0.70711, 0.70711), (-1, 0), (-0.70711, -0.70711), (0, -1),
            (0.70711, -0.70711)]  # ALAN:31-38
        self.gamma, self.timewindow, self.online_temp = gamma, timewindow, online_temp  # ALAN:47-49
        self.sim = _make_sim(scn, env_index, sim_cls)
        self.targets = [(tuple(map(float, scn.goal[env_index, i])), tuple(map(float, scn.goal2[env_index, i])))
                        for i in range(self.N)]
        A = len(self.online_actions)
        self.action_weights = [[0.0] * A for _ in range(self.N)]
        self.action_times = [[0.0] * A for _ in range(self.N)]
        self.step_count = 0
        self.max_step = int((10 / self.timeStep) * self.N)  # ALAN:59
        self.agents_done = [0] * self.N
        self.agents_time = [self.max_step * self.timeStep] * self.N  # ALAN:62
        self.update_pref_vel()
        # min TTime, ALAN:161-172
        times = []
        for i in range(self.N):
            start, goal = self.sim.getAgentPosition(i), self.targets[i][0]
            times.append(self.maxSpeed * sqrt((goal[0] - start[0]) ** 2 + (goal[1] - start[1]) ** 2))
        times = np.array(times)
        self.min_TTime = np.average(times) + 3 * np.std(times, 0)
        self.last = {}

    def comp_pref_vel(self, i):
        return _goal_dir(self.sim.getAgentPosition(i), self.targets[i][0])

    def update_pref_vel(self):  # ALAN:483-486
        for i in range(self.N):
            self.sim.setAgentPrefVelocity(i, self.comp_pref_vel(i))

    def done_test(self):  # ALAN:547-566
        for i in range(self.N):
            if self.agents_done[i] == 0:
                pos, t_pos = self.sim.getAgentPosition(i), self.targets[i][0]
                if sqrt((pos[0] - t_pos[0]) ** 2 + (pos[1] - t_pos[1]) ** 2) < 2 * self.radius:
                    self.agents_done[i] = 1
                    self.agents_time[i] = self.step_count * self.timeStep
                    self.targets[i] = (self.targets[i][1], self.targets[i][1])
        return 0 not in self.agents_done

    def online_step(self, uniforms):
        """ALAN:569-628.  ``uniforms[i]`` replaces the global-RNG draw inside
        np.random.choice(A, 1, p=ps): numpy's choice takes cdf = cumsum(p) / cdf[-1] and
        returns searchsorted(cdf, u, side='right')."""
        action_vels, pref_vels, action_ids = [], [], []
        for i in range(self.N):
            weights = np.array(self.action_weights[i])
            ps = np.exp(weights / self.online_temp)
            ps /= np.sum(ps)
            cdf = np.cumsum(ps)
            cdf /= cdf[-1]
            action_id = int(min(np.searchsorted(cdf, uniforms[i], side="right"), len(ps) - 1))
            action = self.online_actions[action_id]
            action_ids.append(action_id)
            pref_vel = np.array(self.comp_pref_vel(i))
            pref_vels.append(pref_vel)
            goal_theta = np.arctan2(pref_vel[1], pref_vel[0]) + np.arctan2(action[1], action[0])
            action_vel = (cos(goal_theta), sin(goal_theta))
            action_vels.append(action_vel)
            self.sim.setAgentPrefVelocity(i, (float(action_vel[0]), float(action_vel[1])))
        self.sim.doStep()
        rewards = []
        for i in range(self.N):
            orca_vel = self.sim.getAgentVelocity(i)
            R_goal = np.dot(orca_vel, pref_vels[i])
            R_polite = np.dot(orca_vel, action_vels[i])
            R = self.gamma * R_goal + (1 - self.gamma) * R_polite
            rewards.append(R)
            for act in range(len(self.online_actions)):
                self.action_times[i][act] += self.timeStep
                if self.action_times[i][act] >= self.timewindow:
                    self.action_times[i][act] = 0
                    self.action_weights[i][act] = 0
            self.action_weights[i][action_ids[i]] = R
        self.last = dict(action_ids=action_ids, rewards=rewards, pref_vels=pref_vels, action_vels=action_vels)

    def orca_step(self):  # ALAN:631-636
        self.sim.doStep()
        self.update_pref_vel()

    def run_sim(self, mode=1, uniforms=None, max_steps=None):
        """ALAN:106-131.  ``uniforms``: [steps, N] draws for mode 1."""
        success = False
        for t in range(self.max_step if max_steps is None else max_steps):
            if mode == 1:
                self.online_step(uniforms[t])
            else:
                self.orca_step()
            self.step_count += 1
            success = self.done_test()
            if success:
                break
        times = np.array(self.agents_time)
        TTime = np.average(times) + 3 * np.std(times, 0)
        return success, self.step_count * self.timeStep, TTime, self.min_TTime


class EnvShellOracle:
    """env:23-123,151-162,231-416,461-488 for ONE world (Tk, gym spaces and time.clock left out)."""

    def __init__(self, scn, env_index=0, max_step=1000, sim_cls=None):
        self.P = scn.params
        self.N = scn.agents_per_env
        self.neighborDist = self.P["neighborDist"]
        self.radius = self.P["radius"]
        self.laser_num, self.circle_approx_num = 16, 8  # env:34-35
        self.ray_lines = laser_rays(self.laser_num, self.neighborDist)
        self.approx_lines = circle_approx(self.circle_approx_num, self.radius)
        self.sim = _make_sim(scn, env_index, sim_cls)
        self.targets = [tuple(map(float, scn.goal[env_index, i])) for i in range(self.N)]
        self.targets2 = [tuple(map(float, scn.goal2[env_index, i])) for i in range(self.N)]
        self.step_count, self.max_step = 0, max_step
        self.agents_done = [0] * self.N
        self.update_pref_vel()

    def comp_pref_vel(self, i):
        return _goal_dir(self.sim.getAgentPosition(i), self.targets[i])

    def update_pref_vel(self):
        for i in range(self.N):
            self.sim.setAgentPrefVelocity(i, self.comp_pref_vel(i))

    def done_test(self):  # env:352-365
        for i in range(self.N):
            if self.agents_done[i] == 0:
                if self.sim.getAgentPosition(i)[0] < 2.0:
                    self.agents_done[i] = 1
                    self.targets[i] = self.targets2[i]
        return 0 not in self.agents_done

    def get_obs(self):  # env:231-318
        obs = []
        for i in range(self.N):
            pref_vel = self.comp_pref_vel(i)
            lines = []
            my = self.sim.getAgentPosition(i)
            for j in range(self.sim.getAgentNumAgentNeighbors(i)):
                nid = self.sim.getAgentAgentNeighbor(i, j)
                npos = self.sim.getAgentPosition(nid)
                rel = (npos[0] - my[0], npos[1] - my[1])
                nvel = self.sim.getAgentVelocity(nid)
                for a, b in self.approx_lines:
                    lines.append((((a[0] + rel[0], a[1] + rel[1]), (b[0] + rel[0], b[1] + rel[1])), nvel))
            for j in range(self.sim.getAgentNumObstacleNeighbors(i)):
                v1 = self.sim.getAgentObstacleNeighbor(i, j)
                v2 = self.sim.getNextObstacleVertexNo(v1)
                p1, p2 = self.sim.getObstacleVertex(v1), self.sim.getObstacleVertex(v2)
                lines.append((((p1[0] - my[0], p1[1] - my[1]), (p2[0] - my[0], p2[1] - my[1])), (0, 0)))
            if lines:
                res = comp_laser(self.ray_lines, lines, pref_vel)
            else:
                res = [((0, 0), (0, 0))] * self.laser_num
            o = []
            for hit, vel in res:
                o += [hit[0], hit[1], vel[0], vel[1]]
            obs.append(o)
        return obs

    def step(self, thetas, scale=0.3):  # env:367-416
        rl_vels, pref_vels = [], []
        for i in range(self.N):
            pref_vel = np.array(self.comp_pref_vel(i))
            pref_vels.append(pref_vel)
            goal_theta = np.arctan2(pref_vel[1], pref_vel[0]) + float(thetas[i])
            rl_vel = (cos(goal_theta), sin(goal_theta))
            rl_vels.append(rl_vel)
            self.sim.setAgentPrefVelocity(i, (float(rl_vel[0]), float(rl_vel[1])))
        self.sim.doStep()
        rewards = []
        for i in range(self.N):
            orca_vel = self.sim.getAgentVelocity(i)
            R_goal = np.dot(orca_vel, pref_vels[i])
            R_polite = np.dot(orca_vel, rl_vels[i])
            rewards.append(scale * R_goal + (1 - scale) * R_polite)
        done_all = self.done_test()
        self.step_count += 1
        if self.step_count >= self.max_step:
            done_all = True
        return self.get_obs(), rewards, done_all

    def orca_step(self):  # env:447-450
        self.sim.doStep()
        self.update_pref_vel()
        return self.get_obs()

    def reset(self, positions):  # env:461-488 (positions replace the unseeded uniform draws)
        for i in range(self.N):
            self.sim.setAgentPosition(i, tuple(map(float, positions[i])))
        self.update_pref_vel()
        self.step_count = 0
        self.agents_done = [0] * self.N
        return self.get_obs()
