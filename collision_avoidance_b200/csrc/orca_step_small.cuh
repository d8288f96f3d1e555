// orca_step_small.cuh -- fused ORCA environment step for worlds that fit one thread block
// (agents_per_env <= 256): the shape of BASELINE configs 1-4.
//
// One thread per agent, one or more whole envs per block.  The block stages the pre-step
// positions/velocities of its envs in shared memory (one coalesced float2 load each), so the
// brute-force neighbor scan and every neighbor fetch after it are shared-memory reads and HBM
// sees exactly the algorithmic traffic: pos + vel + goal in, pos + vel out (40 B / agent-step,
// SURVEY.md 8d).  Because a whole env lives in one block and all reads of other agents go
// through the staged copy, the update is done in place (RVO2's two-phase doStep, SURVEY 3.4).
//
// Replaces, per step and for every env of the batch at once:
//   RVO2 doStep (kd-tree build + computeNeighbors + computeNewVelocity + update)
//       <- collision_avoidence_env.py:385,448 ; ALAN_true.py:601,632
//   comp_pref_vel / update_pref_vel            <- env :151-162 ; ALAN :483-495
//   action rotation, reward                    <- env :371-400 ; ALAN :588-618
//   done test / goal switch                    <- env :352-365 ; ALAN :547-566
//   ALAN softmax bandit select + update        <- ALAN :576-586, 620-628
#pragma once

#include "orca_core.cuh"

namespace orca {

constexpr int kMaxDevices = 64;  // size of the per-device "attribute already set" tables of the launchers

enum : int { POLICY_EXTERNAL = 0, POLICY_GOAL = 1, POLICY_RL = 2, POLICY_ALAN = 3 };
enum : int { DONE_NONE = 0, DONE_GOAL_RADIUS = 1, DONE_X_BELOW = 2, DONE_GOAL_RADIUS_DEFERRED = 3 };
enum : int {
  STAT_AGENT_STEPS = 0,
  STAT_FINISHED = 1,
  STAT_COLLISIONS = 2,
  STAT_LP3_CALLS = 3,
  STAT_OVERFLOW = 4,
  STAT_SUM_ARRIVAL = 5,
  STAT_SUM_ARRIVAL2 = 6,
  STAT_SUM_REWARD = 7
};

struct StepArgs {
  // shape: the launch covers envs [env_base, E)
  int E, N, envs_per_block, env_base;
  // simulator parameters (uniform over the batch)
  int k;
  float dt, inv_dt, nd_sq, inv_th, inv_tho, radius, vmax, obst_range_sq;
  // state
  float2* pos;
  float2* vel;
  const float2* pref;
  float2* goal;
  const float2* goal2;
  // RL policy
  const float* action_theta;
  float rl_scale, done_x;
  // ALAN
  float* alan_w;
  const float2* alan_actions;
  uint8_t* alan_action_out;
  const float* alan_uniform_in;
  int A, alan_window;
  float alan_gamma, alan_inv_temp;
  unsigned long long seed;
  const int* alan_A_env;  // per-env action count (NULL: A everywhere)
  int alan_env_stride;    // per-env action table stride in float2 (0: shared table)
  // outputs
  float* reward;
  uint8_t* done;
  float* arrival;
  int* env_step;
  int* env_done_cnt;
  int done_mode;
  int* nbr_idx;
  float* nbr_dsq;
  int* nbr_cnt;
  int* onbr_idx;
  int* onbr_cnt;
  unsigned long long* stats;
  // obstacles
  const float4* vert_pd;
  const int4* vert_link;
  const int4* bsp;
  const float4* bsp_seg;
  const int* env_nodes;  // per-env node count, or NULL when the world is shared
  int shared_nodes;      // node count of the shared world
  int vert_stride;       // per-env table stride (0 when shared)
  int world_slots;       // vertex slots of the obstacle tables a block stages in shared memory (0: read global)
  int world_verts;       // number of rows in one obstacle table (shared world: its vertex count)
  // 1: stop after the neighbor search (orca_neighbors parity hook)
  int neighbors_only;
  // 1: uniform-grid path; an env spans several blocks, so its step counter is bumped by a
  // separate kernel instead of by the env's first agent
  int grid_path;
  // optional second destination of the post-step state: the caller's host buffers mapped into
  // the device address space (orca_step_host), written by the kernel itself over PCIe
  float2* pos_mirror;
  float2* vel_mirror;
  // 1 / cell side of the in-block neighbor grid (tile kernel, worlds of more than 32 agents); 0: off
  float tile_grid_inv_cell;
  // [E*N] starting threshold (squared) of each agent's neighbor search, written by the previous step
  // (library scratch; nullptr: always start from the neighbor range), and the margin added to the k-th
  // distance: what two agents can approach each other within one step, 2 * maxSpeed * timeStep + 25 %
  float* nbr_hint;
  float hint_slack;
  // obstacle-free maps: 32 row words + one float4 of geometry per world (stride 0 when the world is shared)
  const uint32_t* cull_rows;
  const float4* cull_geo;
};

// Per-agent ORCA parameters (orca_set_agent_params), read by the HETERO kernels only, from a table that
// travels next to StepArgs (whose scalars stay the handle's values): two float4 per agent,
// {radius, maxSpeed, 1 / timeHorizon, 1 / timeHorizonObst} and {neighborDist^2, obstacle range^2,
// maxNeighbors (int bits), 0}.  AgentParams = one agent's record.
struct AgentParams {
  int k;
  float nd_sq, obst_range_sq, radius, vmax, inv_th, inv_tho;
};
ORCA_HD AgentParams load_agent_params(const float4* table, const int g) {
  const float4 r0 = ORCA_LDG(&table[2 * (size_t)g]);
  const float4 r1 = ORCA_LDG(&table[2 * (size_t)g + 1]);
  AgentParams q;
  q.radius = r0.x;
  q.vmax = r0.y;
  q.inv_th = r0.z;
  q.inv_tho = r0.w;
  q.nd_sq = r1.x;
  q.obst_range_sq = r1.y;
  q.k = float_to_bits(r1.z);
  return q;
}

// Where an agent's neighbor candidates come from.  TileSource: the pre-step snapshot of the
// agent's own env in shared memory, candidates = every other agent of the env in id order.
//
// For worlds of more than 32 agents the block first bins its envs' agents into a small uniform
// grid in shared memory (kTileGrid x kTileGrid cells of side neighborDist per env, anchored at
// the env's bounding-box corner; see build_tile_grid): candidates = the agents of the 3 x 3 cells
// around the agent -- about a fifth of a 256-agent dense crowd instead of all of it.  They no
// longer arrive in id order, so equal distances are ranked by id explicitly (offer_ranked), which
// gives the same list as the ascending-id scan.
constexpr int kTileGrid = 8;                          // cells per side
constexpr int kTileCells = kTileGrid * kTileGrid;     // 64
constexpr int kTileStartStride = kTileCells + 2;      // cell_start row per env (u16), padded

// SMALL = the kernel only ever sees worlds of at most 32 agents (the slim kernel): the candidate-buffer
// and in-block-grid searches, and the threshold hint with them, are not compiled at all.
template <bool SMALL>
struct TileSourceT {
  static constexpr bool kObstacleCull = false;
  const float2* env_pos;
  const float2* env_vel;
  int n;
  int self;
  // in-block grid of this agent's env (nullptr: scan every agent of the env)
  const unsigned short* cell_start = nullptr;  // [kTileCells + 1] exclusive prefix of the cell populations
  const unsigned char* sorted = nullptr;       // [n] agent ids ordered by cell
  int cx = 0, cy = 0;                          // the agent's own cell
  float ox = 0.f, oy = 0.f;                    // grid origin (the env's bounding-box corner)

  struct LowerIdFirst {
    ORCA_HD bool operator()(int a, int b) const { return b >= 0 && a < b; }
  };
  template <int K, bool KFULL>
  using List = NearestKeys<K, KFULL>;
  // Worlds of at most 32 agents: rank every candidate by counting instead of inserting into a
  // sorted list.  rank(j) = number of candidates that go in front of j in (distSq, id) order;
  // the accepted neighbors are the in-range candidates of rank < k, already in RVO2's order
  // (stable insertion in ascending-id visiting order gives exactly this permutation, and the
  // "range shrinks to the k-th best" rule rejects exactly the candidates of rank >= k).
  // M (M - 1) / 2 independent compare/accumulate pairs with every lane live, against ~80
  // instructions per candidate under a divergent branch for the insertion (DESIGN.md section 5).
  // The sorted ids are scattered as bytes into the agent's first line slot (not in use yet) and
  // read back with one 16-byte load.
  template <int M, class NK>
  ORCA_HD void gather_ranked(NK& nk, float2 p, const Lines& scratch) const {
    float d[M];
#pragma unroll
    for (int j = 0; j < M; ++j) {
      const float2 q = env_pos[j < n ? j : 0];
      // candidates that do not exist (j >= n) and the agent itself sit at distance +inf; adding
      // the pad (instead of selecting) keeps the shared-memory load unconditional
      const float pad = (j < n && j != self) ? 0.f : INFINITY;
      d[j] = abs_sq(sub(p, q)) + pad;
    }
    int r[M];
    rank_count<M>(d, r);
    unsigned char* slot = reinterpret_cast<unsigned char*>(scratch.base);
    int cnt = 0;
#pragma unroll
    for (int j = 0; j < M; ++j) {
      const bool in = d[j] < nk.range_sq && r[j] < nk.k;  // k <= 16: the rank fits the 16-byte slot
      cnt += in ? 1 : 0;
      ORCA_DCHECK(!in || (r[j] >= 0 && r[j] < 16));
      if (in) slot[r[j]] = (unsigned char)j;
    }
    nk.set_sorted_ids(*reinterpret_cast<const uint4*>(scratch.base), cnt);
  }
  // Worlds of 17..32 agents: the same ranks without 32 keys + 32 counters live in registers at once
  // (gather_ranked<32> peaks above 64 registers, which the 4-blocks-per-SM kernel does not have).
  // Keys 0..15 (A) stay in registers, keys 16..31 (B) go to the agent's (still unused) line column.
  //   rank(a) = rank within A + #{b : d_b <  d_a}      (a tie keeps the lower index, an A key, in front)
  //   rank(b) = rank within B + #{a : !(d_b < d_a)}
  // 120 + 256 + 120 pair tests -- as many as rank_count<32> -- with the 256 cross tests in a rolled loop.
  // (One rolled body for both halves, cross counts by unsigned compares of the distance bits, halves
  // the code again but tests every cross pair twice: measured 248 vs 225 us in config 3, not kept.)
  // Column layout: slot 0 = the sorted id bytes (output), slots 1-4 = d_B, slots 5-8 = #A keys in front of b.
  template <class NK>
  ORCA_HD void gather_ranked32(NK& nk, float2 p, const Lines& scratch) const {
    float dA[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float2 q = env_pos[j < n ? j : 0];
      const float pad = (j < n && j != self) ? 0.f : INFINITY;
      dA[j] = abs_sq(sub(p, q)) + pad;
    }
#pragma unroll
    for (int g4 = 0; g4 < 4; ++g4) {
      float t[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = 16 + 4 * g4 + u;
        const float2 q = env_pos[j < n ? j : 0];
        const float pad = (j < n && j != self) ? 0.f : INFINITY;
        t[u] = abs_sq(sub(p, q)) + pad;
      }
      float4 w;
      w.x = t[0];
      w.y = t[1];
      w.z = t[2];
      w.w = t[3];
      scratch.base[(1 + g4) * scratch.stride] = w;
    }
    int rA[16];
    rank_count<16>(dA, rA);
    // counts as sums of the BIT PATTERN of 1.0f (see rank_count): one FSET per pair, integer adds
    unsigned crossA[16];
#pragma unroll
    for (int a = 0; a < 16; ++a) crossA[a] = 0u;
#pragma unroll 1
    for (int g4 = 0; g4 < 4; ++g4) {
      const float4 w = scratch.base[(1 + g4) * scratch.stride];
      const float b[4] = {w.x, w.y, w.z, w.w};
      unsigned sum[4] = {0u, 0u, 0u, 0u};
#pragma unroll
      for (int a = 0; a < 16; ++a) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const unsigned f = lt_as_one_bits(b[u], dA[a]);
          crossA[a] += f;
          sum[u] += f;
        }
      }
      float4 o;  // #A keys in front of b = 16 - #{a : d_b < d_a}
      o.x = bits_to_float(16 - one_bits_count(sum[0]));
      o.y = bits_to_float(16 - one_bits_count(sum[1]));
      o.z = bits_to_float(16 - one_bits_count(sum[2]));
      o.w = bits_to_float(16 - one_bits_count(sum[3]));
      scratch.base[(5 + g4) * scratch.stride] = o;
    }
    float dB[16];
    int crossB[16];
#pragma unroll
    for (int g4 = 0; g4 < 4; ++g4) {
      const float4 w = scratch.base[(1 + g4) * scratch.stride];
      const float4 o = scratch.base[(5 + g4) * scratch.stride];
      dB[4 * g4] = w.x;
      dB[4 * g4 + 1] = w.y;
      dB[4 * g4 + 2] = w.z;
      dB[4 * g4 + 3] = w.w;
      crossB[4 * g4] = float_to_bits(o.x);
      crossB[4 * g4 + 1] = float_to_bits(o.y);
      crossB[4 * g4 + 2] = float_to_bits(o.z);
      crossB[4 * g4 + 3] = float_to_bits(o.w);
    }
    unsigned char* slot = reinterpret_cast<unsigned char*>(scratch.base);
    int cnt = 0;
#pragma unroll
    for (int a = 0; a < 16; ++a) {
      const int r = rA[a] + one_bits_count(crossA[a]);
      const bool in = dA[a] < nk.range_sq && r < nk.k;
      cnt += in ? 1 : 0;
      ORCA_DCHECK(!in || (r >= 0 && r < 16));
      if (in) slot[r] = (unsigned char)a;
    }
    int rB[16];
    rank_count<16>(dB, rB);
#pragma unroll
    for (int b = 0; b < 16; ++b) {
      const int r = rB[b] + crossB[b];
      const bool in = dB[b] < nk.range_sq && r < nk.k;
      cnt += in ? 1 : 0;
      ORCA_DCHECK(!in || (r >= 0 && r < 16));
      if (in) slot[r] = (unsigned char)(16 + b);
    }
    nk.set_sorted_ids(*reinterpret_cast<const uint4*>(scratch.base), cnt);
  }
  // true when gather() searches through the candidate buffer with a shrinking threshold and knows how
  // to search again: it can start from a tighter threshold than the neighbor range (see agent_front)
  ORCA_HD bool threshold_search() const { return !SMALL && cell_start != nullptr; }
  float full_range_sq = 0.f;  // the neighbor range (squared), for the second pass
  // The list arrives initialised with its STARTING threshold (agent_front): nk.range_sq, the neighbor
  // range or last step's tighter bound.  The threshold paths search again from the full range
  // (`range_sq`) for the lanes whose list did not fill up from a tighter start.
  template <class NK>
  ORCA_HD void gather(NK& nk, float2 p, const Lines& scratch, int scratch_slots, unsigned mask) const {
#ifndef ORCA_NO_RANKED16  // A/B switch: -DORCA_NO_RANKED16 builds the insertion path for small worlds too
    if (n <= 16) {
      gather_ranked<16>(nk, p, scratch);
      return;
    }
    if (SMALL || n <= 32) {
#ifdef ORCA_RANKED32_FLAT  // A/B switch: all 32 keys in registers
      gather_ranked<32>(nk, p, scratch);
#else
      gather_ranked32(nk, p, scratch);
#endif
      return;
    }
#endif
    if (n <= 32) {
      // few candidates, most of them accepted by most lanes: insert directly
      for (int j = 0; j < n; ++j) {
        if (j == self) continue;
        const float2 q = env_pos[j];
        nk.offer(abs_sq(sub(p, q)), j);
      }
      nk.finish();
      return;
    }
    CandidateBuffer buf;
    buf.base = scratch.base;
    buf.stride = scratch.stride;
    buf.cap = 2 * scratch_slots;  // two (distSq, id) entries per 16-byte line slot
    buf.cnt = 0;
    if (cell_start != nullptr) {
      LowerIdFirst before;
      auto insert_ranked = [&nk, &before](float d, int id) { nk.offer_ranked(d, id, before); };
      const int x0 = cx > 0 ? cx - 1 : 0, x1 = cx + 1 < kTileGrid ? cx + 1 : kTileGrid - 1;
      bool enabled = true;
      // three rows of cells; the cells (x0..x1, row) have consecutive keys, i.e. they are one
      // contiguous run of `sorted`.  Lanes walk their own runs but vote together every iteration.
      // The agent's own row goes first: the nearest candidates tighten the threshold early.
      // Rows 3-5 = the second pass: lanes that started from a tighter threshold than the range and
      // did not fill their list search again from the range (rare; the others keep them company).
#pragma unroll 1
      for (int r = 0; r < 6; ++r) {
        if (r == 3) {
          buf.drain(mask, insert_ranked);
          nk.finish();
          enabled = nk.range_sq < full_range_sq && !nk.full();
          if (!ORCA_ANY(mask, enabled)) break;
          if (enabled) nk.init(nk.k, full_range_sq);
        }
        const int rr = r < 3 ? r : r - 3;
        const int yy = cy + (rr == 0 ? 0 : (rr == 1 ? -1 : 1));
        int q = 0, last = 0;
        if (enabled && yy >= 0 && yy < kTileGrid) {
          q = cell_start[yy * kTileGrid + x0];
          last = cell_start[yy * kTileGrid + x1 + 1];
        }
        while (ORCA_ANY(mask, q < last)) {  // two candidates per pair of warp votes
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            if (q < last) {
              const int j = sorted[q];
              ORCA_DCHECK(q >= 0 && q < n && j >= 0 && j < n);
              if (j != self) {
                const float d = abs_sq(sub(p, env_pos[j]));
                if (d <= nk.thresh()) buf.push(d, j);
              }
              ++q;
            }
          }
          buf.drain_if_full(mask, insert_ranked, 2);
        }
      }
      buf.drain(mask, insert_ranked);
      nk.finish();
      nk.pack_ids();
      return;
    }
    auto insert = [&nk](float d, int id) { nk.offer(d, id); };
    for (int j = 0; j < n; ++j) {  // n is uniform over the warp's envs
      if (j != self) {
        const float2 q = env_pos[j];
        const float d = abs_sq(sub(p, q));
        if (d < nk.thresh()) buf.push(d, j);
      }
      buf.drain_if_full(mask, insert);
    }
    buf.drain(mask, insert);
    nk.finish();
    nk.pack_ids();
  }
  ORCA_HD float2 pos(int q) const { return env_pos[q]; }
  ORCA_HD float2 vel(int q) const { return env_vel[q]; }
  ORCA_HD int local_id(int q) const { return q; }
  // per-agent radii of the env, staged next to the snapshot (HETERO kernels only)
  const float* env_rad = nullptr;
  ORCA_HD float radius(int q) const { return env_rad[q]; }
};
using TileSource = TileSourceT<false>;

// atomics: device atomics in the kernels, plain adds in the single-threaded host emulation
ORCA_HD void stat_add_u64(unsigned long long* stats, int slot, unsigned long long v) {
  if (stats != nullptr && v != 0ull) {
#if defined(__CUDA_ARCH__)
    atomicAdd(&stats[slot], v);
#else
    stats[slot] += v;
#endif
  }
}
ORCA_HD void stat_add_f64(unsigned long long* stats, int slot, double v) {
  if (stats != nullptr) {
#if defined(__CUDA_ARCH__)
    atomicAdd(reinterpret_cast<double*>(&stats[slot]), v);
#else
    *reinterpret_cast<double*>(&stats[slot]) += v;
#endif
  }
}
// One atomic per warp instead of one per thread: every live lane of the warp calls this together
// (a converged point of the step), the lanes' values are summed with one REDUX instruction and the
// first live lane issues the atomic -- and none at all when the warp's sum is zero.  With per-thread
// atomics the LP3 / collision counters were up to 400,000 same-address atomics per launch.
ORCA_HD void stat_add_u64_warp(unsigned long long* stats, int slot, unsigned v) {
#if defined(__CUDA_ARCH__)
  if (stats == nullptr) return;  // uniform over the launch
  const unsigned m = __activemask();
  const unsigned total = __reduce_add_sync(m, v);
  if (total != 0u && (int)(threadIdx.x & 31u) == __ffs((int)m) - 1) atomicAdd(&stats[slot], (unsigned long long)total);
#else
  stat_add_u64(stats, slot, (unsigned long long)v);
#endif
}
ORCA_HD void stat_add_f64_warp(unsigned long long* stats, int slot, float v) {
#if defined(__CUDA_ARCH__)
  if (stats == nullptr) return;
  const unsigned m = __activemask();
  double total = (double)v;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double other = __shfl_xor_sync(m, total, o);
    // lanes outside m return their own value for the partner; only add partners that are live
    if ((m >> ((threadIdx.x & 31u) ^ o)) & 1u) total += other;
  }
  if ((int)(threadIdx.x & 31u) == __ffs((int)m) - 1) atomicAdd(reinterpret_cast<double*>(&stats[slot]), total);
#else
  stat_add_f64(stats, slot, (double)v);
#endif
}
ORCA_HD void counter_inc(int* c) {
#if defined(__CUDA_ARCH__)
  atomicAdd(c, 1);
#else
  *c += 1;
#endif
}

// What an agent carries from the front half of the step (policy, neighbors, half-planes, LP2)
// across the LP3 stage to the back half (integration, reward, bandit update, done test).
struct AgentCarry {
  float2 p, v;     // pre-step state
  float2 aim;      // the agent's input of the step, loaded by the caller as early as possible (it may
                   // live in mapped host memory, a PCIe round trip away): goal, or pref when EXTERNAL
  float2 gdir;     // unit vector to the goal (pre-step position)
  float2 pref;     // preferred velocity handed to ORCA
  float2 nv;       // new velocity
  int act;         // ALAN: chosen action
  int n, n_obst;   // ORCA lines, obstacle lines among them
  int fail;        // LP2 failure index (== n when feasible)
  unsigned collisions;
  bool overflow;
};

// The obstacle tables of env `env` as they sit in global memory.
ORCA_HD ObstacleWorld global_world(const StepArgs& a, int env) {
  ObstacleWorld W;
  const size_t voff = (size_t)env * a.vert_stride;
  W.vert_pd = a.vert_pd + voff;
  W.vert_link = a.vert_link + voff;
  W.bsp = a.bsp + voff;
  W.bsp_seg = a.bsp_seg + voff;
  W.n_nodes = (a.env_nodes != nullptr) ? a.env_nodes[env] : a.shared_nodes;
  W.cull_rows = nullptr;
  return W;
}
// ... plus the obstacle-free map of the env's world (obstacle_world.h: build_cull_map), for the sources that use it
ORCA_HD ObstacleWorld global_world_with_cull(const StepArgs& a, int env) {
  ObstacleWorld W = global_world(a, env);
  if (a.cull_rows != nullptr) {
    const size_t w = (a.vert_stride > 0) ? (size_t)env : 0;
    W.cull_rows = a.cull_rows + w * 32;
    W.cull_geo = ORCA_LDG(&a.cull_geo[w]);
  }
  return W;
}

// ALAN action selection (ALAN_true.py:580-586): p = softmax(w / temp); the action is the first one
// whose running sum of UNNORMALISED weights exceeds u * total -- np.random.choice's inverse-CDF draw.
template <int MAXA>
ORCA_HD int alan_select(const float* wrow, const int nA, const float inv_temp, const float u) {
  float w_act[MAXA];
  float total = 0.f;
#pragma unroll
  for (int i = 0; i < MAXA; ++i) {
    if (i < nA) {
      w_act[i] = expf(wrow[i] * inv_temp);
      total += w_act[i];
    }
  }
  const float target = u * total;
  float run = 0.f;
  int act = nA - 1;
  bool found = false;
#pragma unroll
  for (int i = 0; i < MAXA; ++i) {
    if (i < nA) {
      run += w_act[i];
      if (!found && run > target) {
        act = i;
        found = true;
      }
    }
  }
  return act;
}

// Front half.  `src` yields the PRE-step state of the other agents (shared-memory tile or
// uniform-grid cells), `L` is the agent's private line storage, `estep` the env's step counter
// before this step.  Returns false when the step ends here (neighbors-only parity hook).
// OL = obstacle-line slots of the agent's line storage (agents that need more take agent_slow_path).
// HETERO = the agent's ORCA parameters come from its record in `agent_params` (neighbor radii from
// src.radius); a compile-time variant, so the uniform kernels are the code they were.  Per-agent k
// needs the K-slot lists of KFULL = false, whose searches start from the agent's own range (no hint).
template <int K, bool KFULL, int POLICY, int OL = ORCA_MAX_OBST_LINES, bool HETERO = false, class Src>
ORCA_HD bool agent_front(const StepArgs& a, const int env, const int g, const int estep, const Src& src,
                         const ObstacleWorld& W, const Lines L, const unsigned warp_mask, AgentCarry& c,
                         const float4* agent_params = nullptr) {
  static_assert(!(HETERO && KFULL), "per-agent maxNeighbors needs the KFULL = false lists");
  const float2 p = c.p, v = c.v;
  const AgentParams ap = HETERO ? load_agent_params(agent_params, g) : AgentParams{};

  // ---------------- preferred velocity (policy) ----------------
  float2 gdir = v2(0.f, 0.f);
  float2 pref;
  int act = 0;
  if (POLICY == POLICY_EXTERNAL) {
    pref = c.aim;
  } else {
    gdir = goal_direction(p, c.aim);
    pref = gdir;
    if (POLICY == POLICY_RL) {
      float sn, cs;
      sincosf(a.action_theta[g], &sn, &cs);
      pref = rotate(gdir, v2(cs, sn));
    }
    if (POLICY == POLICY_ALAN) {
      // softmax over the last rewards; inverse-CDF draw like np.random.choice(p=ps)
      const float* wrow = a.alan_w + (size_t)g * a.A;
      const int nA = (a.alan_A_env != nullptr) ? a.alan_A_env[env] : a.A;  // this env's action count
      const float2* table = a.alan_actions + (size_t)env * a.alan_env_stride;
      const float u = (a.alan_uniform_in != nullptr)
                          ? a.alan_uniform_in[g]
                          : philox_uniform(a.seed, (uint32_t)g, (uint32_t)estep);
      // the loops are unrolled to a compile-time bound (the weights stay in registers); the common
      // sets (the reference's default 8 actions and every .act table but two) take the short one
      act = (a.A <= 8) ? alan_select<8>(wrow, nA, a.alan_inv_temp, u) : alan_select<ORCA_MAX_ACTIONS>(wrow, nA, a.alan_inv_temp, u);
      pref = rotate(gdir, table[act]);
      if (a.alan_action_out != nullptr) a.alan_action_out[g] = (uint8_t)act;
    }
  }
  c.gdir = gdir;
  c.pref = pref;
  c.act = act;

  // ---------------- neighbors ----------------
  bool overflow = false;
  float od[ORCA_MAX_OBST_NEIGHBORS];
  int oid[ORCA_MAX_OBST_NEIGHBORS];
  int ocnt = 0;
  // (the obstacle-free map pays where warps are spatially coherent and the world is mostly empty: the
  // uniform-grid kernel, 367 -> 357 us in config 5; in the tile kernels it measured 0 to +3.5 %, so they
  // do not compile the lookup)
  if (W.n_nodes > 0 && (!Src::kObstacleCull || obstacles_may_be_near(W, p)))
    obstacle_neighbors(W, p, HETERO ? ap.obst_range_sq : a.obst_range_sq, od, oid, &ocnt, &overflow);

  // Temporal coherence: where the search runs on a shrinking threshold (candidate buffer paths), it
  // starts from last step's k-th neighbor distance plus what two agents can approach each other in one
  // step, instead of the neighbor range: candidates that cannot make the list are never parked or
  // inserted (27 -> ~12 insertions per agent in a dense crowd).  EXACT whatever happened in between:
  // if k candidates lie below the starting threshold the k nearest overall are among them; if fewer
  // do (the neighborhood thinned out, the caller moved agents, a first step), the lane searches again
  // from the full range.  The hint is the library's own scratch (StepArgs::nbr_hint), per agent.
  typename Src::template List<K, KFULL> nk;
  const bool hinted = KFULL && a.nbr_hint != nullptr && src.threshold_search();
  if (HETERO)
    nk.init(ap.k, ap.nd_sq);
  else
    nk.init(a.k, hinted ? fminf(a.nbr_hint[g], a.nd_sq) : a.nd_sq);
  src.gather(nk, p, L, K + OL, warp_mask);
  if (hinted) {
    float hint = INFINITY;
    if (nk.full()) {
      const float reach = sqrtf(nk.kth_dist_sq()) + a.hint_slack;
      hint = reach * reach;
    }
    a.nbr_hint[g] = hint;
  }

  if (a.nbr_idx != nullptr) {
    if (nk.packed_cnt >= 0) nk.unpack_ids();
    int cnt = 0;
#pragma unroll
    for (int s = 0; s < K; ++s) {
      if (s < a.k) {
        a.nbr_idx[(size_t)g * a.k + s] = (nk.id[s] >= 0) ? src.local_id(nk.id[s]) : -1;
        // recomputed with the expression of the search (same bits): the ranked path keeps no distances
        if (a.nbr_dsq != nullptr) a.nbr_dsq[(size_t)g * a.k + s] = (nk.id[s] >= 0) ? abs_sq(sub(p, src.pos(nk.id[s]))) : 0.f;
        cnt += (nk.id[s] >= 0) ? 1 : 0;
      }
    }
    a.nbr_cnt[g] = cnt;
  }
  if (a.onbr_idx != nullptr) {
    int* row = a.onbr_idx + (size_t)g * ORCA_MAX_OBST_NEIGHBORS;
    if ((reinterpret_cast<uintptr_t>(a.onbr_idx) & 15u) == 0u) {  // uniform; 16-byte stores: a quarter of the store wavefronts
#pragma unroll
      for (int s = 0; s < ORCA_MAX_OBST_NEIGHBORS; s += 4) {
        int4 w;
        w.x = (s + 0 < ocnt) ? oid[s + 0] : -1;
        w.y = (s + 1 < ocnt) ? oid[s + 1] : -1;
        w.z = (s + 2 < ocnt) ? oid[s + 2] : -1;
        w.w = (s + 3 < ocnt) ? oid[s + 3] : -1;
        *reinterpret_cast<int4*>(row + s) = w;
      }
    } else {
      for (int s = 0; s < ORCA_MAX_OBST_NEIGHBORS; ++s) row[s] = (s < ocnt) ? oid[s] : -1;
    }
    a.onbr_cnt[g] = ocnt;
  }
  if (a.neighbors_only) return false;

  // ---------------- ORCA lines ----------------
  int n_obst = 0;
  if (ocnt > 0)
    n_obst = obstacle_lines<OL>(W, p, v, HETERO ? ap.radius : a.radius, HETERO ? ap.inv_tho : a.inv_tho, od, oid, ocnt, L,
                                &overflow);
  const float inv_th = HETERO ? ap.inv_th : a.inv_th;
  int n = n_obst;
  unsigned collisions = 0;
  {
    const float cr = a.radius + a.radius;
#ifndef ORCA_UNROLLED_LINES  // A/B switch
    if (nk.packed_cnt >= 0) {
      // ranked selection (small worlds): the ids sit in `packed`, a byte each.  One ROLLED loop over
      // them -- K unrolled copies of the half-plane construction are ~13 KB of straight-line code,
      // a quarter of the hot instruction footprint of the kernel (DESIGN.md section 5).
      unsigned w0 = nk.packed.x, w1 = nk.packed.y, w2 = nk.packed.z, w3 = nk.packed.w;
      const int cnt = nk.packed_cnt;
#pragma unroll 1
      for (int s = 0; s < cnt; ++s) {
        const int j = (int)(w0 & 255u);
        w0 = (w0 >> 8) | (w1 << 24);
        w1 = (w1 >> 8) | (w2 << 24);
        w2 = (w2 >> 8) | (w3 << 24);
        w3 >>= 8;
        bool hit;
        ORCA_DCHECK(n < K + OL);
        const float4 ln = agent_line(p, v, src.pos(j), src.vel(j), HETERO ? ap.radius + src.radius(j) : cr, inv_th, a.inv_dt, &hit);
        L.base[n * L.stride] = ln;
        ++n;
        collisions += hit ? 1u : 0u;
      }
    } else {
      // ids that do not fit a byte (sorted slots of the uniform grid): the list goes through a small
      // local-memory array so that the loop can still be rolled; its valid entries are a prefix
      int ids[K + 1];
#pragma unroll
      for (int s = 0; s < K; ++s) ids[s] = nk.id[s];
      ids[K] = -1;
      // the state of the NEXT neighbor is fetched (global memory here) while the current line is built
      int j = ids[0];
      float2 pj = v2(0.f, 0.f), vj = v2(0.f, 0.f);
      if (j >= 0) {
        pj = src.pos(j);
        vj = src.vel(j);
      }
#pragma unroll 1
      for (int s = 1; j >= 0; ++s) {
        const int jn = ids[s];
        float2 pn = pj, vn = vj;
        if (jn >= 0) {
          pn = src.pos(jn);
          vn = src.vel(jn);
        }
        bool hit;
        const float4 ln = agent_line(p, v, pj, vj, HETERO ? ap.radius + src.radius(j) : cr, inv_th, a.inv_dt, &hit);
        L.base[n * L.stride] = ln;
        ++n;
        collisions += hit ? 1u : 0u;
        j = jn;
        pj = pn;
        vj = vn;
      }
    }
#else
    {
      if (nk.packed_cnt >= 0) nk.unpack_ids();
#pragma unroll
      for (int s = 0; s < K; ++s) {
        const int j = nk.id[s];
        if (j >= 0) {
          bool hit;
          const float4 ln = agent_line(p, v, src.pos(j), src.vel(j), HETERO ? ap.radius + src.radius(j) : cr, inv_th, a.inv_dt, &hit);
          L.base[n * L.stride] = ln;
          ++n;
          collisions += hit ? 1u : 0u;
        }
      }
    }
#endif
  }
  c.n = n;
  c.n_obst = n_obst;
  c.collisions = collisions;
  c.overflow = overflow;

  // ---------------- LP2 ----------------
  c.fail = lp2(warp_mask, true, L, n, HETERO ? ap.vmax : a.vmax, pref, false, c.nv);
  return true;
}

// The uncapped path.  RVO2 keeps EVERY obstacle edge in range and every ORCA line built from them
// (insertObstacleNeighbor has no cap, SURVEY A.4); the front half above holds 16 edges and 6
// obstacle lines per agent in registers / shared memory, which covers every agent of every
// scenario of the reference.  An agent that exceeds either capacity is redone here from scratch
// with room for ORCA_SLOW_MAX_OBST edges and lines in LOCAL memory: same neighbor search, same
// half-planes, same LP2 / LP3 (projections recomputed on access), so it gets exactly the result an
// unbounded implementation gives.  Not inlined: the hot code does not grow.  `mask` = the lanes of
// the warp that take this path together.  `scratch` = the agent's own (now dead) line column, used
// by the neighbor search as candidate buffer.  Leaves c.overflow set only if even this capacity
// was exceeded (the statistic the shells turn into an error).
// Everything crosses the call BY VALUE: a reference to the kernel's AgentCarry, neighbor source or
// parameter block would force those into local memory for the whole (hot) kernel.
struct SlowParams {
  int k;
  float nd_sq, inv_th, inv_tho, inv_dt, radius, vmax, obst_range_sq;
};
struct SlowResult {
  float2 nv;
  int n, n_obst, fail;
  unsigned collisions;
  bool overflow;
};
ORCA_HD SlowParams slow_params(const StepArgs& a) {
  SlowParams q;
  q.k = a.k;
  q.nd_sq = a.nd_sq;
  q.inv_th = a.inv_th;
  q.inv_tho = a.inv_tho;
  q.inv_dt = a.inv_dt;
  q.radius = a.radius;
  q.vmax = a.vmax;
  q.obst_range_sq = a.obst_range_sq;
  return q;
}
// ... of agent g from its record (HETERO kernels)
ORCA_HD SlowParams slow_params(const StepArgs& a, const float4* agent_params, const int g) {
  const AgentParams ap = load_agent_params(agent_params, g);
  SlowParams q;
  q.k = ap.k;
  q.nd_sq = ap.nd_sq;
  q.inv_th = ap.inv_th;
  q.inv_tho = ap.inv_tho;
  q.inv_dt = a.inv_dt;
  q.radius = ap.radius;
  q.vmax = ap.vmax;
  q.obst_range_sq = ap.obst_range_sq;
  return q;
}
template <int K, bool KFULL, class Src, bool HETERO = false>
ORCA_HD_NOINLINE SlowResult agent_slow_path(const SlowParams a, const Src src, const ObstacleWorld W, const Lines scratch,
                                            const int scratch_slots, const unsigned mask, const float2 p, const float2 v,
                                            const float2 pref) {
  bool overflow = false;
  float od[ORCA_SLOW_MAX_OBST];
  int oid[ORCA_SLOW_MAX_OBST];
  int ocnt = 0;
  obstacle_neighbors<ORCA_SLOW_MAX_OBST>(W, p, a.obst_range_sq, od, oid, &ocnt, &overflow);
  float4 buf[ORCA_SLOW_MAX_OBST + K];
  Lines L;
  L.base = buf;
  L.stride = 1;
  const int n_obst = obstacle_lines<ORCA_SLOW_MAX_OBST>(W, p, v, a.radius, a.inv_tho, od, oid, ocnt, L, &overflow);
  typename Src::template List<K, KFULL> nk;
  nk.init(a.k, a.nd_sq);
  src.gather(nk, p, scratch, scratch_slots, mask);
  if (nk.packed_cnt >= 0) nk.unpack_ids();
  int n = n_obst;
  unsigned collisions = 0;
  const float cr = a.radius + a.radius;
  for (int s = 0; s < K; ++s) {
    const int j = nk.id[s];
    if (j >= 0) {
      bool hit;
      buf[n++] = agent_line(p, v, src.pos(j), src.vel(j), HETERO ? a.radius + src.radius(j) : cr, a.inv_th, a.inv_dt, &hit);
      collisions += hit ? 1u : 0u;
    }
  }
  SlowResult r;
  r.n = n;
  r.n_obst = n_obst;
  r.collisions = collisions;
  r.overflow = overflow;
  r.nv = v2(0.f, 0.f);
  r.fail = lp2(mask, true, L, n, a.vmax, pref, false, r.nv);
  float2 nv = r.nv;
  lp3(mask, r.fail < n, L, n, n_obst, r.fail, a.vmax, nv);
  r.nv = nv;
  return r;
}
ORCA_HD void apply_slow_result(const SlowResult& r, AgentCarry& c) {
  c.nv = r.nv;
  c.n = r.n;
  c.n_obst = r.n_obst;
  c.fail = r.fail;
  c.collisions = r.collisions;
  c.overflow = r.overflow;
}

// Back half: Agent::update + reward + bandit update + done test, with c.nv final.
// `live`: the agent's world had not finished its episode when this step began.  In a batch, worlds that
// finish early keep being stepped until the slowest one is done (run_sim), but their idle steps must not
// leak into the episode statistics (the reference's run_sim stops stepping a finished world, ALAN_true.py:121).
template <int POLICY>
ORCA_HD void agent_back(const StepArgs& a, const int env, const int la, const int g, const int estep,
                        const AgentCarry& c, const bool live = true) {
  stat_add_u64_warp(a.stats, STAT_AGENT_STEPS, live ? 1u : 0u);
  stat_add_u64_warp(a.stats, STAT_LP3_CALLS, (live && c.fail < c.n) ? 1u : 0u);

  // ---------------- integrate (Agent::update) ----------------
  const float2 v = c.nv;
  const float2 p = add(c.p, mul(a.dt, v));  // position += velocity * timeStep
  a.pos[g] = p;
  a.vel[g] = v;
  if (a.pos_mirror != nullptr) a.pos_mirror[g] = p;
  if (a.vel_mirror != nullptr) a.vel_mirror[g] = v;

  // ---------------- reward / bandit update ----------------
  if (POLICY == POLICY_RL || POLICY == POLICY_ALAN) {
    const float r_goal = dot(v, c.gdir);
    const float r_polite = dot(v, c.pref);
    float R;
    if (POLICY == POLICY_RL)
      R = a.rl_scale * r_goal + (1.f - a.rl_scale) * r_polite;
    else
      R = a.alan_gamma * r_goal + (1.f - a.alan_gamma) * r_polite;
    if (a.reward != nullptr) a.reward[g] = R;
    stat_add_f64_warp(a.stats, STAT_SUM_REWARD, live ? R : 0.f);
    if (POLICY == POLICY_ALAN) {
      float* wrow = a.alan_w + (size_t)g * a.A;
      // every per-action timer advances in lock step, so the 2 s window expires for all of
      // them on the same step (SURVEY Q7): zero the table, then store the fresh reward
      if (a.alan_window > 0 && ((estep + 1) % a.alan_window) == 0) {
        for (int i = 0; i < a.A; ++i) wrow[i] = 0.f;
      }
      wrow[c.act] = R;
    }
  }

  // ---------------- done test ----------------
  // DONE_GOAL_RADIUS_DEFERRED is the order of run_sim(mode=0) (ALAN_true.py:116-120,631-633): there
  // the preferred velocity of the NEXT doStep is computed (update_pref_vel) before done_test swaps
  // the target, so the step after an arrival still aims at the old goal.  The flag value 2 =
  // "arrived in the previous step, goal swap pending" carries that over one step.
  if (a.done_mode != DONE_NONE) {
    const uint8_t flag = a.done[g];
    if (flag == 2) {
      a.done[g] = 1;
      if (a.goal2 != nullptr) a.goal[g] = a.goal2[g];
    } else if (flag == 0) {
      bool hit;
      if (a.done_mode != DONE_X_BELOW) {
        const float2 d = sub(p, a.goal[g]);
        hit = sqrtf(abs_sq(d)) < 2.f * a.radius;
      } else {
        hit = p.x < a.done_x;
      }
      if (hit) {
        const bool defer = a.done_mode == DONE_GOAL_RADIUS_DEFERRED;
        a.done[g] = defer ? 2 : 1;
        const float t_arr = (float)(estep + 1) * a.dt;
        if (a.arrival != nullptr) a.arrival[g] = t_arr;
        if (a.goal2 != nullptr && !defer) a.goal[g] = a.goal2[g];
        if (a.env_done_cnt != nullptr) counter_inc(&a.env_done_cnt[env]);
        stat_add_u64(a.stats, STAT_FINISHED, 1ull);
        stat_add_f64(a.stats, STAT_SUM_ARRIVAL, (double)t_arr);
        stat_add_f64(a.stats, STAT_SUM_ARRIVAL2, (double)t_arr * (double)t_arr);
      }
    }
  }
  if (a.env_step != nullptr && la == 0 && !a.grid_path) a.env_step[env] = estep + 1;
  stat_add_u64_warp(a.stats, STAT_COLLISIONS, live ? c.collisions : 0u);
  stat_add_u64_warp(a.stats, STAT_OVERFLOW, c.overflow ? 1u : 0u);
}

// Front + LP3 + back for one agent, no work redistribution (host emulation; reference order).
template <int K, bool KFULL, int POLICY, bool HETERO = false, class Src>
ORCA_HD void agent_step_body(const StepArgs& a, const int env, const int la, const int g, float2 p, float2 v,
                             const int estep, const Src& src, const Lines L, const unsigned warp_mask,
                             const float4* agent_params = nullptr) {
  AgentCarry c;
  c.p = p;
  c.v = v;
  c.aim = (POLICY == POLICY_EXTERNAL) ? a.pref[g] : a.goal[g];
  const ObstacleWorld W = Src::kObstacleCull ? global_world_with_cull(a, env) : global_world(a, env);
  if (!agent_front<K, KFULL, POLICY, ORCA_MAX_OBST_LINES, HETERO>(a, env, g, estep, src, W, L, warp_mask, c, agent_params)) return;
  if (c.overflow)
    apply_slow_result(agent_slow_path<K, KFULL, Src, HETERO>(HETERO ? slow_params(a, agent_params, g) : slow_params(a), src, global_world(a, env), L,
                                                             K + ORCA_MAX_OBST_LINES, warp_mask, c.p, c.v, c.pref), c);
  else
    lp3(warp_mask, c.fail < c.n, L, c.n, c.n_obst, c.fail, HETERO ? load_agent_params(agent_params, g).vmax : a.vmax, c.nv);
  agent_back<POLICY>(a, env, la, g, estep, c);
}

#if defined(__CUDACC__)

// register budget of the step kernel: 65536 / (threads * min blocks) registers per thread
#ifndef ORCA_STEP_MAX_THREADS
#define ORCA_STEP_MAX_THREADS 256
#endif
#ifndef ORCA_STEP_MIN_BLOCKS
#define ORCA_STEP_MIN_BLOCKS 3
#endif

#ifndef ORCA_LP3_SMEM_POOL
#define ORCA_LP3_SMEM_POOL 0
#endif
// dynamic shared memory of the step kernels: [pos|vel tile (tile path only)] + lines + LP3 queue
inline size_t step_smem_bytes(int K, int tpb, bool tile, int world_slots = 0, int obst_lines = ORCA_MAX_OBST_LINES,
                              bool hetero = false) {
  size_t b = (size_t)world_slots * 64 + 16;  // staged obstacle tables: 4 x 16 B per vertex slot
  // HETERO kernels: each thread's agent's maxSpeed (for block_lp3) and, in the tile, the agents' radii
  if (hetero) b += (size_t)tpb * (tile ? 8 : 4);
  // per thread: tile (pos, vel) + lines + LP3 queue (nv 8, meta 4, queue entry 1); per block: 8 warp counters
  b += (size_t)tpb * ((tile ? 16 : 0) + (size_t)(K + obst_lines) * 16 + 8 + 4 + 1) + 8 * 4;
#if ORCA_LP3_SMEM_POOL
  b += (size_t)(tpb / 2) * (K + obst_lines) * 16 + 16;  // LP3 projected-line pool
#endif
  return b;
}

// LP3 with block-level work compaction.  Only the agents whose LP2 was infeasible need LP3
// (0-40 % of them, scattered over the block's warps); left in place every warp would walk the
// LP3 loops with a few live lanes.  Instead the block builds a dense queue of those agents and
// threads 0..count-1 each solve one of them -- the ORCA lines already live in shared memory
// (line i of agent o at lines[i * blockDim + o]), so any thread can work on any agent.
//   s_meta[t] = n | n_obst << 8 | fail << 16,  s_nv[t] = LP2 result in / LP3 result out.
// Must be called by every thread of the block (it contains barriers).
#ifndef ORCA_BLOCK_LP3
#define ORCA_BLOCK_LP3 1
#endif
#ifndef ORCA_LP3_SMEM_POOL
#define ORCA_LP3_SMEM_POOL 0
#endif
// HETERO: a solver works on another thread's agent and takes that OWNER's maxSpeed from s_vmax
// (one entry per thread, written before the call); otherwise every agent has `vmax`.
template <int K, bool HETERO = false>
__device__ __forceinline__ void block_lp3(float4* s_lines, float4* s_pool, int* s_meta, float2* s_nv,
                                          unsigned char* s_queue, int* s_warp_cnt, const bool need, const AgentCarry& c, const float vmax,
                                          const bool area_was_borrowed = false, const float* s_vmax = nullptr) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  // the queue area doubled as the in-block neighbor grid during the front half: nobody may
  // overwrite it while another warp still searches its neighbors
  if (area_was_borrowed) __syncthreads();
#if !ORCA_BLOCK_LP3
  {  // in-place variant (kept for A/B measurements): every thread solves its own agent
    Lines L;
    L.base = s_lines + tid;
    L.stride = blockDim.x;
    float2 nv = c.nv;
    lp3(0xffffffffu, need, L, c.n, c.n_obst, c.fail, HETERO ? s_vmax[tid] : vmax, nv);
    s_nv[tid] = nv;
    __syncwarp();
    return;
  }
#endif
  s_meta[tid] = c.n | (c.n_obst << 8) | (c.fail << 16);
  s_nv[tid] = c.nv;
  const unsigned bal = __ballot_sync(0xffffffffu, need);
  if (lane == 0) s_warp_cnt[warp] = __popc(bal);
  __syncthreads();
  int offset = 0, total = 0;
  for (int w = 0; w < nwarps; ++w) {
    const int cw = s_warp_cnt[w];
    offset += (w < warp) ? cw : 0;
    total += cw;
  }
  // queue of the agents that need LP3 from the front of s_queue; from its back, the list of the
  // columns of s_lines whose owner does NOT need LP3 (their lines are dead after LP2)
  {
    const unsigned below = (1u << lane) - 1u;
    if (need)
      s_queue[offset + __popc(bal & below)] = (unsigned char)tid;  // blocks have at most 256 threads
    else
      s_queue[blockDim.x - 1 - ((warp << 5) - offset + __popc(~bal & below))] = (unsigned char)tid;
  }
  __syncthreads();
#if ORCA_LP3_SMEM_POOL
  // projected lines in a shared-memory pool of blockDim/2 entries (SoA, stride = pool size);
  // the queue is drained in passes of that many agents by the first half of the block
  const int pool = blockDim.x >> 1;
  for (int first = 0; first < total; first += pool) {
    if ((warp << 5) < pool && first + (warp << 5) < total) {  // warp-uniform
      const int slot = first + tid;
      const bool mine = slot < total;
      const int owner = mine ? (int)s_queue[slot] : tid;
      const int meta = s_meta[owner];
      Lines L;
      L.base = s_lines + owner;
      L.stride = blockDim.x;
      Lines P;
      P.base = s_pool + tid;
      P.stride = pool;
      float2 nv = s_nv[owner];
      lp3_stored(0xffffffffu, mine, L, meta & 0xff, (meta >> 8) & 0xff, (meta >> 16) & 0xff, HETERO ? s_vmax[owner] : vmax, P, nv);
      if (mine) s_nv[owner] = nv;
    }
  }
#else
  (void)s_pool;
  // Each solver thread borrows one dead column to keep the projected programme of its current
  // LP3 round (computed once per round instead of once per access).  When more than half of the
  // block needs LP3 there are not enough dead columns: the warps beyond them recompute the
  // projections on access (lp3) -- same arithmetic, same result.
  const int nfree = blockDim.x - total;
  int nstored = total < nfree ? total : nfree;
  if (nstored < total) nstored &= ~31;  // whole warps only: the LPs vote warp-wide
  if ((warp << 5) < total) {  // warp-uniform: this warp owns queue entries
    const bool mine = tid < total;
    const int owner = mine ? (int)s_queue[tid] : tid;
    const int meta = s_meta[owner];
    Lines L;
    L.base = s_lines + owner;
    L.stride = blockDim.x;
    float2 nv = s_nv[owner];
    if ((warp << 5) < nstored) {
#if defined(ORCA_DEBUG_CHECKS)
      if (mine) {  // the borrowed column belongs to a thread that is NOT in the LP3 queue, and to nobody else
        const int col = (int)s_queue[blockDim.x - 1 - tid];
        assert(col >= 0 && col < (int)blockDim.x && tid < nfree);
        for (int q = 0; q < total; ++q) assert((int)s_queue[q] != col);
        for (int q = 0; q < nstored; ++q) assert(q == tid || (int)s_queue[blockDim.x - 1 - q] != col);
        assert(owner >= 0 && owner < (int)blockDim.x && (meta & 0xff) <= K + ORCA_MAX_OBST_LINES);
        (void)K;
      }
#endif
      Lines P;
      P.base = s_lines + (mine ? (int)s_queue[blockDim.x - 1 - tid] : tid);
      P.stride = blockDim.x;
      lp3_stored(0xffffffffu, mine, L, meta & 0xff, (meta >> 8) & 0xff, (meta >> 16) & 0xff, HETERO ? s_vmax[owner] : vmax, P, nv);
    } else {
      lp3(0xffffffffu, mine, L, meta & 0xff, (meta >> 8) & 0xff, (meta >> 16) & 0xff, HETERO ? s_vmax[owner] : vmax, nv);
    }
    if (mine) s_nv[owner] = nv;
  }
#endif
  __syncthreads();
}

// order-preserving float -> int mapping for the bounding-box atomicMin
__device__ __forceinline__ int tile_float_to_ordered(float f) {
  const int i = __float_as_int(f);
  return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float tile_ordered_to_float(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }

// Bins the agents of the block's envs into per-env kTileGrid x kTileGrid grids (counting sort in
// shared memory) and points `src` at the tables of the thread's env.  `area` is the LP3 queue
// area, free during the front half of the step: per env 64 counters + 2 bounding-box words +
// 66 cell starts (u16), then one id byte per thread; 13 bytes per thread at most, the area has 14.
// Cell side = neighborDist (+0.1 %), origin = the env's bounding-box corner; coordinates beyond
// the last cell are clamped into it (a superset of the 3 x 3 neighborhood, never a subset).
// The order of ids inside a cell depends on the order of the atomics; the neighbor list does not
// (equal distances are ranked by id).  Called by every thread of the block.
template <class Src>
__device__ __forceinline__ void build_tile_grid(const StepArgs& a, void* area, const bool valid, const int le, const int la,
                                                const float2 p, Src& src) {
  const int tid = threadIdx.x, tpb = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = tpb >> 5;
  const int envs = a.envs_per_block;
  int* cnt = reinterpret_cast<int*>(area);
  int* bbox = cnt + envs * kTileCells;
  unsigned short* start = reinterpret_cast<unsigned short*>(bbox + envs * 2);
  unsigned char* sorted = reinterpret_cast<unsigned char*>(start + envs * kTileStartStride);
  for (int i = tid; i < envs * kTileCells; i += tpb) cnt[i] = 0;
  if (tid < envs * 2) bbox[tid] = 0x7fffffff;
  __syncthreads();
  if (valid) {
    atomicMin(&bbox[2 * le], tile_float_to_ordered(p.x));
    atomicMin(&bbox[2 * le + 1], tile_float_to_ordered(p.y));
  }
  __syncthreads();
  int ck = 0, slot = 0, cx = 0, cy = 0;
  if (valid) {
    const float ox = tile_ordered_to_float(bbox[2 * le]), oy = tile_ordered_to_float(bbox[2 * le + 1]);
    cx = (int)floorf((p.x - ox) * a.tile_grid_inv_cell);
    cy = (int)floorf((p.y - oy) * a.tile_grid_inv_cell);
    cx = cx < 0 ? 0 : (cx >= kTileGrid ? kTileGrid - 1 : cx);
    cy = cy < 0 ? 0 : (cy >= kTileGrid ? kTileGrid - 1 : cy);
    ck = cy * kTileGrid + cx;
    slot = atomicAdd(&cnt[le * kTileCells + ck], 1);
  }
  __syncthreads();
  for (int e = warp; e < envs; e += nwarps) {  // exclusive scan of the 64 cell populations, 2 per lane
    const int c0 = cnt[e * kTileCells + 2 * lane], c1 = cnt[e * kTileCells + 2 * lane + 1];
    int incl = c0 + c1;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int up = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += up;
    }
    const int excl = incl - (c0 + c1);
    start[e * kTileStartStride + 2 * lane] = (unsigned short)excl;
    start[e * kTileStartStride + 2 * lane + 1] = (unsigned short)(excl + c0);
    if (lane == 31) start[e * kTileStartStride + kTileCells] = (unsigned short)incl;
  }
  __syncthreads();
  ORCA_DCHECK(!valid || (start[le * kTileStartStride + ck] + slot < a.N && start[le * kTileStartStride + kTileCells] == a.N));
  ORCA_DCHECK((char*)(sorted + envs * a.N) - (char*)area <= 13 * (int)blockDim.x + 32);  // the borrowed LP3 queue area
  if (valid) sorted[le * a.N + start[le * kTileStartStride + ck] + slot] = (unsigned char)la;
  __syncthreads();
  src.cell_start = start + le * kTileStartStride;
  src.sorted = sorted + le * a.N;
  src.cx = cx;
  src.cy = cy;
  if (valid) {
    src.ox = tile_ordered_to_float(bbox[2 * le]);
    src.oy = tile_ordered_to_float(bbox[2 * le + 1]);
  }
}

// OL = obstacle-line slots per agent.  Worlds whose processed obstacle table has at most 4 vertices (no
// obstacles, or one enclosing wall: BASELINE configs 2 and 3) never give an agent more than 2 obstacle
// lines (the two edges of a corner), so their kernel keeps K + 2 line slots: 222 instead of 286 bytes of
// shared memory per thread, which lets FOUR 256-thread blocks share an SM (64 registers) instead of three.
// Measured (config 2, 214 us at 3 blocks): 2 blocks 272 us, 1 block 480 us -- resident warps are what hides
// the dependent-instruction latency of the LP chains.
// HETERO: per-agent parameters (agent_front); the radii of the block's agents are staged after the
// obstacle tables, next to one maxSpeed per thread for block_lp3.
template <int K, bool KFULL, int POLICY, int OL = ORCA_MAX_OBST_LINES, bool HETERO = false>
__global__ void __launch_bounds__(ORCA_STEP_MAX_THREADS, ((OL <= 2 || K <= 5) ? 4 : ORCA_STEP_MIN_BLOCKS)) step_small_kernel(const StepArgs a, const float4* __restrict__ agent_params) {
  extern __shared__ float4 smem4[];
  const int tpb = blockDim.x;
  // [pos | vel] tile: 2 * tpb float2 = tpb float4 ; lines: (K + OL) * tpb float4 ;
  // LP3 queue: nv (tpb float2), meta (tpb int), warp counters, queue (tpb bytes)
  float2* s_pos = reinterpret_cast<float2*>(smem4);
  float2* s_vel = s_pos + tpb;
  float4* s_lines = smem4 + tpb;
  float4* s_pool = s_lines + (K + OL) * tpb;
  float2* s_nv = reinterpret_cast<float2*>(s_pool + (ORCA_LP3_SMEM_POOL ? (K + OL) * (tpb / 2) : 0));
  int* s_meta = reinterpret_cast<int*>(s_nv + tpb);
  int* s_warp_cnt = s_meta + tpb;
  unsigned char* s_queue = reinterpret_cast<unsigned char*>(s_warp_cnt + 8);
  // staged obstacle tables (16-byte aligned, after the queue): vert_pd | vert_link | bsp | bsp_seg
  float4* s_world = reinterpret_cast<float4*>((reinterpret_cast<uintptr_t>(s_queue + tpb) + 15) & ~(uintptr_t)15);
  float* s_rad = reinterpret_cast<float*>(s_world + 4 * a.world_slots);
  float* s_vmax = s_rad + tpb;

  const int tid = threadIdx.x;
  const int N = a.N;
  const int le = tid / N;
  int la = tid - le * N;
  const int env0 = a.env_base + blockIdx.x * a.envs_per_block;  // first env of this block
  const int env = env0 + le;
  const bool valid = (le < a.envs_per_block) && (env < a.E);
  int g = env * N + la;
  const bool tile_grid = !(OL <= 2) && a.tile_grid_inv_cell > 0.f;  // uniform over the grid; never in the slim kernel

  AgentCarry c;
  c.p = v2(0.f, 0.f);
  c.v = v2(0.f, 0.f);
  c.nv = v2(0.f, 0.f);
  c.n = c.n_obst = c.fail = 0;
  int estep = 0;
  bool env_live = true;
  c.aim = v2(0.f, 0.f);
  if (valid) {
    // consumed after the barrier (with the in-block grid the thread changes agents below and loads it then)
    if (!a.neighbors_only && !tile_grid) c.aim = (POLICY == POLICY_EXTERNAL) ? a.pref[g] : a.goal[g];
    c.p = a.pos[g];
    c.v = a.vel[g];
    s_pos[tid] = c.p;
    s_vel[tid] = c.v;
    if (HETERO) s_rad[tid] = ORCA_LDG(&agent_params[2 * (size_t)g]).x;
    if (a.env_step != nullptr) estep = a.env_step[env];
    // read before the first barrier: nobody of this env (= this block) has counted an arrival of this step yet
    if (a.env_done_cnt != nullptr) env_live = a.env_done_cnt[env] < N;
  }
  // The BSP walk is a chain of dependent node loads done by every agent every step: from global
  // memory each hop is an L2 round trip.  The tables are tiny (64 B per vertex), so the block
  // copies the ones of its envs into shared memory first.
  const int slots = a.world_slots;
  if (slots > 0) {
    const size_t first = (size_t)env0 * a.vert_stride;  // 0 for a shared world
    const size_t limit = (a.vert_stride > 0) ? (size_t)a.E * a.vert_stride : (size_t)a.world_verts;
    for (int s = tid; s < slots; s += tpb) {
      if (first + s < limit) {
        s_world[s] = a.vert_pd[first + s];
        s_world[slots + s] = *reinterpret_cast<const float4*>(&a.vert_link[first + s]);
        s_world[2 * slots + s] = *reinterpret_cast<const float4*>(&a.bsp[first + s]);
        s_world[3 * slots + s] = a.bsp_seg[first + s];
      }
    }
  }
  __syncthreads();
  const unsigned warp_mask = __ballot_sync(0xffffffffu, valid);  // lanes that run the step
  bool alive = valid;
  using Source = TileSourceT<(OL <= 2)>;  // the slim kernel is launched for worlds of at most 32 agents only
  Source src;
  if (tile_grid) {
    build_tile_grid(a, s_nv, valid, le, la, c.p, src);
    // From here on the thread works on the la-th agent of its env IN CELL ORDER instead of agent la:
    // the lanes of a warp then sit in the same few cells, so their candidate runs have similar
    // lengths, they accept and insert at similar times and they walk the obstacle BSP along the
    // same path (live lanes per instruction in config 4: 17 with agent order).  A pure permutation of
    // who computes what: results are unchanged.
    if (valid) {
      la = (int)src.sorted[la];
      g = env * N + la;
      c.p = s_pos[le * N + la];
      c.v = s_vel[le * N + la];
      int cx = (int)floorf((c.p.x - src.ox) * a.tile_grid_inv_cell);
      int cy = (int)floorf((c.p.y - src.oy) * a.tile_grid_inv_cell);
      src.cx = cx < 0 ? 0 : (cx >= kTileGrid ? kTileGrid - 1 : cx);
      src.cy = cy < 0 ? 0 : (cy >= kTileGrid ? kTileGrid - 1 : cy);
      if (!a.neighbors_only) c.aim = (POLICY == POLICY_EXTERNAL) ? a.pref[g] : a.goal[g];
    }
  }
  c.overflow = false;
  if (valid) {
    ObstacleWorld W = global_world(a, env);
    if (slots > 0) {
      const int off = le * a.vert_stride;  // 0 for a shared world
      W.vert_pd = s_world + off;
      W.vert_link = reinterpret_cast<const int4*>(s_world + slots) + off;
      W.bsp = reinterpret_cast<const int4*>(s_world + 2 * slots) + off;
      W.bsp_seg = s_world + 3 * slots + off;
    }
    Lines L;
    L.base = s_lines + tid;
    L.stride = tpb;
    src.env_pos = s_pos + le * N;
    src.env_vel = s_vel + le * N;
    src.n = N;
    src.self = la;
    src.full_range_sq = HETERO ? ORCA_LDG(&agent_params[2 * (size_t)g + 1]).x : a.nd_sq;
    if (HETERO) src.env_rad = s_rad + le * N;
    alive = agent_front<K, KFULL, POLICY, OL, HETERO>(a, env, g, estep, src, W, L, warp_mask, c, agent_params);
    if (HETERO) s_vmax[tid] = ORCA_LDG(&agent_params[2 * (size_t)g]).y;
  }
  if (a.neighbors_only) return;  // uniform over the grid
  block_lp3<K, HETERO>(s_lines, s_pool, s_meta, s_nv, s_queue, s_warp_cnt, alive && !c.overflow && c.fail < c.n, c, a.vmax, tile_grid,
                       s_vmax);
  const unsigned slow_mask = __ballot_sync(0xffffffffu, alive && c.overflow);
  if (!alive) return;
  c.nv = s_nv[tid];
  if (c.overflow) {  // rare: more obstacle edges / lines than the fast path holds
    // Everything the slow path needs is rebuilt HERE from scalars (a plain scan of the env's tile --
    // it yields the same list as the in-block grid -- and the obstacle tables in global memory), so
    // that nothing of the hot path above has to live in local memory for the sake of this call.
    Lines L;
    L.base = s_lines + tid;
    L.stride = tpb;
    Source scan;
    scan.env_pos = s_pos + le * N;
    scan.env_vel = s_vel + le * N;
    scan.n = N;
    scan.self = la;
    if (HETERO) scan.env_rad = s_rad + le * N;
    apply_slow_result(agent_slow_path<K, KFULL, Source, HETERO>(HETERO ? slow_params(a, agent_params, g) : slow_params(a), scan, global_world(a, env), L,
                                                                K + OL, slow_mask, c.p, c.v, c.pref), c);
  }
  agent_back<POLICY>(a, env, la, g, estep, c, env_live);
}

#endif  // __CUDACC__

}  // namespace orca
