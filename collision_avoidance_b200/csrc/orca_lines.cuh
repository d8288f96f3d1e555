// orca_lines.cuh -- the ORCA half-planes every agent would solve in a step from a given (pos, vel)
// state: RVO2's getAgentNumORCALines / getAgentORCALine for a whole batch (orca_agent_lines).
//
// The step kernels build these lines in shared memory and drop them after the LP.  Recording them
// there would grow kernels whose instruction cache and registers are already their limits
// (DESIGN.md section 5), so this is a query of its own: one thread per agent rebuilds its programme
// the way the uncapped path (agent_slow_path) does -- obstacle_neighbors / obstacle_lines with room
// for ORCA_SLOW_MAX_OBST edges and lines, a neighbor source's gather, agent_line -- i.e. with the
// float32 expressions of the step, so the lines are the step's bit for bit:
//   * obstacle lines first, in obstacle-neighbor order (edges RVO2 finds "already covered" skipped),
//   * agent lines after them, in neighbor order: ascending (distSq, id),
//   * each line (point.x, point.y, direction.x, direction.y).
// They depend on the pre-step positions and velocities, the obstacle world, the agent's parameters
// and 1 / timeStep (collision branch), not on the preferred velocity.
//
// Tile kernel (worlds of at most 256 agents): whole envs per block, (pos, vel) of the block's envs
// staged in shared memory, candidates = a plain scan of the env (TileSource without its in-block grid:
// same list, the order is (distSq, id)).  Grid kernel (larger worlds): the step's cell-sorted snapshot
// (grid prep G1-G4 of orca_grid.cuh, run again by the caller) and GridSource.
//
// Per-agent parameters: a runtime test of the table pointer (this is not a hot step kernel); lists
// are the KFULL = false ones, exact for any k <= K.
#pragma once

#include "orca_grid.cuh"

namespace orca {

// Where the lines go.  Row r < max_lines of agent g: lines[g * max_lines + r]; later rows are dropped,
// the counts are complete.  cnt[g] = -1: the agent exceeds even the uncapped path's capacity (the step
// counts it in STAT_OVERFLOW); its rows are then unspecified.  obst_cnt may be nullptr.
struct LinesOut {
  float4* lines;
  int* cnt;
  int* obst_cnt;
  int max_lines;
};

// candidate-buffer slots per thread of the tile kernel (the ranked searches of worlds of <= 32 agents
// need 9 of them; beyond that the size only sets how often a warp drains its buffers)
constexpr int kLinesScratch = 12;

// One agent's programme.  `walk` = false: the obstacle-free map says no edge is in range.
// `scratch` = the agent's candidate-buffer column, `mask` = the lanes of the warp that call this together.
template <int K, class Src>
ORCA_HD void agent_orca_lines(const SlowParams q, const bool hetero, const Src& src, const ObstacleWorld& W, const bool walk,
                              const Lines scratch, const int scratch_slots, const unsigned mask, const float2 p,
                              const float2 v, const LinesOut o, const size_t g) {
  bool overflow = false;
  float od[ORCA_SLOW_MAX_OBST];
  int oid[ORCA_SLOW_MAX_OBST];
  int ocnt = 0;
  if (walk) obstacle_neighbors<ORCA_SLOW_MAX_OBST>(W, p, q.obst_range_sq, od, oid, &ocnt, &overflow);
  // obstacle lines are read back by the "already covered" test while they are built: a private buffer
  float4 obuf[ORCA_SLOW_MAX_OBST];
  Lines obst;
  obst.base = obuf;
  obst.stride = 1;
  const int n_obst = obstacle_lines<ORCA_SLOW_MAX_OBST>(W, p, v, q.radius, q.inv_tho, od, oid, ocnt, obst, &overflow);
  float4* row = o.lines + g * (size_t)o.max_lines;
  for (int i = 0; i < n_obst && i < o.max_lines; ++i) row[i] = obuf[i];

  typename Src::template List<K, false> nk;
  nk.init(q.k, q.nd_sq);
  src.gather(nk, p, scratch, scratch_slots, mask);
  if (nk.packed_cnt >= 0) nk.unpack_ids();
  int n = n_obst;
  const float cr = q.radius + q.radius;
  for (int s = 0; s < K; ++s) {
    const int j = nk.id[s];
    if (j >= 0) {
      bool hit;
      const float4 ln = agent_line(p, v, src.pos(j), src.vel(j), hetero ? q.radius + src.radius(j) : cr, q.inv_th, q.inv_dt, &hit);
      if (n < o.max_lines) row[n] = ln;
      ++n;
      ORCA_COUNT(10, hit ? 1 : 0);  // collision lines (host test builds)
    }
  }
  o.cnt[g] = overflow ? -1 : n;
  if (o.obst_cnt != nullptr) o.obst_cnt[g] = overflow ? -1 : n_obst;
}

#if defined(__CUDACC__)

constexpr int kLinesTileThreads = 256;
constexpr int kLinesGridThreads = 128;

// shared memory of the tile kernel: (pos, vel) tile + candidate buffers + radii (per-agent parameters)
inline size_t lines_tile_smem_bytes(int tpb) { return (size_t)tpb * (16 + kLinesScratch * 16 + 4); }

// a.envs_per_block whole envs per block; a.pos / a.vel = the state the lines are built from
template <int K>
__global__ void __launch_bounds__(kLinesTileThreads) agent_lines_tile_kernel(const StepArgs a, const float4* __restrict__ agent_params,
                                                                             const LinesOut o) {
  extern __shared__ float4 smem4[];
  const int tpb = blockDim.x;
  float2* s_pos = reinterpret_cast<float2*>(smem4);
  float2* s_vel = s_pos + tpb;
  float4* s_scratch = smem4 + tpb;
  float* s_rad = reinterpret_cast<float*>(s_scratch + kLinesScratch * tpb);
  const int tid = threadIdx.x;
  const int N = a.N;
  const int le = tid / N;
  const int la = tid - le * N;
  const int env = blockIdx.x * a.envs_per_block + le;
  const bool valid = le < a.envs_per_block && env < a.E;
  const size_t g = (size_t)env * N + la;
  const bool hetero = agent_params != nullptr;
  float2 p = v2(0.f, 0.f), v = v2(0.f, 0.f);
  if (valid) {
    p = a.pos[g];
    v = a.vel[g];
    s_pos[tid] = p;
    s_vel[tid] = v;
    if (hetero) s_rad[tid] = ORCA_LDG(&agent_params[2 * g]).x;
  }
  __syncthreads();
  const unsigned mask = __ballot_sync(0xffffffffu, valid);
  if (!valid) return;
  TileSource src;
  src.env_pos = s_pos + le * N;
  src.env_vel = s_vel + le * N;
  src.n = N;
  src.self = la;
  if (hetero) src.env_rad = s_rad + le * N;
  Lines scratch;
  scratch.base = s_scratch + tid;
  scratch.stride = tpb;
  agent_orca_lines<K>(hetero ? slow_params(a, agent_params, (int)g) : slow_params(a), hetero, src, global_world(a, env), true,
                      scratch, kLinesScratch, mask, p, v, o, g);
}

// thread j = the agent in sorted slot j of the grid prep's snapshot (a warp's agents share cells)
template <int K>
__global__ void __launch_bounds__(kLinesGridThreads) agent_lines_grid_kernel(const StepArgs a, const float4* __restrict__ spv,
                                                                             const int* __restrict__ sidx,
                                                                             const int* __restrict__ cell_start,
                                                                             const GridParams* __restrict__ gpp,
                                                                             const float4* __restrict__ agent_params,
                                                                             const LinesOut o) {
  extern __shared__ float4 smem4[];
  const int T = a.E * a.N;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = j < T;
  const unsigned mask = __ballot_sync(0xffffffffu, valid);
  if (!valid) return;
  const bool hetero = agent_params != nullptr;
  const int g = sidx[j];
  const int env = g / a.N;
  const SlowParams q = hetero ? slow_params(a, agent_params, g) : slow_params(a);
  GridSource src;
  src.spv = spv;
  src.orig = sidx;
  src.cell_start = cell_start;
  src.gp = *gpp;
  src.env = env;
  src.env_n0 = env * a.N;
  src.self = j;
  src.full_range_sq = q.nd_sq;  // the list starts from the full range: no second pass
  if (hetero) src.params = agent_params;
  const float4 pv = spv[j];
  const float2 p = v2(pv.x, pv.y), v = v2(pv.z, pv.w);
  const ObstacleWorld W = global_world_with_cull(a, env);
  Lines scratch;
  scratch.base = smem4 + threadIdx.x;
  scratch.stride = blockDim.x;
  agent_orca_lines<K>(q, hetero, src, W, obstacles_may_be_near(W, p), scratch, K + ORCA_MAX_OBST_LINES, mask, p, v, o,
                      (size_t)g);
}

#endif  // __CUDACC__

}  // namespace orca
