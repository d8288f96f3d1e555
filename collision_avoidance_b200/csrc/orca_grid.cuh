// orca_grid.cuh -- uniform-grid neighbor pipeline for large worlds (agents_per_env > 256,
// BASELINE config 5: one world of 1,000,000 agents).
//
// Replaces RVO2's per-step kd-tree (KdTree::buildAgentTree + queryAgentTreeRecursive, reached
// through doStep: collision_avoidence_env.py:385,448 ; ALAN_true.py:601,632 ; SURVEY A.2) by
// FIVE launches per step:
//   G1 grid_bounds    min/max of all positions; the last block to finish derives the grid (cell
//                     size = neighborDist, origin, dims) and re-arms the accumulators  (rd 8 B/agent)
//   G2 grid_count     cell key per agent + slot inside the cell (atomics); also snapshots and
//                     bumps the env step counters                              (rd 8, wr 8)
//   G3 grid_scan      exclusive scan of the cell populations, ONE pass with decoupled look-back
//                     (epoch-tagged tile states: nothing to reset); zeroes the counters it read
//   G4 grid_scatter   counting-sort scatter of (pos, vel) as one float4 + id   (rd 28, wr 20)
//   G5 step_grid      fused step, candidates = the 3 x 3 cells around the agent
// A counting sort by cell key is all the "cell-key sort" this needs: keys are dense small
// integers, and the order inside a cell is irrelevant because equal distances are ranked by
// agent id (NearestK::offer_ranked), which also makes the result independent of the atomics'
// arrival order.  The sorted copies of pos / vel are the PRE-step snapshot every candidate read
// goes to, so the step itself updates the caller's arrays in place (RVO2's two-phase doStep).
//
// Positions outside the grid box are clamped into the border cells: clamping is monotone and
// 1-Lipschitz on cell coordinates, so two agents within one cell size of each other always
// land in cells at most one apart -- the 3 x 3 scan never misses a neighbor.
#pragma once

#if defined(__CUDACC__)
#include <cuda_runtime.h>
#endif

#include <atomic>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <string>

#include "orca_step_small.cuh"

namespace orca {

struct GridParams {
  float origin_x, origin_y, inv_cell;
  int W, H;    // cells per env
  int ncells;  // E * W * H
};

// Cell size: neighbor_dist / kGridReach (plus 0.1 %), searched kGridReach cells out in every direction.
// The 0.1 % absorbs the rounding of (x - origin) * inv_cell (about 1.2e-7 relative, i.e. < 1e-3 cells
// up to ~8000 cells per side), so two agents closer than neighbor_dist always land at most kGridReach
// cells apart; exactly neighbor_dist (inv_cell = 0.2f is a hair above 1/5) would let pairs at
// 4.9999999 fall one cell too far.  The search skips rows and columns of cells whose gap to the agent
// exceeds the list's CURRENT k-th distance (with a margin of kGapMargin cells for the same rounding).
// Measured, config 5: reach 1 (cells of nd, 3 x 3) 457 us; reach 2 (cells of nd / 2, 5 x 5 with
// pruning: 30 instead of 56 candidates per agent) 464 us -- the candidate walk is warp-synchronous
// (its length is the longest lane's), and the insertions, which dominate, depend on the threshold, not
// on how many candidates are looked at.
#ifndef ORCA_GRID_REACH
#define ORCA_GRID_REACH 1
#endif
constexpr int kGridReach = ORCA_GRID_REACH;  // cells searched on each side of the agent's own
constexpr float kGapMargin = 4.0e-3f;        // cells
ORCA_HD float grid_cell_size(float neighbor_dist) { return (neighbor_dist > 0.f ? neighbor_dist : 1.f) * (1.001f / kGridReach); }

#if defined(__CUDACC__)
struct GridScratch {
  int T = 0;          // agents covered by the allocation
  int cap_cells = 0;  // capacity of the cell arrays
  int E = 0;          // envs covered by the allocation
  int sm_count = 0;   // multiprocessors of the device the scratch lives on
  unsigned epoch = 0; // launch counter of the scan: tags the tile states, so they never need a reset
  float4* sorted_pv = nullptr;  // (pos.x, pos.y, vel.x, vel.y) in cell order: the pre-step snapshot
  int* sorted_idx = nullptr;
  int* key = nullptr;
  int* slot = nullptr;
  int* cell_count = nullptr;  // [cap_cells + 1], all zero between steps (the scan re-zeroes what it reads)
  int* cell_start = nullptr;  // [cap_cells + 1]
  unsigned long long* tile_state = nullptr;  // [scan tiles] decoupled look-back states
  int* counters = nullptr;    // [0..3] bounds (order-preserving ints: min x, min y, max x, max y),
                              // [4] blocks of G1 that finished, [5] tile ticket of G3
  int* env_step_snap = nullptr;  // [E] step counters as they were before this step
  GridParams* params = nullptr;
};

inline void grid_free(GridScratch& g) {
  cudaFree(g.sorted_pv);
  cudaFree(g.sorted_idx);
  cudaFree(g.key);
  cudaFree(g.slot);
  cudaFree(g.cell_count);
  cudaFree(g.cell_start);
  cudaFree(g.tile_state);
  cudaFree(g.counters);
  cudaFree(g.env_step_snap);
  cudaFree(g.params);
  g = GridScratch();
}
#endif

// Candidates of an agent = agents in the 3 x 3 cells around it, read from the cell-sorted
// snapshot.  Entries are identified by their sorted slot; `orig` maps a slot to the agent id.
struct GridSource {
  static constexpr bool kObstacleCull = true;
  const float4* spv;  // (pos, vel) per sorted slot
  const int* orig;
  const int* cell_start;
  GridParams gp;
  int env;     // env of the agent
  int env_n0;  // global id of the env's first agent
  int self;    // sorted slot of the agent itself

  template <int K, bool KFULL>
  using List = NearestK<K, KFULL>;
  struct Before {
    const int* orig;
    ORCA_HD bool operator()(int a, int b) const { return b >= 0 && ORCA_LDG(&orig[a]) < ORCA_LDG(&orig[b]); }
  };

  ORCA_HD static int cell_coord(float x, float origin, float inv_cell, int n) {
    int c = (int)floorf((x - origin) * inv_cell);
    c = c < 0 ? 0 : c;
    return c >= n ? n - 1 : c;
  }

  ORCA_HD bool threshold_search() const { return true; }
  float full_range_sq = 0.f;  // the neighbor range (squared), for the second pass
  // The list arrives initialised with its STARTING threshold (agent_front): the neighbor range or last
  // step's tighter bound.  Lanes whose list did not fill up from a tighter start search again from the
  // full range in a second pass over the same rows.
  template <class NK>
  ORCA_HD void gather(NK& nk, float2 p, const Lines& scratch, int scratch_slots, unsigned mask) const {
    // cell coordinates as floats: same expression as cell_coord, so "agent q is in cell c" means
    // floor(f(q)) == c for exactly this f
    const float fx = (p.x - gp.origin_x) * gp.inv_cell, fy = (p.y - gp.origin_y) * gp.inv_cell;
    const int cx = cell_coord(p.x, gp.origin_x, gp.inv_cell, gp.W);
    const int cy = cell_coord(p.y, gp.origin_y, gp.inv_cell, gp.H);
    const float inv_cell_sq = gp.inv_cell * gp.inv_cell;
    const int base = env * gp.W * gp.H;
    Before before;
    before.orig = orig;
    CandidateBuffer buf;
    buf.base = scratch.base;
    buf.stride = scratch.stride;
    buf.cap = 2 * scratch_slots;  // two (distSq, id) entries per 16-byte line slot
    buf.cnt = 0;
    auto insert = [&nk, &before](float d, int id) { nk.offer_ranked(d, id, before); };
    // 2 * kGridReach + 1 rows of cells, the agent's own first, then outwards: the nearest candidates
    // tighten the threshold early (the list itself does not depend on the visiting order).  The cells
    // (x0..x1, row) have consecutive keys, i.e. they are ONE contiguous range of the sorted arrays;
    // lanes walk their own ranges but vote together on every iteration.
    // A row is skipped, and its column range narrowed, by the gap (in cells, minus a rounding margin)
    // between the agent and the row / column: an agent binned there cannot be nearer than the gap.
    // Border cells also hold the agents clamped into them from outside the box, which are farther
    // still; the agent's OWN row and column are never pruned (it may itself be a clamped one).
    constexpr int kRows = 2 * kGridReach + 1;
    bool enabled = true;
#pragma unroll 1
    for (int rr = 0; rr < 2 * kRows; ++rr) {
      if (rr == kRows) {  // second pass?
        buf.drain(mask, insert);
        enabled = nk.range_sq < full_range_sq && !nk.full();
        if (!ORCA_ANY(mask, enabled)) break;
        if (enabled) nk.init(nk.k, full_range_sq);
      }
      const int r = rr < kRows ? rr : rr - kRows;
      const int dy = (r & 1) ? -((r + 1) >> 1) : (r >> 1);  // 0, -1, +1, -2, +2
      const int yy = cy + dy;
      int q = 0, last = 0;
      if (enabled && yy >= 0 && yy < gp.H) {
        int x0 = cx - kGridReach > 0 ? cx - kGridReach : 0;
        int x1 = cx + kGridReach < gp.W ? cx + kGridReach : gp.W - 1;
        bool visit = true;
        if (kGridReach > 1) {  // pruning pays only with cells finer than the range (measured: costs 6 us at reach 1)
          float gy = (dy < 0) ? fy - (float)(yy + 1) : ((dy > 0) ? (float)yy - fy : 0.f);
          gy = fmaxf(gy - kGapMargin, 0.f);
          const float rem = nk.thresh() * inv_cell_sq - gy * gy;  // what is left for the column gap, in cells^2
          visit = rem >= 0.f;
          while (visit && x0 < cx) {
            const float gx = fmaxf(fx - (float)(x0 + 1) - kGapMargin, 0.f);
            if (!(gx * gx > rem)) break;
            ++x0;
          }
          while (visit && x1 > cx) {
            const float gx = fmaxf((float)x1 - fx - kGapMargin, 0.f);
            if (!(gx * gx > rem)) break;
            --x1;
          }
        }
        if (visit) {
          q = ORCA_LDG(&cell_start[base + yy * gp.W + x0]);
          last = ORCA_LDG(&cell_start[base + yy * gp.W + x1 + 1]);
        }
      }
      // the position of the NEXT candidate is fetched while the current one is tested and parked:
      // the load (L1 / L2 latency) is the longest single wait of this loop
      float2 nxt = v2(0.f, 0.f);
      if (q < last) nxt = pos(q);
      // two candidates per pair of warp votes (loop condition, buffer check): the votes were a third
      // of this loop's instructions
      while (ORCA_ANY(mask, q < last)) {
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          if (q < last) {
            const float2 o = nxt;
            const int cur = q;
            ++q;
            if (q < last) nxt = pos(q);
            if (cur != self) {
              const float d = abs_sq(sub(p, o));
              if (d <= nk.thresh()) buf.push(d, cur);
            }
          }
        }
        buf.drain_if_full(mask, insert, 2);
      }
    }
    buf.drain(mask, insert);
  }
  ORCA_HD float2 pos(int q) const { return ORCA_LDG(reinterpret_cast<const float2*>(&spv[q])); }
  ORCA_HD float2 vel(int q) const { return ORCA_LDG(reinterpret_cast<const float2*>(&spv[q]) + 1); }
  ORCA_HD int local_id(int q) const { return ORCA_LDG(&orig[q]) - env_n0; }
  // per-agent records (orca_set_agent_params' table, HETERO kernels only): the radius by original id
  const float4* params = nullptr;
  ORCA_HD float radius(int q) const { return ORCA_LDG(&params[2 * (size_t)ORCA_LDG(&orig[q])]).x; }
};

#if defined(__CUDACC__)

// order-preserving float <-> int mapping for atomicMin / atomicMax
__device__ __forceinline__ int float_to_ordered(float f) {
  const int i = __float_as_int(f);
  return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float ordered_to_float(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }

// Grid geometry from the bounding box; the cell is enlarged if the box would need more cells than allocated.
__device__ __forceinline__ void grid_derive_params(const int* bounds, float neighbor_dist, int E, int cap_cells, GridParams* out) {
  float mnx = ordered_to_float(bounds[0]), mny = ordered_to_float(bounds[1]);
  float mxx = ordered_to_float(bounds[2]), mxy = ordered_to_float(bounds[3]);
  if (!(mnx <= mxx) || !(mny <= mxy)) {
    mnx = mny = 0.f;
    mxx = mxy = 0.f;
  }
  float cell = grid_cell_size(neighbor_dist);
  int W, H;
  for (;;) {
    const float fw = floorf((mxx - mnx) / cell) + 1.f, fh = floorf((mxy - mny) / cell) + 1.f;
    if (fw * fh * (float)E <= (float)cap_cells && fw < 1.0e9f && fh < 1.0e9f) {
      W = (int)fw;
      H = (int)fh;
      break;
    }
    cell *= 1.5f;
  }
  out->origin_x = mnx;
  out->origin_y = mny;
  out->inv_cell = 1.0f / cell;
  out->W = W;
  out->H = H;
  out->ncells = E * W * H;
}

__global__ void grid_arm_kernel(int* counters) {  // first use only: the kernels re-arm the counters themselves
  counters[0] = counters[1] = 0x7fffffff;
  counters[2] = counters[3] = (int)0x80000000;
  counters[4] = counters[5] = 0;
}

// G1: bounding box of all positions -> grid geometry.  One atomic quadruple per BLOCK (it was one per
// warp: 19,000 same-address atomics took longer than reading the positions); the block that finishes
// last derives the geometry and re-arms the accumulators for the next step, so neither a reset nor a
// parameter kernel is launched.
constexpr int kBoundsThreads = 512;
__global__ void __launch_bounds__(kBoundsThreads) grid_bounds_kernel(const float2* __restrict__ pos, int T, int* counters,
                                                                      float neighbor_dist, int E, int cap_cells,
                                                                      GridParams* params) {
  float mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < T; i += gridDim.x * blockDim.x) {
    const float2 p = pos[i];
    if (isfinite(p.x) && isfinite(p.y)) {
      mnx = fminf(mnx, p.x);
      mny = fminf(mny, p.y);
      mxx = fmaxf(mxx, p.x);
      mxy = fmaxf(mxy, p.y);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mnx = fminf(mnx, __shfl_xor_sync(0xffffffffu, mnx, o));
    mny = fminf(mny, __shfl_xor_sync(0xffffffffu, mny, o));
    mxx = fmaxf(mxx, __shfl_xor_sync(0xffffffffu, mxx, o));
    mxy = fmaxf(mxy, __shfl_xor_sync(0xffffffffu, mxy, o));
  }
  __shared__ float s_red[4][kBoundsThreads / 32];
  __shared__ bool s_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) {
    s_red[0][warp] = mnx;
    s_red[1][warp] = mny;
    s_red[2][warp] = mxx;
    s_red[3][warp] = mxy;
  }
  __syncthreads();
  if (warp == 0) {
    const bool in = lane < kBoundsThreads / 32;
    mnx = in ? s_red[0][lane] : INFINITY;
    mny = in ? s_red[1][lane] : INFINITY;
    mxx = in ? s_red[2][lane] : -INFINITY;
    mxy = in ? s_red[3][lane] : -INFINITY;
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      mnx = fminf(mnx, __shfl_xor_sync(0xffffffffu, mnx, o));
      mny = fminf(mny, __shfl_xor_sync(0xffffffffu, mny, o));
      mxx = fmaxf(mxx, __shfl_xor_sync(0xffffffffu, mxx, o));
      mxy = fmaxf(mxy, __shfl_xor_sync(0xffffffffu, mxy, o));
    }
    if (lane == 0) {
      atomicMin(&counters[0], float_to_ordered(mnx));
      atomicMin(&counters[1], float_to_ordered(mny));
      atomicMax(&counters[2], float_to_ordered(mxx));
      atomicMax(&counters[3], float_to_ordered(mxy));
      __threadfence();
      s_last = atomicAdd(&counters[4], 1) == (int)gridDim.x - 1;
    }
  }
  __syncthreads();
  if (s_last && threadIdx.x == 0) {
    __threadfence();
    int b[4];
    for (int i = 0; i < 4; ++i) b[i] = atomicAdd(&counters[i], 0);  // the other blocks' atomics, read at L2
    grid_derive_params(b, neighbor_dist, E, cap_cells, params);
    counters[0] = counters[1] = 0x7fffffff;
    counters[2] = counters[3] = (int)0x80000000;
    counters[4] = 0;
  }
}

// G2: cell key + slot per agent.  Its first E threads also copy the env step counters aside and bump
// them: an env spans many blocks of the step kernel, so those read the copy while the caller's
// counters already hold the value the call leaves behind.
__global__ void __launch_bounds__(256) grid_count_kernel(const float2* __restrict__ pos, int T, int N,
                                                         const GridParams* __restrict__ gpp, int* cell_count,
                                                         int* __restrict__ key, int* __restrict__ slot, int* env_step,
                                                         const int* __restrict__ env_done_cnt,
                                                         int* __restrict__ env_step_snap, int E, int bump) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (env_step != nullptr && i < E) {
    const int s0 = env_step[i];
    env_step_snap[i] = s0;
    if (bump) env_step[i] = s0 + 1;
  }
  // [E, 2E): how many agents of the env had arrived when this step began (the step kernel's blocks of one
  // env must agree on whether the episode was still running; its own arrivals are counted as it goes)
  if (i < E) env_step_snap[E + i] = (env_done_cnt != nullptr) ? env_done_cnt[i] : 0;
  if (i >= T) return;
  const GridParams gp = *gpp;
  const float2 p = pos[i];
  const int cx = GridSource::cell_coord(p.x, gp.origin_x, gp.inv_cell, gp.W);
  const int cy = GridSource::cell_coord(p.y, gp.origin_y, gp.inv_cell, gp.H);
  const int k = (i / N) * gp.W * gp.H + cy * gp.W + cx;
  key[i] = k;
  slot[i] = atomicAdd(&cell_count[k], 1);
}

// ---- G3: exclusive scan of cell_count[0 .. ncells) into cell_start (ncells + 1 entries) --------------
// Single pass, decoupled look-back (Merrill & Garland): a block takes the next tile from a ticket
// counter, publishes the tile's sum, walks back over its predecessors' states until it meets an
// inclusive prefix, publishes its own.  A state word = epoch << 34 | flag << 32 | value; states of an
// earlier launch carry an older epoch and read as "not there yet", so nothing is ever cleared.
// The counters a tile has read are zeroed on the way: cell_count is all zero again for the next step.
constexpr int kScanThreads = 256;
constexpr int kScanItems = 8;  // per thread
constexpr int kScanTile = kScanThreads * kScanItems;

__device__ __forceinline__ int block_exclusive_scan(int v, int* total) {
  __shared__ int warp_sums[kScanThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) warp_sums[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int w = lane < kScanThreads / 32 ? warp_sums[lane] : 0;
#pragma unroll
    for (int o = 1; o < kScanThreads / 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += t;
    }
    if (lane < kScanThreads / 32) warp_sums[lane] = w;
  }
  __syncthreads();
  const int warp_off = warp > 0 ? warp_sums[warp - 1] : 0;
  *total = warp_sums[kScanThreads / 32 - 1];
  __syncthreads();
  return warp_off + inc - v;
}

__global__ void __launch_bounds__(kScanThreads) grid_scan_kernel(int* __restrict__ cnt, const GridParams* __restrict__ gpp,
                                                                 unsigned long long* tile_state, int* ticket,
                                                                 unsigned epoch, int* __restrict__ start) {
  __shared__ int s_tile, s_prefix;
  if (threadIdx.x == 0) {
    const int t = atomicAdd(ticket, 1);
    if (t == (int)gridDim.x - 1) *ticket = 0;  // every block has drawn: re-arm for the next launch
    s_tile = t;
  }
  __syncthreads();
  const int tile = s_tile;
  const int n = gpp->ncells;
  if (tile * kScanTile >= n) return;  // tiles are handed out in order: everything in front of a live tile is live
  const int base = tile * kScanTile + threadIdx.x * kScanItems;
  int v[kScanItems];
  int s = 0;
#pragma unroll
  for (int t = 0; t < kScanItems; ++t) {
    v[t] = 0;
    if (base + t < n) {
      v[t] = cnt[base + t];
      cnt[base + t] = 0;
    }
    s += v[t];
  }
  int total;
  const int local = block_exclusive_scan(s, &total);
  const unsigned long long tag = (unsigned long long)epoch << 34;
  if (threadIdx.x < 32) {  // warp 0 looks back over 32 predecessors at a time
    volatile unsigned long long* st = tile_state;
    const int lane = threadIdx.x;
    if (lane == 0 && tile > 0) st[tile] = tag | (1ull << 32) | (unsigned)total;  // aggregate available
    int prefix = 0;
    for (int hi = tile - 1; hi >= 0; hi -= 32) {
      const int pidx = hi - lane;
      unsigned long long w = tag | (2ull << 32);  // lanes in front of tile 0: an inclusive prefix of 0
      if (pidx >= 0) {
        do {
          w = st[pidx];
        } while ((w >> 34) != epoch || ((w >> 32) & 3ull) == 0ull);
      }
      const unsigned incl = __ballot_sync(0xffffffffu, ((w >> 32) & 3ull) == 2ull);
      // nearest predecessor with an inclusive prefix: everything nearer contributes its aggregate
      const int stop = incl ? __ffs((int)incl) - 1 : 31;
      int v = (lane <= stop) ? (int)(unsigned)(w & 0xffffffffull) : 0;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      prefix += v;
      if (incl) break;
    }
    if (lane == 0) {
      __threadfence();
      st[tile] = tag | (2ull << 32) | (unsigned)(prefix + total);  // inclusive prefix available
      s_prefix = prefix;
    }
  }
  __syncthreads();
  int off = local + s_prefix;
#pragma unroll
  for (int t = 0; t < kScanItems; ++t) {
    if (base + t < n) start[base + t] = off;
    off += v[t];
    if (base + t == n - 1) start[n] = off;  // sentinel: total agent count
  }
}

// G4: one 16-byte store of (pos, vel) + one 4-byte store of the id per agent, to its sorted slot
__global__ void __launch_bounds__(256) grid_scatter_kernel(const float2* __restrict__ pos, const float2* __restrict__ vel,
                                                           int T, const int* __restrict__ key, const int* __restrict__ slot,
                                                           const int* __restrict__ cell_start, float4* __restrict__ spv,
                                                           int* __restrict__ sidx) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= T) return;
  const int j = cell_start[key[i]] + slot[i];
  ORCA_DCHECK(j >= 0 && j < T);
  const float2 p = pos[i], v = vel[i];
  spv[j] = make_float4(p.x, p.y, v.x, v.y);
  sidx[j] = i;
}

#ifndef ORCA_GRID_TPB
#define ORCA_GRID_TPB 64  // threads per block of the uniform-grid step kernel: 32 / 64 / 128 / 256 -> 466 / 469 / 483 / 506 us (cfg 5)
#endif
// G6: the fused step over the cell-sorted order.  Thread j handles the agent in sorted slot j, so a
// warp's agents share cells (coherent candidate loops, cache-friendly reads).
// OL: obstacle-line slots per agent, as in step_small_kernel: the K + 2 variant (worlds of at most 4
// obstacle vertices) fits 1024 instead of 768 threads per SM.
// HETERO: per-agent parameters (agent_front), neighbor radii gathered from the records by original id.
template <int K, bool KFULL, int POLICY, int OL = ORCA_MAX_OBST_LINES, bool HETERO = false>
__global__ void __launch_bounds__(ORCA_GRID_TPB, (OL <= 2 ? 1024 : 768) / ORCA_GRID_TPB) step_grid_kernel(const StepArgs a, const float4* __restrict__ spv,
                                                           const int* __restrict__ sidx,
                                                           const int* __restrict__ cell_start,
                                                           const GridParams* __restrict__ gpp,
                                                           const int* __restrict__ env_step_snap,
                                                           const float4* __restrict__ agent_params) {
  extern __shared__ float4 smem4[];
  const int tpb = blockDim.x;
  float4* s_lines = smem4;
  float4* s_pool = s_lines + (K + OL) * tpb;
  float2* s_nv = reinterpret_cast<float2*>(s_pool + (ORCA_LP3_SMEM_POOL ? (K + OL) * (tpb / 2) : 0));
  int* s_meta = reinterpret_cast<int*>(s_nv + tpb);
  int* s_warp_cnt = s_meta + tpb;
  unsigned char* s_queue = reinterpret_cast<unsigned char*>(s_warp_cnt + 8);
  float* s_vmax = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(s_queue + tpb) + 15) & ~(uintptr_t)15);
  const int T = a.E * a.N;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = j < T;
  const unsigned warp_mask = __ballot_sync(0xffffffffu, valid);
  AgentCarry c;
  c.p = v2(0.f, 0.f);
  c.v = v2(0.f, 0.f);
  c.nv = v2(0.f, 0.f);
  c.aim = v2(0.f, 0.f);
  c.n = c.n_obst = c.fail = 0;
  int g = 0, env = 0, la = 0, estep = 0;
  bool alive = valid, env_live = true;
  c.overflow = false;
  if (valid) {
    g = sidx[j];
    env = g / a.N;
    la = g - env * a.N;
    estep = (a.env_step != nullptr) ? env_step_snap[env] : 0;
    env_live = env_step_snap[a.E + env] < a.N;
    GridSource src;
    src.spv = spv;
    src.full_range_sq = HETERO ? ORCA_LDG(&agent_params[2 * (size_t)g + 1]).x : a.nd_sq;
    if (HETERO) src.params = agent_params;
    src.orig = sidx;
    src.cell_start = cell_start;
    src.gp = *gpp;
    src.env = env;
    src.env_n0 = env * a.N;
    src.self = j;
    Lines L;
    L.base = s_lines + threadIdx.x;
    L.stride = tpb;
    const float4 pv = spv[j];
    c.p = v2(pv.x, pv.y);
    c.v = v2(pv.z, pv.w);
    if (!a.neighbors_only) c.aim = (POLICY == POLICY_EXTERNAL) ? a.pref[g] : a.goal[g];
    const ObstacleWorld W = global_world_with_cull(a, env);
    alive = agent_front<K, KFULL, POLICY, OL, HETERO>(a, env, g, estep, src, W, L, warp_mask, c, agent_params);
    if (HETERO) s_vmax[threadIdx.x] = ORCA_LDG(&agent_params[2 * (size_t)g]).y;
  }
  if (a.neighbors_only) return;  // uniform over the grid
  block_lp3<K, HETERO>(s_lines, s_pool, s_meta, s_nv, s_queue, s_warp_cnt, alive && !c.overflow && c.fail < c.n, c, a.vmax, false,
                       s_vmax);
  const unsigned slow_mask = __ballot_sync(0xffffffffu, alive && c.overflow);
  if (!alive) return;
  c.nv = s_nv[threadIdx.x];
  if (c.overflow) {  // rare: more obstacle edges / lines than the fast path holds (see agent_slow_path)
    // the neighbor source is rebuilt here from the kernel arguments: nothing of the hot path has to
    // live in local memory for the sake of this call
    Lines L;
    L.base = s_lines + threadIdx.x;
    L.stride = tpb;
    GridSource again;
    again.spv = spv;
    again.orig = sidx;
    again.cell_start = cell_start;
    again.gp = *gpp;
    again.env = env;
    again.env_n0 = env * a.N;
    again.self = j;
    if (HETERO) again.params = agent_params;
    apply_slow_result(agent_slow_path<K, KFULL, GridSource, HETERO>(HETERO ? slow_params(a, agent_params, g) : slow_params(a), again, global_world(a, env), L,
                                                                    K + OL, slow_mask, c.p, c.v, c.pref), c);
  }
  agent_back<POLICY>(a, env, la, g, estep, c, env_live);
}

#define ORCA_GRID_TRY(expr)                                                         \
  do {                                                                              \
    cudaError_t e_ = (expr);                                                        \
    if (e_ != cudaSuccess) {                                                        \
      *err = std::string(#expr) + " failed: " + cudaGetErrorString(e_);             \
      return -2;                                                                    \
    }                                                                               \
  } while (0)

inline int grid_ensure(GridScratch& G, const StepArgs& a, cudaStream_t st, std::string* err) {
  const int T = a.E * a.N;
  if (G.T == T && G.E == a.E && G.sorted_pv != nullptr) return 0;
  grid_free(G);
  int dev = 0;
  ORCA_GRID_TRY(cudaGetDevice(&dev));
  ORCA_GRID_TRY(cudaDeviceGetAttribute(&G.sm_count, cudaDevAttrMultiProcessorCount, dev));
  // size the cell arrays from the current extent of the world (one host sync, first call only)
  ORCA_GRID_TRY(cudaMalloc(&G.counters, 8 * sizeof(int)));
  ORCA_GRID_TRY(cudaMalloc(&G.params, sizeof(GridParams)));
  grid_arm_kernel<<<1, 1, 0, st>>>(G.counters);
  grid_bounds_kernel<<<G.sm_count * 2, kBoundsThreads, 0, st>>>(a.pos, T, G.counters, sqrtf(a.nd_sq), a.E, 1 << 30, G.params);
  GridParams hp;
  ORCA_GRID_TRY(cudaMemcpyAsync(&hp, G.params, sizeof(hp), cudaMemcpyDeviceToHost, st));
  ORCA_GRID_TRY(cudaStreamSynchronize(st));
  // room for the world to spread to ~2x its current side before the cell size has to grow
  double cells = (2.0 * hp.W + 2.0) * (2.0 * hp.H + 2.0) * (double)a.E;
  if (cells < 1024) cells = 1024;
  if (cells > 1.6e7) cells = 1.6e7;
  G.cap_cells = (int)cells;
  G.T = T;
  G.E = a.E;
  G.epoch = 0;
  const size_t tiles = ((size_t)G.cap_cells + kScanTile - 1) / kScanTile;
  ORCA_GRID_TRY(cudaMalloc(&G.sorted_pv, (size_t)T * sizeof(float4)));
  ORCA_GRID_TRY(cudaMalloc(&G.sorted_idx, (size_t)T * sizeof(int)));
  ORCA_GRID_TRY(cudaMalloc(&G.key, (size_t)T * sizeof(int)));
  ORCA_GRID_TRY(cudaMalloc(&G.slot, (size_t)T * sizeof(int)));
  ORCA_GRID_TRY(cudaMalloc(&G.cell_count, ((size_t)G.cap_cells + 1) * sizeof(int)));
  ORCA_GRID_TRY(cudaMalloc(&G.cell_start, ((size_t)G.cap_cells + 1) * sizeof(int)));
  ORCA_GRID_TRY(cudaMalloc(&G.tile_state, tiles * sizeof(unsigned long long)));
  ORCA_GRID_TRY(cudaMalloc(&G.env_step_snap, 2 * (size_t)a.E * sizeof(int)));
  ORCA_GRID_TRY(cudaMemsetAsync(G.cell_count, 0, ((size_t)G.cap_cells + 1) * sizeof(int), st));
  ORCA_GRID_TRY(cudaMemsetAsync(G.tile_state, 0, tiles * sizeof(unsigned long long), st));
  return 0;
}

constexpr int kGridLaunchesPerStep = 5;  // G1 bounds, G2 count, G3 scan, G4 scatter, G5 step

// G1-G4: the cell-sorted snapshot of (a.pos, a.vel) in G.  `bump`: G2 also bumps the env step counters
// (a.env_step, when given).  Any number of runs may follow each other on one stream: the accumulators
// re-arm themselves, the scan re-zeroes the counts it read and tags its tile states with a fresh epoch.
// Runs on the same GridScratch from two streams at once would race; orca_agent_lines has a scratch of
// its own, orca_neighbors uses the step's and is ordered with the steps by the caller's stream.
inline int grid_prep(GridScratch& G, const StepArgs& a, int bump, cudaStream_t st, std::string* err) {
  const int T = a.E * a.N;
  const int rc = grid_ensure(G, a, st, err);
  if (rc != 0) return rc;
  const int tpb = 256;
  const int nb_agents = (T + tpb - 1) / tpb;
  grid_bounds_kernel<<<G.sm_count * 2, kBoundsThreads, 0, st>>>(a.pos, T, G.counters, sqrtf(a.nd_sq), a.E, G.cap_cells, G.params);
  grid_count_kernel<<<nb_agents, tpb, 0, st>>>(a.pos, T, a.N, G.params, G.cell_count, G.key, G.slot, a.env_step,
                                               a.env_done_cnt, G.env_step_snap, a.E, bump);
  const int scan_blocks = (G.cap_cells + kScanTile - 1) / kScanTile;
  G.epoch = (G.epoch + 1u) & 0x3fffffffu;
  if (G.epoch == 0u) G.epoch = 1u;  // 0 is the state of freshly cleared words
  grid_scan_kernel<<<scan_blocks, kScanThreads, 0, st>>>(G.cell_count, G.params, G.tile_state, G.counters + 5, G.epoch,
                                                        G.cell_start);
  grid_scatter_kernel<<<nb_agents, tpb, 0, st>>>(a.pos, a.vel, T, G.key, G.slot, G.cell_start, G.sorted_pv, G.sorted_idx);
  return 0;
}

template <int K, bool KFULL, int POLICY, int OL, bool HETERO = false>
int launch_grid_kpo(GridScratch& G, const StepArgs& a, cudaStream_t st, int64_t* launches, std::string* err,
                    const float4* agent_params = nullptr) {
  const int T = a.E * a.N;
  const int rc = grid_prep(G, a, a.neighbors_only ? 0 : 1, st, err);
  if (rc != 0) return rc;
  StepArgs args = a;
  // the step kernel only READS the step counters in this path, from the copy G2 made
  const int stpb = ORCA_GRID_TPB;
  const size_t smem = step_smem_bytes(K, stpb, false, 0, OL, HETERO);
  auto kern = step_grid_kernel<K, KFULL, POLICY, OL, HETERO>;
  int dev = 0;
  ORCA_GRID_TRY(cudaGetDevice(&dev));
  // function attributes are per device; setting one is idempotent, so a racing second thread is harmless
  static std::atomic<bool> attr_set[kMaxDevices];
  if (dev >= kMaxDevices || !attr_set[dev].load(std::memory_order_acquire)) {
    ORCA_GRID_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ORCA_GRID_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    if (dev < kMaxDevices) attr_set[dev].store(true, std::memory_order_release);
  }
  args.grid_path = 1;
  kern<<<(T + stpb - 1) / stpb, stpb, smem, st>>>(args, G.sorted_pv, G.sorted_idx, G.cell_start, G.params, G.env_step_snap, agent_params);
  ORCA_GRID_TRY(cudaGetLastError());
  *launches += kGridLaunchesPerStep;
  return 0;
}

template <int K, bool KFULL, int POLICY>
int launch_grid_kp(GridScratch& G, const StepArgs& a, cudaStream_t st, int64_t* launches, std::string* err) {
  // at most 4 obstacle vertices (none, or one wall): an agent never has more than 2 obstacle lines
  if (K == 10 && a.world_verts <= 4 && a.vert_stride == 0 && std::getenv("ORCA_B200_NO_SLIM_KERNEL") == nullptr)
    return launch_grid_kpo<10, true, POLICY, 2>(G, a, st, launches, err);
  return launch_grid_kpo<K, KFULL, POLICY, ORCA_MAX_OBST_LINES>(G, a, st, launches, err);
}

template <int K, bool KFULL>
int launch_grid_k(GridScratch& G, const StepArgs& a, int policy, cudaStream_t st, int64_t* launches, std::string* err) {
  switch (policy) {
    case POLICY_EXTERNAL:
      return launch_grid_kp<K, KFULL, POLICY_EXTERNAL>(G, a, st, launches, err);
    case POLICY_GOAL:
      return launch_grid_kp<K, KFULL, POLICY_GOAL>(G, a, st, launches, err);
    case POLICY_RL:
      return launch_grid_kp<K, KFULL, POLICY_RL>(G, a, st, launches, err);
    case POLICY_ALAN:
      return launch_grid_kp<K, KFULL, POLICY_ALAN>(G, a, st, launches, err);
    default:
      *err = "unknown policy";
      return -1;
  }
}

inline int launch_grid_step(GridScratch& G, const StepArgs& a, int policy, cudaStream_t st, int64_t* launches,
                            std::string* err) {
  if (a.k == 5) return launch_grid_k<5, true>(G, a, policy, st, launches, err);
  if (a.k == 10) return launch_grid_k<10, true>(G, a, policy, st, launches, err);
  if (a.k <= 16) return launch_grid_k<16, false>(G, a, policy, st, launches, err);
  *err = "max_neighbors > 16 is not supported";
  return -3;
}

#endif  // __CUDACC__

}  // namespace orca
