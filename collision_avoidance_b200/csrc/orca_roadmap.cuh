// orca_roadmap.cuh -- line-of-sight queries on the obstacle BSP and roadmap navigation.
//
// RVO2's RVOSimulator::queryVisibility(point1, point2, radius) and the roadmap of its obstacle example
// (examples/Roadmap.cpp: buildRoadmap, setPreferredVelocities without the random perturbation), over
// the processed obstacle tables the step kernels already read (ObstacleWorld, orca_core.cuh).
//
// Visibility restates RVO2 2.0.x KdTree::queryVisibilityRecursive.  For the node edge p1 -> p2:
//
//   a = leftOf(p1, p2, q1); b = leftOf(p1, p2, q2); invLenI = 1 / absSq(p2 - p1)
//   clear = sqr(a) * invLenI >= sqr(r) && sqr(b) * invLenI >= sqr(r)
//   a >= 0 && b >= 0 : vis(left)  && (clear || vis(right))
//   a <= 0 && b <= 0 : vis(right) && (clear || vis(left))
//   a >= 0 && b <= 0 : vis(left)  && vis(right)        (one can see through the edge from left to right)
//   otherwise        : c = leftOf(q1, q2, p1); d = leftOf(q1, q2, p2); invLenQ = 1 / absSq(q2 - q1)
//                      c * d >= 0 && sqr(c) * invLenQ > sqr(r) && sqr(d) * invLenQ > sqr(r)
//                      && vis(left) && vis(right)
//   vis(no node) = true
//
// The answer is the AND of one local predicate per visited node, and which children a node visits
// depends only on that node's own case.  So the walk below uses an explicit stack in any order and
// stops at the first node whose predicate is false.  The float32 expressions are the recursion's
// (reciprocal then multiply, >= versus >, no contraction: the library is built with -fmad=false), so
// the answer is RVO2's bit for bit, degenerate queries included (q1 == q2 makes invLenQ infinite and
// the products NaN or infinite, and NaN compares false exactly as on the host).
//
// The functions are ORCA_HD like those of orca_core.cuh: tests compile them for the host.
#pragma once

#include "orca_core.cuh"

namespace orca {

constexpr float kRoadmapInf = 9e9f;        // Roadmap.cpp's "no path" distance
constexpr int kRoadmapMaxVertices = 512;   // the distance relaxation keeps a world's roadmap in shared memory

ORCA_HD bool query_visibility(const ObstacleWorld& W, float2 q1, float2 q2, float radius) {
  if (W.n_nodes <= 0) return true;
  const float r_sq = sqr(radius);
  // a node at depth L leaves at most one pending sibling per level above it: the stack never holds
  // more than the BSP's depth, which orca_set_obstacles keeps below ORCA_MAX_BSP_DEPTH
  int stk[ORCA_MAX_BSP_DEPTH];
  int sp = 0;
  stk[sp++] = 0;
  while (sp > 0) {
    const int node = stk[--sp];
    const int4 nd = ORCA_LD(&W.bsp[node]);
    const float4 sg = ORCA_LD(&W.bsp_seg[node]);
    const float2 p1 = v2(sg.x, sg.y), p2 = v2(sg.z, sg.w);
    const float a = left_of(p1, p2, q1);
    const float b = left_of(p1, p2, q2);
    const float inv_len_i = 1.0f / abs_sq(sub(p2, p1));
    bool go_left = true, go_right = true;
    if (a >= 0.f && b >= 0.f) {
      const bool clear = sqr(a) * inv_len_i >= r_sq && sqr(b) * inv_len_i >= r_sq;
      ORCA_COUNT(0, 1);
      ORCA_COUNT(clear ? 4 : 5, 1);
      go_right = !clear;
    } else if (a <= 0.f && b <= 0.f) {
      const bool clear = sqr(a) * inv_len_i >= r_sq && sqr(b) * inv_len_i >= r_sq;
      ORCA_COUNT(1, 1);
      ORCA_COUNT(clear ? 6 : 7, 1);
      go_left = !clear;
    } else if (a >= 0.f && b <= 0.f) {
      ORCA_COUNT(2, 1);
    } else {
      const float c = left_of(q1, q2, p1);
      const float d = left_of(q1, q2, p2);
      const float inv_len_q = 1.0f / abs_sq(sub(q2, q1));
      const bool pass = c * d >= 0.f && sqr(c) * inv_len_q > r_sq && sqr(d) * inv_len_q > r_sq;
      ORCA_COUNT(3, 1);
      ORCA_COUNT(pass ? 8 : 9, 1);
      if (!pass) return false;
    }
    if (go_left && nd.y >= 0 && sp < ORCA_MAX_BSP_DEPTH) stk[sp++] = nd.y;
    if (go_right && nd.z >= 0 && sp < ORCA_MAX_BSP_DEPTH) stk[sp++] = nd.z;
  }
  return true;
}

// Roadmap.cpp's edge weight: RVO::abs(p_v - p_u).
ORCA_HD float roadmap_edge_length(float2 pu, float2 pv) { return sqrtf(abs_sq(sub(pv, pu))); }

// One relaxation of vertex v's distance to a goal: the smallest of d[v] and d[u] + |p_v - p_u| over the
// edges u -> v (adj row u, bit v; `words` 32-bit words per row).  d and xy may be read while other
// vertices are being relaxed: any value read is the length of some path, which is all the fixed point
// argument below needs.
ORCA_HD float roadmap_relax_vertex(int v, int R, int words, const uint32_t* adj, const float* d, const float2* xy) {
  float dv = d[v];
  const float2 pv = xy[v];
  const uint32_t bit = 1u << (v & 31);
  const int wv = v >> 5;
  for (int u = 0; u < R; ++u) {
    if ((adj[u * words + wv] & bit) == 0u) continue;
    const float cand = d[u] + roadmap_edge_length(xy[u], pv);
    if (cand < dv) dv = cand;
  }
  return dv;
}

// Roadmap.cpp setPreferredVelocities' choice of vertex, without the perturbation: the lowest index among
// the vertices of smallest cost |p_j - pos| + dist[j] that have cost < 9e9f and are visible from pos for
// a disc of `radius`; -1 when there is none.  `dist` is the goal's row of distances.  Roadmap.cpp's loop:
// the BSP is walked for every vertex that would lower the running minimum, in index order.  (Testing
// candidates in (cost, index) order instead, stopping at the first visible one, halves the walks but
// costs 3.4 times as much: DESIGN.md section 5.)
ORCA_HD int roadmap_choose(const ObstacleWorld& W, const float2* xy, const float* dist, int R, float2 pos, float radius) {
  float min_cost = kRoadmapInf;
  int best = -1;
  for (int j = 0; j < R; ++j) {
    const float2 pj = xy[j];
    const float cost = sqrtf(abs_sq(sub(pj, pos))) + dist[j];
    if (cost < min_cost && query_visibility(W, pos, pj, radius)) {
      min_cost = cost;
      best = j;
    }
  }
  return best;
}

// The preferred velocity Roadmap.cpp sets for the chosen vertex `best` (RVO::normalize(v) = v / abs(v),
// a multiplication by the reciprocal).
ORCA_HD float2 roadmap_pref(const float2* xy, int best, int goal, float2 pos) {
  if (best < 0) return v2(0.f, 0.f);
  const float2 to_best = sub(xy[best], pos);
  if (abs_sq(to_best) == 0.f) return best == goal ? v2(0.f, 0.f) : unit(sub(xy[goal], pos));
  return unit(to_best);
}

// Obstacle worlds as the step kernels address them: env e reads its own tables at e * vert_stride when
// env_nodes is set, the shared world otherwise.
struct BspTables {
  const int4* bsp;
  const float4* bsp_seg;
  const int* env_nodes;  // per-env node counts, or nullptr when the world is shared
  int shared_nodes;
  int vert_stride;       // 0 when shared

  ORCA_HD ObstacleWorld world(int env) const {
    ObstacleWorld W;
    const size_t voff = (env_nodes != nullptr) ? (size_t)env * vert_stride : 0;
    W.vert_pd = nullptr;
    W.vert_link = nullptr;
    W.bsp = bsp + voff;
    W.bsp_seg = bsp_seg + voff;
    W.n_nodes = (env_nodes != nullptr) ? env_nodes[env] : shared_nodes;
    W.cull_rows = nullptr;
    return W;
  }
};

#if defined(__CUDACC__)

// One thread per query of [E][Q]: env e's own world, or the shared one.
__global__ void visibility_kernel(BspTables T, int E, int Q, const float2* __restrict__ q1, const float2* __restrict__ q2,
                                  const float* __restrict__ radius_q, float radius, uint8_t* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)E * Q) return;
  const int e = (int)(i / Q);
  const float r = radius_q != nullptr ? radius_q[i] : radius;
  out[i] = query_visibility(T.world(e), q1[i], q2[i], r) ? 1 : 0;
}

// Roadmap tables of one handle: W table sets (one per obstacle world, per env when either the obstacles
// or the roadmap are per env), each with R vertices of which the first G are goals.
struct RoadmapArgs {
  BspTables bsp;
  int W, R, G, words;     // words = ceil(R / 32) per adjacency row
  int xy_per_table;       // 1: table t reads vertices xy + t * R; 0: all read the shared vertices
  int obst_per_table;     // 1: table t uses obstacle world t; 0: the shared world
  float radius;           // the disc of the edge queries (Roadmap.cpp: the agents' radius)
  const float2* xy;       // [W or 1][R]
  uint32_t* adj;          // [W][R][words]: row u bit v = queryVisibility(p_u, p_v, radius)
  float* dist;            // [W][G][R]
};

// All ordered pairs (u, v) of every table; one warp per adjacency word.
__global__ void roadmap_edges_kernel(RoadmapArgs a) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long row_threads = (long long)a.words * 32;
  if (t >= (long long)a.W * a.R * row_threads) return;  // whole warps: row_threads is a multiple of 32
  const int col = (int)(t % row_threads);
  const int u = (int)((t / row_threads) % a.R);
  const int w = (int)(t / (row_threads * a.R));
  const float2* xy = a.xy + (a.xy_per_table ? (size_t)w * a.R : 0);
  bool vis = false;
  if (col < a.R) vis = query_visibility(a.bsp.world(a.obst_per_table ? w : 0), xy[u], xy[col], a.radius);
  const unsigned bits = __ballot_sync(0xffffffffu, vis);
  if ((threadIdx.x & 31) == 0) a.adj[((size_t)w * a.R + u) * a.words + col / 32] = bits;
}

// One block per (table, goal): distances to the goal by min-plus relaxation in shared memory, repeated
// until a round changes nothing.
//
// Why this is Dijkstra's result bit for bit: every value the relaxation stores is fl(d[u] + w) for a
// value d[u] it stored before, so each d[v] is the left-to-right rounded length of some path from the
// goal, and at the fixed point d[v] <= fl(d[u] + w) for every edge u -> v.  Rounded addition of a weight
// w >= 0 is monotone in its first operand and never below it, so by induction along any path the fixed
// point is at most that path's rounded length: d[v] is the minimum over paths of the rounded lengths.
// Dijkstra (Roadmap.cpp's multimap queue) computes that same minimum: the same monotonicity is all its
// correctness proof needs, and both start from d[goal] = 0 and 9e9f elsewhere.
__global__ void roadmap_dist_kernel(RoadmapArgs a) {
  extern __shared__ float2 rm_smem[];
  float2* xy = rm_smem;                                                      // [R] (first: 8-byte aligned)
  uint32_t* adj = reinterpret_cast<uint32_t*>(xy + a.R);                     // [R][words]
  float* d = reinterpret_cast<float*>(adj + (size_t)a.R * a.words);          // [R]
  __shared__ int changed;
  const int w = blockIdx.x / a.G, g = blockIdx.x % a.G;
  const float2* gxy = a.xy + (a.xy_per_table ? (size_t)w * a.R : 0);
  const uint32_t* gadj = a.adj + (size_t)w * a.R * a.words;
  for (int i = threadIdx.x; i < a.R * a.words; i += blockDim.x) adj[i] = gadj[i];
  for (int v = threadIdx.x; v < a.R; v += blockDim.x) {
    xy[v] = gxy[v];
    d[v] = (v == g) ? 0.0f : kRoadmapInf;
  }
  for (;;) {
    if (threadIdx.x == 0) changed = 0;
    __syncthreads();
    bool mine = false;
    for (int v = threadIdx.x; v < a.R; v += blockDim.x) {
      const float dv = roadmap_relax_vertex(v, a.R, a.words, adj, d, xy);
      if (dv < d[v]) {
        d[v] = dv;
        mine = true;
      }
    }
    if (mine) changed = 1;
    __syncthreads();
    const int again = changed;
    __syncthreads();  // everyone has read `changed` before thread 0 clears it
    if (!again) break;
  }
  float* out = a.dist + ((size_t)w * a.G + g) * a.R;
  for (int v = threadIdx.x; v < a.R; v += blockDim.x) out[v] = d[v];
}

// One thread per agent: Roadmap.cpp's preferred velocity toward the goal vertex goal_vertex[i].
__global__ void roadmap_pref_kernel(RoadmapArgs a, int E, int N, const float2* __restrict__ pos,
                                    const int32_t* __restrict__ goal_vertex, const float4* __restrict__ agent_params,
                                    float radius, float2* __restrict__ pref, int32_t* __restrict__ vertex_out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)E * N) return;
  const int e = (int)(i / N);
  const int goal = goal_vertex[i];
  float2 p = v2(0.f, 0.f);
  int best = -1;
  if (goal >= 0 && goal < a.G) {
    const int w = a.W > 1 ? e : 0;
    const float2* xy = a.xy + (a.xy_per_table ? (size_t)w * a.R : 0);
    const float* dist = a.dist + ((size_t)w * a.G + goal) * a.R;
    const float r = agent_params != nullptr ? agent_params[2 * i].x : radius;
    const float2 pi = pos[i];
    best = roadmap_choose(a.bsp.world(a.obst_per_table ? e : 0), xy, dist, a.R, pi, r);
    p = roadmap_pref(xy, best, goal, pi);
  }
  pref[i] = p;
  if (vertex_out != nullptr) vertex_out[i] = best;
}

#endif  // __CUDACC__

}  // namespace orca
