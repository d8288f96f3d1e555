// orca_core.cuh -- per-agent ORCA arithmetic shared by every kernel of the library.
//
// Computes what one RVO2 agent does inside doStep (reference call sites:
// collision_avoidence_env.py:385,448 and ALAN_true.py:601,632 -> RVO2
// Agent::computeNeighbors / computeNewVelocity / linearProgram1-3, SURVEY.md A.4-A.6):
//   * obstacle-neighbor query over the processed obstacle BSP,
//   * ORCA half-planes for obstacle edges and for agent neighbors,
//   * the incremental 2-D linear programs LP1/LP2/LP3.
//
// Everything is float32 with one rounding per operation: the translation unit is built
// with -fmad=false (no FMA contraction) and IEEE sqrt/div, so on identical inputs the
// results are bit-identical to a scalar x86 evaluation of the same expressions.
//
// The functions are ORCA_HD so tests can also compile them for the host (tests/host_emul)
// to debug logic without a GPU; the shipped library only ever runs them on the device.
#pragma once

#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define ORCA_HD __host__ __device__ __forceinline__
#define ORCA_HD_NOINLINE __host__ __device__ __noinline__
#else
#define ORCA_HD inline
#define ORCA_HD_NOINLINE inline
#include "host_vec_types.h"
#endif
#include <string.h>

#ifndef ORCA_MAX_OBST_NEIGHBORS
#define ORCA_MAX_OBST_NEIGHBORS 16
#endif
#ifndef ORCA_MAX_OBST_LINES
#define ORCA_MAX_OBST_LINES 6
#endif
#ifndef ORCA_MAX_ACTIONS
#define ORCA_MAX_ACTIONS 16
#endif
#define ORCA_MAX_BSP_DEPTH 64
// capacity of the uncapped ("slow") path taken by agents whose obstacle neighborhood exceeds the
// fixed capacities above: obstacle neighbors AND obstacle lines of one agent.  An agent cannot see
// more edges than the processed world has, so worlds of at most this many vertices can never overflow.
#ifndef ORCA_SLOW_MAX_OBST
#define ORCA_SLOW_MAX_OBST 64
#endif

// Branch counters of host test builds (-DORCA_EMUL_COUNT); nothing at all on the device.  Slots of the LPs:
// 0 lp3 rounds, 2 lp1 calls, 3 lp1 inner iterations, 4 projected-line fetches, 5 LP3 rounds (lp3 and
// lp3_stored) whose projected programme was infeasible, 6 projected lines skipped as parallel in the same
// direction, 7 antiparallel midpoints (6 and 7 per fetch: lp3 fetches a line once per access, lp3_stored
// once per round), 8 lp3_stored rounds, 9 obstacle edges skipped as already covered (obstacle_lines).
#if defined(ORCA_EMUL_COUNT) && !defined(__CUDA_ARCH__)
extern long long g_orca_counters[16];
#define ORCA_COUNT(slot, n) (g_orca_counters[slot] += (n))
#else
#define ORCA_COUNT(slot, n) ((void)0)
#endif

// -DORCA_DEBUG_CHECKS: device-side bounds / ownership asserts on every re-used piece of shared memory
// (line slots <-> candidate buffer, LP3 queue <-> in-block grid, dead line columns <-> LP3 programme).
// compute-sanitizer is not available on the GPU pool this was developed on; a build with these checks
// runs the small-shape smoke (tools/sanitize_smoke.py) and the parity tests instead (profiles/README.md).
#if defined(ORCA_DEBUG_CHECKS)
#include <assert.h>
#define ORCA_DCHECK(cond) assert(cond)
#else
#define ORCA_DCHECK(cond) ((void)0)
#endif

namespace orca {

constexpr float kEps = 0.00001f;  // RVO_EPSILON

// bit casts usable from both sides of ORCA_HD
ORCA_HD float bits_to_float(int i) {
#if defined(__CUDA_ARCH__)
  return __int_as_float(i);
#else
  float f;
  memcpy(&f, &i, 4);
  return f;
#endif
}
ORCA_HD int float_to_bits(float f) {
#if defined(__CUDA_ARCH__)
  return __float_as_int(f);
#else
  int i;
  memcpy(&i, &f, 4);
  return i;
#endif
}

// ---- tiny 2-vector algebra (operation order fixed; see header comment) -----------------
ORCA_HD float2 v2(float x, float y) {
  float2 r;
  r.x = x;
  r.y = y;
  return r;
}
ORCA_HD float2 add(float2 a, float2 b) { return v2(a.x + b.x, a.y + b.y); }
ORCA_HD float2 sub(float2 a, float2 b) { return v2(a.x - b.x, a.y - b.y); }
ORCA_HD float2 neg(float2 a) { return v2(-a.x, -a.y); }
ORCA_HD float2 mul(float s, float2 a) { return v2(s * a.x, s * a.y); }
ORCA_HD float dot(float2 a, float2 b) { return a.x * b.x + a.y * b.y; }
ORCA_HD float det(float2 a, float2 b) { return a.x * b.y - a.y * b.x; }
ORCA_HD float abs_sq(float2 a) { return a.x * a.x + a.y * a.y; }
ORCA_HD float sqr(float s) { return s * s; }
// vector / scalar is "multiply by reciprocal" in RVO2 (SURVEY Appendix A helpers)
ORCA_HD float2 div_s(float2 a, float s) {
  const float inv = 1.0f / s;
  return v2(a.x * inv, a.y * inv);
}
ORCA_HD float2 unit(float2 a) { return div_s(a, sqrtf(abs_sq(a))); }
ORCA_HD float left_of(float2 a, float2 b, float2 c) { return det(sub(a, c), sub(b, a)); }
ORCA_HD float fmin_first(float a, float b) { return (b < a) ? b : a; }  // std::min(a, b)
ORCA_HD float fmax_first(float a, float b) { return (a < b) ? b : a; }  // std::max(a, b)

ORCA_HD float dist_sq_point_segment(float2 a, float2 b, float2 c) {
  const float2 ab = sub(b, a);
  const float r = dot(sub(c, a), ab) / abs_sq(ab);
  if (r < 0.f) return abs_sq(sub(c, a));
  if (r > 1.f) return abs_sq(sub(c, b));
  return abs_sq(sub(c, add(a, mul(r, ab))));
}

// ---- line storage: line i of this agent lives at base[i * stride] ------------------------
// (point.x, point.y, dir.x, dir.y).  In the kernels `base` points into shared memory with
// stride = blockDim.x so consecutive lanes hit consecutive 16-byte words (conflict-free).
struct Lines {
  float4* base;
  int stride;
  ORCA_HD float4 get(int i) const { return base[i * stride]; }
  // line-source protocol of the LPs: fetch(j, out) -> false when virtual line j does not exist
  ORCA_HD bool fetch(int i, float4& out) const {
    out = base[i * stride];
    return true;
  }
  ORCA_HD void set(int i, float2 point, float2 dir) const {
    float4 v;
    v.x = point.x;
    v.y = point.y;
    v.z = dir.x;
    v.w = dir.y;
    base[i * stride] = v;
  }
};
ORCA_HD float2 pt(float4 l) { return v2(l.x, l.y); }
ORCA_HD float2 dr(float4 l) { return v2(l.z, l.w); }

#if defined(__CUDA_ARCH__)
#define ORCA_LDG(p) __ldg(p)  // read-only global data
#else
#define ORCA_LDG(p) (*(p))
#endif

// ---- processed obstacle world of one env ---------------------------------------------------
// vert_pd[v]   = (point.x, point.y, unitDir.x, unitDir.y)
// vert_link[v] = (next, prev, isConvex, 0)
// bsp[n]       = (vertex, left child, right child, 0); node 0 is the root; -1 = no child
// bsp_seg[n]   = (p1.x, p1.y, p2.x, p2.y) of the node's edge, so that a visit is two independent
//                16-byte loads instead of a node -> vertex -> next-vertex pointer chase
struct ObstacleWorld {
  const float4* vert_pd;
  const int4* vert_link;
  const int4* bsp;
  const float4* bsp_seg;
  int n_nodes;
  // obstacle-free map (obstacle_world.h: build_cull_map): 32 rows of 32 bits over the box that starts at
  // (geo.x, geo.y) with 1 / cell size (geo.z, geo.w); nullptr: none
  const uint32_t* cull_rows;
  float4 cull_geo;
};

// May an agent at p have an obstacle neighbor at all?  false = provably not (skip the BSP walk).
ORCA_HD bool obstacles_may_be_near(const ObstacleWorld& W, float2 p) {
  if (W.cull_rows == nullptr) return true;
  const float fx = (p.x - W.cull_geo.x) * W.cull_geo.z, fy = (p.y - W.cull_geo.y) * W.cull_geo.w;
  if (!(fx >= 0.f && fx < 32.f && fy >= 0.f && fy < 32.f)) return true;  // outside the mapped box (or NaN): walk
  return ((ORCA_LDG(&W.cull_rows[(int)fy]) >> (int)fx) & 1u) != 0u;
}

// obstacle tables may sit in global OR shared memory (staged by the tile kernel): generic load
#define ORCA_LD(p) (*(p))

// ---- linear programs (SURVEY A.6) -------------------------------------------------------------
// The LPs read their constraints through a "line source" S: S.fetch(j, out) yields virtual line j
// or reports that it does not exist.  `Lines` (the agent's ORCA lines in shared memory) always
// has every line; `ProjectedLines` below is LP3's projected programme, computed on the fly.

// LP1: optimise along line i (= li, already fetched) subject to the speed disc and lines [0, i).
template <class LS>
ORCA_HD bool lp1(const LS& S, int i, float4 li, float radius, float2 opt, bool dir_opt, float2& result) {
  const float2 pi = pt(li), di = dr(li);
  const float dp = dot(pi, di);
  const float disc = sqr(dp) + sqr(radius) - abs_sq(pi);
  if (disc < 0.f) return false;
  const float sq = sqrtf(disc);
  float t_lo = -dp - sq;
  float t_hi = -dp + sq;
  ORCA_COUNT(2, 1);  // lp1 calls
  ORCA_COUNT(3, i);  // lp1 inner iterations (upper bound)
  for (int j = 0; j < i; ++j) {
    float4 lj;
    if (!S.fetch(j, lj)) continue;
    const float den = det(di, dr(lj));
    const float num = det(dr(lj), sub(pi, pt(lj)));
    if (fabsf(den) <= kEps) {
      if (num < 0.f) return false;
      continue;
    }
    const float t = num / den;
    if (den >= 0.f)
      t_hi = fmin_first(t_hi, t);
    else
      t_lo = fmax_first(t_lo, t);
    if (t_lo > t_hi) return false;
  }
  float t;
  if (dir_opt) {
    t = (dot(opt, di) > 0.f) ? t_hi : t_lo;
  } else {
    t = dot(di, sub(opt, pi));
    if (t < t_lo)
      t = t_lo;
    else if (t > t_hi)
      t = t_hi;
  }
  result = add(pi, mul(t, di));
  return true;
}

// Warp-synchronous control flow.  LP2/LP3 are data-dependent nested loops; left to the
// compiler, lanes that fail LP2 at different lines jump straight into LP3 and never meet
// again (measured: 2-5 of 32 lanes active in LP3).  Instead every loop below runs
// "while ANY lane of the warp still has work", so all lanes of `mask` stay in lock step:
// each round is [skip to my next violated line] -> converge -> [LP1 / projection] for the
// lanes that have one.  `mask` = lanes of the warp that execute the step (all of them call
// lp2/lp3, lanes without work pass enabled = false).  On the host the vote is the lane itself.
#if defined(__CUDA_ARCH__)
#define ORCA_ANY(mask, pred) __any_sync((mask), (pred))
#define ORCA_CONVERGE(mask) __syncwarp(mask)
#else
#define ORCA_ANY(mask, pred) (pred)
#define ORCA_CONVERGE(mask) ((void)0)
#endif

// LP2 over the virtual lines [0, n) of S: returns the index of the first line that cannot be
// satisfied (n on success).
template <class LS>
ORCA_HD int lp2(unsigned mask, bool enabled, const LS& S, int n, float radius, float2 opt, bool dir_opt,
                float2& result) {
  if (dir_opt) {
    result = mul(radius, opt);  // opt * radius
  } else if (abs_sq(opt) > sqr(radius)) {
    result = mul(radius, unit(opt));  // normalize(opt) * radius
  } else {
    result = opt;
  }
  int i = 0;
  int fail = n;
  bool active = enabled;
  while (ORCA_ANY(mask, active)) {
    float4 li;
    li.x = li.y = li.z = li.w = 0.f;
    if (active) {
      while (i < n) {
        if (S.fetch(i, li) && det(dr(li), sub(pt(li), result)) > 0.f) break;
        ++i;
      }
      active = i < n;
    }
    ORCA_CONVERGE(mask);
    if (active) {
      const float2 keep = result;
      if (!lp1(S, i, li, radius, opt, dir_opt, result)) {
        result = keep;
        fail = i;
        active = false;
      }
      ++i;
    }
  }
  return fail;
}

// LP3's projected programme for ORCA line i, as a line source computed on the fly: virtual
// line j is obstacle line j as it is (j < n_obst, kept hard), or agent line j (n_obst <= j < i)
// projected onto line i; lines parallel to line i in the same direction do not exist
// (RVO2 `continue`s over them).  Recomputing a projection costs ~45 FP32 instructions from two
// shared-memory lines; storing the programme instead needed a per-thread local-memory array
// whose load/store latency made LP3 41 % of the whole step (DESIGN.md section 5).
template <class LS>
struct ProjectedLines {
  LS L;
  float2 pi, di;  // line i
  int n_obst;
  ORCA_HD bool fetch(int j, float4& out) const {
    ORCA_COUNT(4, 1);  // projected-line fetches
    const float4 lj = L.get(j);
    if (j < n_obst) {
      out = lj;
      return true;
    }
    const float2 pj = pt(lj), dj = dr(lj);
    const float d = det(di, dj);
    float2 np;
    if (fabsf(d) <= kEps) {
      if (dot(di, dj) > 0.f) {
        ORCA_COUNT(6, 1);  // parallel, same direction: no line
        return false;
      }
      ORCA_COUNT(7, 1);  // antiparallel: midpoint
      np = mul(0.5f, add(pi, pj));
    } else {
      np = add(pi, mul(det(dj, sub(pi, pj)) / d, di));
    }
    const float2 nd = unit(sub(dj, di));
    out.x = np.x;
    out.y = np.y;
    out.z = nd.x;
    out.w = nd.y;
    return true;
  }
};

// LP3: minimise the maximum violation of the agent lines [n_obst, n), obstacle lines hard.
// Lanes with need = false only take part in the votes.
template <class LS>
ORCA_HD void lp3(unsigned mask, bool need, const LS& L, int n, int n_obst, int begin, float radius, float2& result) {
  float distance = 0.f;
  int i = begin;
  bool active = need;
  while (ORCA_ANY(mask, active)) {
    ProjectedLines<LS> V;
    V.L = L;
    V.pi = v2(0.f, 0.f);
    V.di = v2(0.f, 0.f);
    V.n_obst = n_obst;
    if (active) {
      while (i < n) {
        const float4 li = L.get(i);
        V.pi = pt(li);
        V.di = dr(li);
        if (det(V.di, sub(V.pi, result)) > distance) break;
        ++i;
      }
      active = i < n;
      if (active) ORCA_COUNT(0, 1);  // lp3 rounds
    }
    ORCA_CONVERGE(mask);
    // the programme: every obstacle line, then the projections of agent lines [n_obst, i)
    const int m = active ? (i > n_obst ? i : n_obst) : 0;
    float2 cand = result;
    const int f = lp2(mask, active, V, m, radius, v2(-V.di.y, V.di.x), true, cand);
    if (active) {
      if (f < m) ORCA_COUNT(5, 1);  // infeasible projected programme
      if (!(f < m)) result = cand;  // on failure keep the previous result
      distance = det(V.di, sub(V.pi, result));
      ++i;
    }
  }
}

// LP3 with the projected programme materialised in scratch storage P (shared memory in
// lp3_queue_kernel, where it is free): the projections are computed once per round instead of
// once per access.  Same arithmetic, same results as lp3().
template <class LS, class PS>
ORCA_HD void lp3_stored(unsigned mask, bool need, const LS& L, int n, int n_obst, int begin, float radius, const PS& P,
                        float2& result) {
  float distance = 0.f;
  int i = begin;
  bool active = need;
  while (ORCA_ANY(mask, active)) {
    float2 pi = v2(0.f, 0.f), di = v2(0.f, 0.f);
    if (active) {
      while (i < n) {
        const float4 li = L.get(i);
        pi = pt(li);
        di = dr(li);
        if (det(di, sub(pi, result)) > distance) break;
        ++i;
      }
      active = i < n;
      if (active) ORCA_COUNT(8, 1);  // lp3_stored rounds
    }
    ORCA_CONVERGE(mask);
    int m = 0;
    if (active) {
      ProjectedLines<LS> V;
      V.L = L;
      V.pi = pi;
      V.di = di;
      V.n_obst = n_obst;
      const int hi = i > n_obst ? i : n_obst;
      for (int j = 0; j < hi; ++j) {
        float4 lj;
        if (V.fetch(j, lj)) P.set(m++, pt(lj), dr(lj));
      }
    }
    ORCA_CONVERGE(mask);
    float2 cand = result;
    const int f = lp2(mask, active, P, m, radius, v2(-di.y, di.x), true, cand);
    if (active) {
      if (f < m) ORCA_COUNT(5, 1);  // infeasible projected programme
      if (!(f < m)) result = cand;  // on failure keep the previous result
      distance = det(di, sub(pi, result));
      ++i;
    }
  }
}

// ---- agent-agent half-plane (SURVEY A.5, second half) -------------------------------------------
// cr = r_i + r_j.  Returns the line; *collided is set when distSq <= cr^2 (RVO2's collision branch).
ORCA_HD float4 agent_line(float2 p, float2 v, float2 po, float2 vo, float cr, float inv_th, float inv_dt,
                          bool* collided) {
  const float2 rp = sub(po, p);
  const float2 rv = sub(v, vo);
  const float d_sq = abs_sq(rp);
  const float cr_sq = sqr(cr);
  const bool apart = d_sq > cr_sq;
  // cut-off circle of horizon tau when apart, of horizon dt when already overlapping
  const float inv_t = apart ? inv_th : inv_dt;
  const float2 w = sub(rv, mul(inv_t, rp));
  const float w_sq = abs_sq(w);
  const float dp1 = dot(w, rp);
  const bool on_circle = !apart || (dp1 < 0.f && sqr(dp1) > cr_sq * w_sq);
  // both shapes need exactly one sqrt and one reciprocal; select their operands
  const float root = sqrtf(on_circle ? w_sq : (d_sq - cr_sq));  // |w|  or  leg
  const float inv = 1.0f / (on_circle ? root : d_sq);
  float2 dir, u;
  if (on_circle) {
    const float2 uw = v2(w.x * inv, w.y * inv);
    dir = v2(uw.y, -uw.x);
    u = mul(cr * inv_t - root, uw);
  } else {
    const float leg = root;
    if (det(rp, w) > 0.f) {
      dir = v2((rp.x * leg - rp.y * cr) * inv, (rp.x * cr + rp.y * leg) * inv);
    } else {
      dir = neg(v2((rp.x * leg + rp.y * cr) * inv, (-rp.x * cr + rp.y * leg) * inv));
    }
    const float dp2 = dot(rv, dir);
    u = sub(mul(dp2, dir), rv);
  }
  *collided = !apart;
  const float2 point = add(v, mul(0.5f, u));
  float4 out;
  out.x = point.x;
  out.y = point.y;
  out.z = dir.x;
  out.w = dir.y;
  return out;
}

// ---- ranks of M keys --------------------------------------------------------------------------------
// r[j] = number of keys that sort in front of key j in (value, index) order: the stable sorting
// permutation by counting.  All M (M - 1) / 2 pair comparisons are independent of each other.
// Device version: one FSET per pair yields 1.0f or 0.0f; its BIT PATTERN (0x3f800000 = 127 * 2^23)
// is accumulated with integer adds, two addends per IADD3, so a pair costs 2 instructions
// instead of compare + select + 2 adds.  The sum wraps mod 2^32, i.e. (count * 127 mod 512) sits
// in bits 23..31; 127 is invertible mod 512 (127 * 383 = 95 * 512 + 1), which recovers any
// count below 512.
// bit pattern of 1.0f when x < y, else 0; and the number of such patterns summed into a word
ORCA_HD unsigned lt_as_one_bits(float x, float y) {
#if defined(__CUDA_ARCH__)
  float one_or_zero;
  asm("set.lt.f32.f32 %0, %1, %2;" : "=f"(one_or_zero) : "f"(x), "f"(y));
  return __float_as_uint(one_or_zero);
#else
  return (x < y) ? 0x3f800000u : 0u;
#endif
}
ORCA_HD int one_bits_count(unsigned sum) { return (int)(((sum >> 23) * 383u) & 511u); }  // counts below 512

template <int M>
ORCA_HD void rank_count(const float* d, int* r) {
#if defined(__CUDA_ARCH__)
  unsigned u[M];
#pragma unroll
  for (int j = 0; j < M; ++j) u[j] = (unsigned)j * 0x3f800000u;
#pragma unroll
  for (int i = 0; i < M; ++i) {
#pragma unroll
    for (int j = i + 1; j < M; ++j) {
      float j_first;  // 1.0f when key j goes in front of key i (equal values: the lower index stays in front)
      asm("set.lt.f32.f32 %0, %1, %2;" : "=f"(j_first) : "f"(d[j]), "f"(d[i]));
      u[i] += __float_as_uint(j_first);
      u[j] -= __float_as_uint(j_first);
    }
  }
#pragma unroll
  for (int j = 0; j < M; ++j) r[j] = (int)(((u[j] >> 23) * 383u) & 511u);
#else
  for (int j = 0; j < M; ++j) r[j] = j;
  for (int i = 0; i < M; ++i) {
    for (int j = i + 1; j < M; ++j) {
      const int j_first = (d[j] < d[i]) ? 1 : 0;
      r[i] += j_first;
      r[j] -= j_first;
    }
  }
#endif
}

// ---- k-nearest list in registers ------------------------------------------------------------------
// Sorted ascending (distSq, id).  Slots >= k hold -1 so they never accept a candidate; slots < k
// start at rangeSq, which makes the strict `<` test do double duty as RVO2's range test and its
// "shrink the range to the k-th best" rule (SURVEY A.4).  Equal distances keep the earlier
// entry in front (first visited wins); callers visit candidates in ascending agent id.
// KFULL = the runtime k equals K, so the acceptance threshold is simply the last slot; every
// index below is a compile-time constant, which keeps both arrays in registers.
template <int K, bool KFULL>
struct NearestK {
  float d[K];
  int id[K];
  int k;           // runtime maxNeighbors (<= K)
  float range_sq;  // neighborDist^2
  uint4 packed;    // the sorted ids as bytes, when a caller handed the list over ready-made
  int packed_cnt;  // number of ids in `packed`; -1: the list lives in id[] only
  ORCA_HD void init(int k_, float range_sq_) {
    k = k_;
    range_sq = range_sq_;
    packed_cnt = -1;
#pragma unroll
    for (int s = 0; s < K; ++s) {
      d[s] = (KFULL || s < k) ? range_sq : -1.0f;
      id[s] = -1;
    }
  }
  // The list handed over ready-made by a caller that ranked its candidates itself: the id of slot
  // s in byte s of `packed` (16 bytes), slots 0..cnt-1 valid.  Distances are not kept.
  ORCA_HD void set_sorted_ids(const uint4 packed_, int cnt) {
    packed = packed_;
    packed_cnt = cnt;
  }
  // id[] from the packed list (only the neighbor-list outputs read id[] on that path)
  ORCA_HD void unpack_ids() {
#pragma unroll
    for (int s = 0; s < K; ++s) {
      const unsigned w = (s < 4) ? packed.x : (s < 8) ? packed.y : (s < 12) ? packed.z : packed.w;
      id[s] = (s < packed_cnt) ? (int)((w >> ((s & 3) * 8)) & 255u) : -1;
      d[s] = 0.f;
    }
  }
  // current acceptance threshold: distance of the k-th slot (slots >= k are -1, distances >= 0,
  // and the list is ascending, so that is the maximum over all slots)
  ORCA_HD float thresh() const {
    if (KFULL) return d[K - 1];
    float m = d[0];
#pragma unroll
    for (int s = 1; s < K; ++s) m = fmaxf(m, d[s]);
    return m;
  }
  // Stable sorted insert.  "the candidate goes in front of slot s" is monotone in s because the
  // list is sorted, so every entry from the first such slot on moves up by one and keeps its
  // relative order (RVO2 shifts while distSq < prev.first).  Every slot is compared with the
  // CANDIDATE (not with a carried element), so the K comparisons are independent of each other.
  // Candidates arrive in ascending id: equal distances keep the earlier entry in front.
  ORCA_HD void offer(float cand_d, int cand_id) {
    if (cand_d < thresh()) {
      bool prev_before = false;  // did the candidate go in front of slot s - 1 ?
      float prev_d = cand_d;     // old content of slot s - 1
      int prev_i = cand_id;
#pragma unroll
      for (int s = 0; s < K; ++s) {
        const bool before = cand_d < d[s];
        const float old_d = d[s];
        const int old_i = id[s];
        d[s] = before ? (prev_before ? prev_d : cand_d) : old_d;
        id[s] = before ? (prev_before ? prev_i : cand_id) : old_i;
        prev_before = before;
        prev_d = old_d;
        prev_i = old_i;
      }
    }
  }
  ORCA_HD void finish() {}
  // the list holds k neighbors / squared distance of the k-th (KFULL lists only)
  ORCA_HD bool full() const { return id[K - 1] >= 0; }
  ORCA_HD float kth_dist_sq() const { return d[K - 1]; }
  // Candidates arrive in arbitrary order (uniform-grid cells): order by (distance, rank) where
  // `precedes(a, b)` says whether entry a goes before entry b at equal distance (b may be -1 = empty
  // slot, which nothing precedes).  Gives the same list as ascending-id visiting.
  template <class Before>
  ORCA_HD void offer_ranked(float cand_d, int cand_id, const Before& precedes) {
    // Bit-equal distances are rare: when no slot holds the candidate's distance the tie rule cannot
    // fire and the plain insertion gives the same list without K conditional rank look-ups.
    bool tie = false;
#pragma unroll
    for (int s = 0; s < K; ++s) tie = tie || (cand_d == d[s]);
    if (!tie) {
      offer(cand_d, cand_id);
      return;
    }
    if (cand_d <= thresh()) {
      bool prev_before = false;
      float prev_d = cand_d;
      int prev_i = cand_id;
#pragma unroll
      for (int s = 0; s < K; ++s) {
        bool before = cand_d < d[s];
        if (cand_d == d[s]) before = precedes(cand_id, id[s]);
        const float old_d = d[s];
        const int old_i = id[s];
        d[s] = before ? (prev_before ? prev_d : cand_d) : old_d;
        id[s] = before ? (prev_before ? prev_i : cand_id) : old_i;
        prev_before = before;
        prev_d = old_d;
        prev_i = old_i;
      }
    }
  }
};

// ---- k-nearest list as 64-bit keys -------------------------------------------------------------------
// Same list as NearestK, held as one integer key per slot: (distSq bits << 32) | (id + 1).
// distSq >= +0, so its float bits order like the values and a single unsigned 64-bit compare IS
// the (distance, id) order -- equal distances rank by id whatever order the candidates arrive
// in (needed when they come cell by cell; for an ascending-id scan it equals RVO2's "first
// visited wins").  Insertion is one pass of compare-exchange: every slot keeps min(slot, carry)
// and hands max(slot, carry) on, the largest key falls off the end -- 6 instructions per slot
// with the tie rule included, against ~11 for the compare + rank-by-id + shift form.
// Empty slot = (rangeSq bits << 32): a candidate at exactly rangeSq (id + 1 >= 1) is not below it,
// which is RVO2's strict range test.  Slots >= k hold 0 and never accept anything.
template <int K, bool KFULL>
struct NearestKeys {
  unsigned long long key[K];
  int id[K];       // valid after finish() / set_sorted_ids()
  float d[K];      // not maintained (distances are recomputed where they are reported)
  int k;
  float range_sq;
  uint4 packed;    // see NearestK
  int packed_cnt;
  ORCA_HD void init(int k_, float range_sq_) {
    k = k_;
    range_sq = range_sq_;
    packed_cnt = -1;
    const unsigned long long empty = (unsigned long long)(unsigned)float_to_bits(range_sq_) << 32;
#pragma unroll
    for (int s = 0; s < K; ++s) {
      key[s] = (KFULL || s < k) ? empty : 0ull;
      id[s] = -1;
      d[s] = 0.f;
    }
  }
  // acceptance threshold: the distance of the k-th slot (the largest key of the list)
  ORCA_HD float thresh() const {
    unsigned long long m = key[K - 1];
    if (!KFULL) {
#pragma unroll
      for (int s = 0; s < K - 1; ++s) m = key[s] > m ? key[s] : m;
    }
    return bits_to_float((int)(unsigned)(m >> 32));
  }
  ORCA_HD void offer(float cand_d, int cand_id) {
    unsigned long long x = ((unsigned long long)(unsigned)float_to_bits(cand_d) << 32) | (unsigned)(cand_id + 1);
    if (KFULL && !(x < key[K - 1])) return;  // not among the k best (any more): nothing moves
#pragma unroll
    for (int s = 0; s < K; ++s) {
      const unsigned long long cur = key[s];
      const bool in_front = x < cur;
      key[s] = in_front ? x : cur;
      x = in_front ? cur : x;
    }
  }
  template <class Before>
  ORCA_HD void offer_ranked(float cand_d, int cand_id, const Before&) {
    offer(cand_d, cand_id);
  }
  ORCA_HD void finish() {
#pragma unroll
    for (int s = 0; s < K; ++s) id[s] = (int)(unsigned)(key[s] & 0xffffffffull) - 1;
  }
  // the list holds k neighbors / squared distance of the k-th (KFULL lists only; after finish())
  ORCA_HD bool full() const { return id[K - 1] >= 0; }
  ORCA_HD float kth_dist_sq() const { return bits_to_float((int)(unsigned)(key[K - 1] >> 32)); }
  // ids below 256 (the tile kernel's in-env ids): also hand the list over as bytes, like
  // set_sorted_ids does, so that its consumers can walk it with a rolled loop.  The valid entries
  // are a prefix of the list (empty slots carry the largest key).
  ORCA_HD void pack_ids() {
    unsigned w[4] = {0u, 0u, 0u, 0u};
    int cnt = 0;
#pragma unroll
    for (int s = 0; s < K; ++s) {
      const bool valid = id[s] >= 0;
      w[s >> 2] |= valid ? ((unsigned)id[s] << ((s & 3) * 8)) : 0u;
      cnt += valid ? 1 : 0;
    }
    packed.x = w[0];
    packed.y = w[1];
    packed.z = w[2];
    packed.w = w[3];
    packed_cnt = cnt;
  }
  ORCA_HD void set_sorted_ids(const uint4 packed_, int cnt) {
    packed = packed_;
    packed_cnt = cnt;
  }
  // id[] from the packed list (only the neighbor-list outputs read id[] on that path)
  ORCA_HD void unpack_ids() {
#pragma unroll
    for (int s = 0; s < K; ++s) {
      const unsigned w = (s < 4) ? packed.x : (s < 8) ? packed.y : (s < 12) ? packed.z : packed.w;
      id[s] = (s < packed_cnt) ? (int)((w >> ((s & 3) * 8)) & 255u) : -1;
    }
  }
};

// ---- candidate buffer: warp-efficient feeding of NearestK -------------------------------------------
// Inserting into the sorted list costs ~6 K instructions and runs for the whole warp whenever ANY
// lane accepts a candidate; with hundreds of candidates of which each lane accepts a few, almost
// every candidate triggers it with 1-4 live lanes (measured: 57 % of all instructions of the
// 256-agent step at 4.3 active lanes).  Instead each lane first parks the candidates that pass its
// (possibly stale) threshold in its own line storage -- not yet in use at this point of the step
// -- and the warp drains all buffers together: round r inserts every lane's r-th parked
// candidate, so the insertion code runs max-count times with most lanes live.  Order per lane is
// preserved and NearestK re-checks the live threshold, so the list is exactly the unbuffered one.
#if defined(__CUDA_ARCH__)
#define ORCA_WARP_MAX(mask, v) __reduce_max_sync((mask), (v))
#else
#define ORCA_WARP_MAX(mask, v) (v)
#endif

struct CandidateBuffer {
  float4* base;  // two entries per 16-byte line slot: entry r in half (r & 1) of base[(r >> 1) * stride]
  int stride;
  int cap;       // entries = 2 x line slots
  int cnt;
  ORCA_HD float2* entry(int r) const { return reinterpret_cast<float2*>(&base[(r >> 1) * stride]) + (r & 1); }
  ORCA_HD void push(float d, int id) {
    ORCA_DCHECK(cnt >= 0 && cnt < cap);
    *entry(cnt) = v2(d, bits_to_float(id));  // (distSq, id bits)
    ++cnt;
  }
  template <class Insert>
  ORCA_HD void drain(unsigned mask, const Insert& insert) {
    const int rounds = ORCA_WARP_MAX(mask, cnt);
    for (int r = 0; r < rounds; ++r) {
      if (r < cnt) {
        const float2 e = *entry(r);
        insert(e.x, float_to_bits(e.y));
      }
    }
    cnt = 0;
  }
  // drain when some lane of the warp is full; call once per candidate by every lane of `mask`
  // `room` = pushes a lane may make before the next call (callers that test several candidates per vote)
  template <class Insert>
  ORCA_HD void drain_if_full(unsigned mask, const Insert& insert, int room = 1) {
    if (ORCA_ANY(mask, cnt + room > cap)) drain(mask, insert);
  }
};

// ---- obstacle neighbors (SURVEY A.3 query + A.4 insertObstacleNeighbor) -----------------------------
// Walks the BSP exactly like the recursive query (near side, node, far side if the splitting line
// is within range) so that equal-distance edges keep RVO2's visiting order.  Result: edge ids
// (first vertex of the edge) ascending by distance in od/oid, count in *cnt.
template <int MAXN = ORCA_MAX_OBST_NEIGHBORS>
ORCA_HD void obstacle_neighbors(const ObstacleWorld& W, float2 p, float range_sq, float* od, int* oid, int* cnt,
                                bool* overflow) {
  int n = 0;
  if (W.n_nodes > 0) {
    // explicit stack of (node << 1 | visited-near-side)
    int stk[ORCA_MAX_BSP_DEPTH];
    int sp = 0;
    stk[sp++] = 0;
    while (sp > 0) {
      const int top = stk[sp - 1];
      const int node = top >> 1;
      const int4 nd = ORCA_LD(&W.bsp[node]);
      const float4 sg = ORCA_LD(&W.bsp_seg[node]);
      const int v1 = nd.x;
      const float2 p1 = v2(sg.x, sg.y), p2 = v2(sg.z, sg.w);
      const float side = left_of(p1, p2, p);
      const int near_c = (side >= 0.f) ? nd.y : nd.z;
      const int far_c = (side >= 0.f) ? nd.z : nd.y;
      if ((top & 1) == 0) {
        stk[sp - 1] = top | 1;
        if (near_c >= 0 && sp < ORCA_MAX_BSP_DEPTH) stk[sp++] = near_c << 1;
        continue;
      }
      --sp;
      const float d_line = sqr(side) / abs_sq(sub(p2, p1));
      if (d_line < range_sq) {
        if (side < 0.f) {
          const float d = dist_sq_point_segment(p1, p2, p);
          if (d < range_sq) {
            if (n < MAXN) {
              int i = n++;
              while (i != 0 && d < od[i - 1]) {
                od[i] = od[i - 1];
                oid[i] = oid[i - 1];
                --i;
              }
              od[i] = d;
              oid[i] = v1;
            } else {
              *overflow = true;
              // keep the nearest MAXN: insert only if closer than the last
              if (d < od[n - 1]) {
                int i = n - 1;
                while (i != 0 && d < od[i - 1]) {
                  od[i] = od[i - 1];
                  oid[i] = oid[i - 1];
                  --i;
                }
                od[i] = d;
                oid[i] = v1;
              }
            }
          }
        }
        if (far_c >= 0 && sp < ORCA_MAX_BSP_DEPTH) stk[sp++] = far_c << 1;
      }
    }
  }
  *cnt = n;
}

// ---- obstacle half-planes (SURVEY A.5, first half) ------------------------------------------------------
// Appends at most MAXL lines to L starting at index 0; returns their number.
template <int MAXL = ORCA_MAX_OBST_LINES, class LS>
ORCA_HD int obstacle_lines(const ObstacleWorld& W, float2 p, float2 vel, float radius, float inv_tho,
                           const float* od, const int* oid, int cnt, const LS& L, bool* overflow) {
  (void)od;
  int nl = 0;
  const float r_sq = sqr(radius);
  for (int q = 0; q < cnt; ++q) {
    int o1 = oid[q];
    float4 a = ORCA_LD(&W.vert_pd[o1]);
    int4 la = ORCA_LD(&W.vert_link[o1]);
    int o2 = la.x;
    float4 b = ORCA_LD(&W.vert_pd[o2]);
    int4 lb = ORCA_LD(&W.vert_link[o2]);
    float2 p1 = v2(a.x, a.y), p2 = v2(b.x, b.y);
    float2 dir1 = v2(a.z, a.w), dir2 = v2(b.z, b.w);
    bool cvx1 = la.z != 0, cvx2 = lb.z != 0;
    const float2 rp1 = sub(p1, p), rp2 = sub(p2, p);

    bool covered = false;
    for (int j = 0; j < nl; ++j) {
      const float4 lj = L.get(j);
      if (det(sub(mul(inv_tho, rp1), pt(lj)), dr(lj)) - inv_tho * radius >= -kEps &&
          det(sub(mul(inv_tho, rp2), pt(lj)), dr(lj)) - inv_tho * radius >= -kEps) {
        covered = true;
        break;
      }
    }
    if (covered) { ORCA_COUNT(9, 1); continue; }  // (host test builds count the edges skipped as covered)

    const float d1 = abs_sq(rp1), d2 = abs_sq(rp2);
    const float2 ov = sub(p2, p1);
    const float s = dot(neg(rp1), ov) / abs_sq(ov);
    const float d_line = abs_sq(sub(neg(rp1), mul(s, ov)));

    float2 out_pt = v2(0.f, 0.f), out_dir = v2(0.f, 0.f);
    bool emit = false;
    bool finished = false;

    if (s < 0.f && d1 <= r_sq) {
      if (cvx1) {
        out_dir = unit(v2(-rp1.y, rp1.x));
        emit = true;
      }
      finished = true;
    } else if (s > 1.f && d2 <= r_sq) {
      if (cvx2 && det(rp2, dir2) >= 0.f) {
        out_dir = unit(v2(-rp2.y, rp2.x));
        emit = true;
      }
      finished = true;
    } else if (s >= 0.f && s < 1.f && d_line <= r_sq) {
      out_dir = neg(dir1);
      emit = true;
      finished = true;
    }

    if (!finished) {
      float2 left_leg, right_leg;
      bool same = false;  // obstacle1 == obstacle2
      bool skip = false;
      if (s < 0.f && d_line <= r_sq) {
        if (!cvx1) {
          skip = true;
        } else {
          // viewed obliquely: both legs come from the left vertex
          o2 = o1;
          p2 = p1;
          dir2 = dir1;
          cvx2 = cvx1;
          same = true;
          const float leg1 = sqrtf(d1 - r_sq);
          left_leg = div_s(v2(rp1.x * leg1 - rp1.y * radius, rp1.x * radius + rp1.y * leg1), d1);
          right_leg = div_s(v2(rp1.x * leg1 + rp1.y * radius, -rp1.x * radius + rp1.y * leg1), d1);
        }
      } else if (s > 1.f && d_line <= r_sq) {
        if (!cvx2) {
          skip = true;
        } else {
          o1 = o2;
          p1 = p2;
          dir1 = dir2;
          cvx1 = cvx2;
          la = lb;
          same = true;
          const float leg2 = sqrtf(d2 - r_sq);
          left_leg = div_s(v2(rp2.x * leg2 - rp2.y * radius, rp2.x * radius + rp2.y * leg2), d2);
          right_leg = div_s(v2(rp2.x * leg2 + rp2.y * radius, -rp2.x * radius + rp2.y * leg2), d2);
        }
      } else {
        if (cvx1) {
          const float leg1 = sqrtf(d1 - r_sq);
          left_leg = div_s(v2(rp1.x * leg1 - rp1.y * radius, rp1.x * radius + rp1.y * leg1), d1);
        } else {
          left_leg = neg(dir1);
        }
        if (cvx2) {
          const float leg2 = sqrtf(d2 - r_sq);
          right_leg = div_s(v2(rp2.x * leg2 + rp2.y * radius, -rp2.x * radius + rp2.y * leg2), d2);
        } else {
          right_leg = dir1;
        }
      }
      if (!skip) {
        // a leg may not point into the neighboring edge of a convex vertex: use that edge's
        // cut-off line instead and remember that the leg is "foreign"
        const int left_nbr = la.y;  // obstacle1->prev
        const float4 ln = ORCA_LD(&W.vert_pd[left_nbr]);
        const float2 ln_dir = v2(ln.z, ln.w);
        bool left_foreign = false, right_foreign = false;
        if (cvx1 && det(left_leg, neg(ln_dir)) >= 0.f) {
          left_leg = neg(ln_dir);
          left_foreign = true;
        }
        if (cvx2 && det(right_leg, dir2) <= 0.f) {
          right_leg = dir2;
          right_foreign = true;
        }
        const float2 lc = mul(inv_tho, sub(p1, p));
        const float2 rc = mul(inv_tho, sub(p2, p));
        const float2 cv = sub(rc, lc);
        const float t = same ? 0.5f : dot(sub(vel, lc), cv) / abs_sq(cv);
        const float t_left = dot(sub(vel, lc), left_leg);
        const float t_right = dot(sub(vel, rc), right_leg);
        if ((t < 0.f && t_left < 0.f) || (same && t_left < 0.f && t_right < 0.f)) {
          const float2 uw = unit(sub(vel, lc));
          out_dir = v2(uw.y, -uw.x);
          out_pt = add(lc, mul(radius * inv_tho, uw));
          emit = true;
        } else if (t > 1.f && t_right < 0.f) {
          const float2 uw = unit(sub(vel, rc));
          out_dir = v2(uw.y, -uw.x);
          out_pt = add(rc, mul(radius * inv_tho, uw));
          emit = true;
        } else {
          const float inf = INFINITY;
          const float dc = (t < 0.f || t > 1.f || same) ? inf : abs_sq(sub(vel, add(lc, mul(t, cv))));
          const float dl = (t_left < 0.f) ? inf : abs_sq(sub(vel, add(lc, mul(t_left, left_leg))));
          const float drr = (t_right < 0.f) ? inf : abs_sq(sub(vel, add(rc, mul(t_right, right_leg))));
          if (dc <= dl && dc <= drr) {
            out_dir = neg(dir1);
            out_pt = add(lc, mul(radius * inv_tho, v2(-out_dir.y, out_dir.x)));
            emit = true;
          } else if (dl <= drr) {
            if (!left_foreign) {
              out_dir = left_leg;
              out_pt = add(lc, mul(radius * inv_tho, v2(-out_dir.y, out_dir.x)));
              emit = true;
            }
          } else {
            if (!right_foreign) {
              out_dir = neg(right_leg);
              out_pt = add(rc, mul(radius * inv_tho, v2(-out_dir.y, out_dir.x)));
              emit = true;
            }
          }
        }
      }
    }
    if (emit) {
      if (nl < MAXL) {
        ORCA_DCHECK(nl >= 0);
        L.set(nl++, out_pt, out_dir);
      } else {
        *overflow = true;
      }
    }
  }
  return nl;
}

// ---- goal-directed preferred velocity ----------------------------------------------------------------
// (cos, sin) of atan2(goal - pos)  ==  unit(goal - pos); atan2(0, 0) = 0 gives (1, 0)
// (collision_avoidence_env.py:156-162, ALAN_true.py:489-495).
ORCA_HD float2 goal_direction(float2 pos, float2 goal) {
  const float2 d = sub(goal, pos);
  const float n2 = abs_sq(d);
  if (n2 > 0.f) {
    const float inv = 1.0f / sqrtf(n2);
    return v2(d.x * inv, d.y * inv);
  }
  return v2(1.f, 0.f);
}
// rotate unit vector `a` by the angle of unit vector `b`: (cos(ta+tb), sin(ta+tb))
ORCA_HD float2 rotate(float2 a, float2 b) { return v2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x); }

// ---- Philox4x32-10 counter RNG (Salmon et al. 2011), one draw per (agent, step) ---------------------
ORCA_HD uint32_t mulhi32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32); }
ORCA_HD float philox_uniform(uint64_t seed, uint32_t c0, uint32_t c1) {
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  uint32_t x0 = c0, x1 = c1, x2 = 0u, x3 = 0u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = mulhi32(0xD2511F53u, x0), lo0 = 0xD2511F53u * x0;
    const uint32_t hi1 = mulhi32(0xCD9E8D57u, x2), lo1 = 0xCD9E8D57u * x2;
    const uint32_t y0 = hi1 ^ x1 ^ k0, y1 = lo1, y2 = hi0 ^ x3 ^ k1, y3 = lo0;
    x0 = y0;
    x1 = y1;
    x2 = y2;
    x3 = y3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  // 24 high bits -> [0, 1)
  return (float)(x0 >> 8) * (1.0f / 16777216.0f);
}

}  // namespace orca
