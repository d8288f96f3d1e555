// emul_roadmap.cpp -- TEST-ONLY host build of the library's roadmap device functions.
//
// query_visibility, the distance relaxation and the preferred-velocity choice of
// csrc/orca_roadmap.cuh, compiled with g++ over obstacle tables built by obstacle_world.h exactly as
// orca_set_obstacles builds them.  The CPU suite compares them with the oracle without a GPU; the
// package never loads this library.  Built with ORCA_EMUL_COUNT: g_orca_counters counts the cases of
// the visibility walk (slots 0-3: the four cases; 4/5 and 6/7: clear / not clear in cases 1 and 2;
// 8/9: case 4's test passed / failed).
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../collision_avoidance_b200/csrc/obstacle_world.h"
#include "../../collision_avoidance_b200/csrc/orca_roadmap.cuh"

long long g_orca_counters[16];

namespace {
struct World {
  std::vector<int4> bsp;
  std::vector<float4> seg;
  int depth = 0;
  orca::ObstacleWorld view() const {
    orca::ObstacleWorld W;
    std::memset(&W, 0, sizeof(W));
    W.bsp = bsp.data();
    W.bsp_seg = seg.data();
    W.n_nodes = static_cast<int>(bsp.size());
    return W;
  }
};
}  // namespace

extern "C" {

// Processed obstacle world of polygons back to back in xy (sizes[p] vertices each); nullptr when its
// BSP is too deep for the library.
void* emul_rm_world_new(const float* xy, const int* sizes, int num_polys) {
  orca_host::ObstacleTables T;
  size_t off = 0;
  for (int p = 0; p < num_polys; ++p) {
    orca_host::add_polygon(T, xy + 2 * off, sizes[p]);
    off += static_cast<size_t>(sizes[p]);
  }
  orca_host::process(T);
  if (T.depth > ORCA_MAX_BSP_DEPTH - 1) return nullptr;
  World* w = new World();
  w->depth = T.depth;
  for (int n = 0; n < T.num_nodes(); ++n) {
    const int e1 = T.node_vertex[n], e2 = T.next[e1];
    w->bsp.push_back(int4{e1, T.node_left[n], T.node_right[n], 0});
    w->seg.push_back(float4{T.px[e1], T.py[e1], T.px[e2], T.py[e2]});
  }
  return w;
}
void emul_rm_world_free(void* w) { delete static_cast<World*>(w); }
int emul_rm_world_depth(void* w) { return static_cast<World*>(w)->depth; }

void emul_rm_counters(long long* out, int reset) {
  std::memcpy(out, g_orca_counters, sizeof(g_orca_counters));
  if (reset) std::memset(g_orca_counters, 0, sizeof(g_orca_counters));
}

// n queries q1[i] -> q2[i] ([n][2]), radius radii[i]; out[i] = 0 / 1.
void emul_rm_visibility(void* w, const float* q1, const float* q2, const float* radii, int n, uint8_t* out) {
  const orca::ObstacleWorld W = static_cast<World*>(w)->view();
  for (int i = 0; i < n; ++i)
    out[i] = orca::query_visibility(W, float2{q1[2 * i], q1[2 * i + 1]}, float2{q2[2 * i], q2[2 * i + 1]},
                                    radii[i])
                 ? 1
                 : 0;
}

// roadmap_dist_kernel for one (table, goal), serially: rounds of in-place relaxation until nothing
// changes.  adj [R][words] as the library stores it; dist_out [R].  Returns the number of rounds.
int emul_rm_dist(const float* xy, const uint32_t* adj, int R, int goal, float* dist_out) {
  const int words = (R + 31) / 32;
  std::vector<float2> p(static_cast<size_t>(R));
  for (int v = 0; v < R; ++v) {
    p[v] = float2{xy[2 * v], xy[2 * v + 1]};
    dist_out[v] = (v == goal) ? 0.0f : orca::kRoadmapInf;
  }
  int rounds = 0;
  for (bool changed = true; changed; ++rounds) {
    changed = false;
    for (int v = 0; v < R; ++v) {
      const float dv = orca::roadmap_relax_vertex(v, R, words, adj, dist_out, p.data());
      if (dv < dist_out[v]) {
        dist_out[v] = dv;
        changed = true;
      }
    }
  }
  return rounds;
}

// roadmap_pref_kernel's body for n agents: dist [G][R], goals[i] (out of [0, G): pref (0, 0), vertex
// -1), radii[i].
void emul_rm_pref(void* w, const float* xy, int R, int G, const float* dist, const float* pos, const int* goals,
                  const float* radii, int n, float* pref_out, int* vertex_out) {
  const orca::ObstacleWorld W = static_cast<World*>(w)->view();
  const float2* p = reinterpret_cast<const float2*>(xy);
  for (int i = 0; i < n; ++i) {
    float2 pref = float2{0.f, 0.f};
    int best = -1;
    const int goal = goals[i];
    if (goal >= 0 && goal < G) {
      const float2 pi = float2{pos[2 * i], pos[2 * i + 1]};
      best = orca::roadmap_choose(W, p, dist + static_cast<size_t>(goal) * R, R, pi, radii[i]);
      pref = orca::roadmap_pref(p, best, goal, pi);
    }
    pref_out[2 * i] = pref.x;
    pref_out[2 * i + 1] = pref.y;
    vertex_out[i] = best;
  }
}

}  // extern "C"
