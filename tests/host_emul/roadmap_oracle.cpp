// roadmap_oracle.cpp -- TEST-ONLY extension of the CPU oracle (oracle/rvo2_oracle.cpp) with RVO2's
// queryVisibility and the roadmap of RVO2's obstacle example (examples/Roadmap.cpp).
//
// The oracle is compiled into this library unchanged, so the functions below walk the oracle's own
// BSP through its Sim.  They are literal restatements, independent of the library's device code:
//   rvo_query_visibility  KdTree::queryVisibilityRecursive of RVO2 2.0.x, recursively;
//   rvo_roadmap_build     Roadmap.cpp buildRoadmap: the O(R^2) edge loop and one std::multimap
//                         Dijkstra per goal;
//   rvo_roadmap_pref      Roadmap.cpp setPreferredVelocities without the random perturbation, with the
//                         oracle agents' own radii.
// Build: g++ -O2 -ffp-contract=off (every float operation rounds once, as in a stock x86-64 RVO2).
#include "../../oracle/rvo2_oracle.cpp"

#include <map>

namespace {

bool query_visibility_recursive(const Sim& s, V2 q1, V2 q2, float radius, int node) {
  if (node < 0) return true;
  const ObstVertex& o1 = s.verts[s.bsp[node].vertex];
  const ObstVertex& o2 = s.verts[o1.next];
  const float q1_left_of_i = left_of(o1.point, o2.point, q1);
  const float q2_left_of_i = left_of(o1.point, o2.point, q2);
  const float inv_length_i = 1.0f / abs_sq(o2.point - o1.point);
  const int left = s.bsp[node].left, right = s.bsp[node].right;
  if (q1_left_of_i >= 0.0f && q2_left_of_i >= 0.0f) {
    return query_visibility_recursive(s, q1, q2, radius, left) &&
           ((sqr(q1_left_of_i) * inv_length_i >= sqr(radius) && sqr(q2_left_of_i) * inv_length_i >= sqr(radius)) ||
            query_visibility_recursive(s, q1, q2, radius, right));
  } else if (q1_left_of_i <= 0.0f && q2_left_of_i <= 0.0f) {
    return query_visibility_recursive(s, q1, q2, radius, right) &&
           ((sqr(q1_left_of_i) * inv_length_i >= sqr(radius) && sqr(q2_left_of_i) * inv_length_i >= sqr(radius)) ||
            query_visibility_recursive(s, q1, q2, radius, left));
  } else if (q1_left_of_i >= 0.0f && q2_left_of_i <= 0.0f) {
    // one can see through the obstacle from left to right
    return query_visibility_recursive(s, q1, q2, radius, left) && query_visibility_recursive(s, q1, q2, radius, right);
  } else {
    const float point1_left_of_q = left_of(q1, q2, o1.point);
    const float point2_left_of_q = left_of(q1, q2, o2.point);
    const float inv_length_q = 1.0f / abs_sq(q2 - q1);
    return point1_left_of_q * point2_left_of_q >= 0.0f && sqr(point1_left_of_q) * inv_length_q > sqr(radius) &&
           sqr(point2_left_of_q) * inv_length_q > sqr(radius) && query_visibility_recursive(s, q1, q2, radius, left) &&
           query_visibility_recursive(s, q1, q2, radius, right);
  }
}

// RVOSimulator::queryVisibility: the tree exists once processObstacles ran (an empty world has none)
bool query_visibility(const Sim& s, V2 q1, V2 q2, float radius) {
  return query_visibility_recursive(s, q1, q2, radius, s.bsp_root);
}

}  // namespace

extern "C" {

int rvo_query_visibility(void* h, float x1, float y1, float x2, float y2, float radius) {
  return query_visibility(*S(h), V2(x1, y1), V2(x2, y2), radius) ? 1 : 0;
}

// xy [R][2]; the first G vertices are the goals.  adj_out [R][R] bytes (row u, column v: v is in
// roadmap[u].neighbors), dist_out [G][R] = roadmap[v].distToGoal[g].
void rvo_roadmap_build(void* h, const float* xy, int R, int G, float radius, uint8_t* adj_out, float* dist_out) {
  const Sim& s = *S(h);
  std::vector<V2> p(static_cast<size_t>(R));
  for (int i = 0; i < R; ++i) p[i] = V2(xy[2 * i], xy[2 * i + 1]);
  std::vector<std::vector<int>> neighbors(static_cast<size_t>(R));
  std::vector<std::vector<float>> dist_to_goal(static_cast<size_t>(R));
  for (int i = 0; i < R; ++i) {
    for (int j = 0; j < R; ++j) {
      const bool vis = query_visibility(s, p[i], p[j], radius);
      adj_out[static_cast<size_t>(i) * R + j] = vis ? 1 : 0;
      if (vis) neighbors[i].push_back(j);
    }
    dist_to_goal[i].resize(static_cast<size_t>(G), 9e9f);
  }
  for (int i = 0; i < G; ++i) {
    std::multimap<float, int> Q;
    std::vector<std::multimap<float, int>::iterator> pos_in_q(static_cast<size_t>(R), Q.end());
    dist_to_goal[i][i] = 0.0f;
    pos_in_q[i] = Q.insert(std::make_pair(0.0f, i));
    while (!Q.empty()) {
      const int u = Q.begin()->second;
      Q.erase(Q.begin());
      pos_in_q[u] = Q.end();
      for (size_t j = 0; j < neighbors[u].size(); ++j) {
        const int v = neighbors[u][j];
        const float dist_uv = vabs(p[v] - p[u]);
        if (dist_to_goal[v][i] > dist_to_goal[u][i] + dist_uv) {
          dist_to_goal[v][i] = dist_to_goal[u][i] + dist_uv;
          if (pos_in_q[v] == Q.end()) {
            pos_in_q[v] = Q.insert(std::make_pair(dist_to_goal[v][i], v));
          } else {
            Q.erase(pos_in_q[v]);
            pos_in_q[v] = Q.insert(std::make_pair(dist_to_goal[v][i], v));
          }
        }
      }
    }
  }
  for (int g = 0; g < G; ++g)
    for (int v = 0; v < R; ++v) dist_out[static_cast<size_t>(g) * R + v] = dist_to_goal[v][g];
}

// For every agent of the oracle simulator: goals[i] is its goal vertex, dist [G][R] from
// rvo_roadmap_build.  pref_out [n][2], vertex_out [n] (minVertex, -1 when none).
void rvo_roadmap_pref(void* h, const float* xy, int R, int G, const float* dist, const int* goals, float* pref_out,
                      int* vertex_out) {
  Sim& s = *S(h);
  (void)G;
  for (size_t i = 0; i < s.agents.size(); ++i) {
    const V2 pos = s.agents[i].pos;
    const float radius = s.agents[i].radius;
    const float* to_goal = dist + static_cast<size_t>(goals[i]) * R;
    float min_dist = 9e9f;
    int min_vertex = -1;
    for (int j = 0; j < R; ++j) {
      const V2 pj(xy[2 * j], xy[2 * j + 1]);
      if (vabs(pj - pos) + to_goal[j] < min_dist && query_visibility(s, pos, pj, radius)) {
        min_dist = vabs(pj - pos) + to_goal[j];
        min_vertex = j;
      }
    }
    V2 pref(0.f, 0.f);
    if (min_vertex != -1) {
      const V2 pm(xy[2 * min_vertex], xy[2 * min_vertex + 1]);
      if (abs_sq(pm - pos) == 0.0f) {
        if (min_vertex != goals[i]) pref = unit(V2(xy[2 * goals[i]], xy[2 * goals[i] + 1]) - pos);
      } else {
        pref = unit(pm - pos);
      }
    }
    pref_out[2 * i] = pref.x;
    pref_out[2 * i + 1] = pref.y;
    vertex_out[i] = min_vertex;
  }
}

}  // extern "C"
