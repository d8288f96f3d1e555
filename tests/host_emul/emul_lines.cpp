// emul_lines.cpp -- TEST-ONLY host build of the library's ORCA-line query (csrc/orca_lines.cuh).
//
// agent_orca_lines compiled with g++ and run serially over a batch through the tile source (as the
// tile kernel: the env's (pos, vel) staged, a plain scan) and through the grid source (as the grid
// kernel, over a serial counting sort of the cells).  The CPU suite compares it with the oracle's
// lines without a GPU; the package never loads it.  Built with ORCA_EMUL_COUNT: g_orca_counters
// slot 9 counts obstacle edges skipped as already covered, slot 10 collision lines.
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../collision_avoidance_b200/csrc/obstacle_world.h"
#include "../../collision_avoidance_b200/csrc/orca_lines.cuh"

long long g_orca_counters[16];

namespace {
orca::SlowParams params_of(const orca::StepArgs& a, const float4* table, int g) {
  return table != nullptr ? orca::slow_params(a, table, g) : orca::slow_params(a);
}

template <int K>
void run_tile(const orca::StepArgs& a, const float4* table, const orca::LinesOut& o) {
  const int E = a.E, N = a.N;
  std::vector<float2> spos((size_t)N), svel((size_t)N);
  std::vector<float> srad((size_t)N);
  std::vector<float4> scratch((size_t)orca::kLinesScratch);
  for (int e = 0; e < E; ++e) {
    for (int i = 0; i < N; ++i) {
      spos[(size_t)i] = a.pos[(size_t)e * N + i];
      svel[(size_t)i] = a.vel[(size_t)e * N + i];
      srad[(size_t)i] = table != nullptr ? table[2 * ((size_t)e * N + i)].x : 0.f;
    }
    for (int i = 0; i < N; ++i) {
      const int g = e * N + i;
      orca::TileSource src;
      src.env_pos = spos.data();
      src.env_vel = svel.data();
      src.env_rad = srad.data();
      src.n = N;
      src.self = i;
      orca::Lines L;
      L.base = scratch.data();
      L.stride = 1;
      orca::agent_orca_lines<K>(params_of(a, table, g), table != nullptr, src, orca::global_world(a, e), true, L,
                                orca::kLinesScratch, 0xffffffffu, spos[(size_t)i], svel[(size_t)i], o, (size_t)g);
    }
  }
}

template <int K>
void run_grid(const orca::StepArgs& a, const float4* table, const orca::LinesOut& o) {
  const int E = a.E, N = a.N, T = E * N;
  float mnx = INFINITY, mny = INFINITY, mxx = -INFINITY, mxy = -INFINITY;
  for (int i = 0; i < T; ++i) {
    mnx = std::fmin(mnx, a.pos[i].x); mny = std::fmin(mny, a.pos[i].y);
    mxx = std::fmax(mxx, a.pos[i].x); mxy = std::fmax(mxy, a.pos[i].y);
  }
  orca::GridParams gp;
  const float cell = orca::grid_cell_size(std::sqrt(a.nd_sq));  // nd_sq = the largest neighborDist, squared
  gp.origin_x = mnx; gp.origin_y = mny; gp.inv_cell = 1.0f / cell;
  gp.W = (int)(std::floor((mxx - mnx) / cell) + 1.f);
  gp.H = (int)(std::floor((mxy - mny) / cell) + 1.f);
  gp.ncells = E * gp.W * gp.H;
  std::vector<int> key((size_t)T), start((size_t)gp.ncells + 1, 0), sidx((size_t)T);
  for (int i = 0; i < T; ++i) {
    const int cx = orca::GridSource::cell_coord(a.pos[i].x, gp.origin_x, gp.inv_cell, gp.W);
    const int cy = orca::GridSource::cell_coord(a.pos[i].y, gp.origin_y, gp.inv_cell, gp.H);
    key[(size_t)i] = (i / N) * gp.W * gp.H + cy * gp.W + cx;
    start[(size_t)key[(size_t)i] + 1]++;
  }
  for (int c = 0; c < gp.ncells; ++c) start[(size_t)c + 1] += start[(size_t)c];
  std::vector<int> fill(start.begin(), start.end() - 1);
  for (int i = T - 1; i >= 0; --i) sidx[(size_t)fill[(size_t)key[(size_t)i]]++] = i;  // reversed order on purpose
  std::vector<float4> spv((size_t)T);
  for (int j = 0; j < T; ++j) {
    const float2 p = a.pos[sidx[(size_t)j]], v = a.vel[sidx[(size_t)j]];
    spv[(size_t)j].x = p.x; spv[(size_t)j].y = p.y; spv[(size_t)j].z = v.x; spv[(size_t)j].w = v.y;
  }
  std::vector<float4> scratch((size_t)(K + ORCA_MAX_OBST_LINES));
  for (int j = 0; j < T; ++j) {
    const int g = sidx[(size_t)j], env = g / N;
    const orca::SlowParams q = params_of(a, table, g);
    orca::GridSource src;
    src.spv = spv.data(); src.orig = sidx.data(); src.cell_start = start.data(); src.params = table;
    src.full_range_sq = q.nd_sq;
    src.gp = gp; src.env = env; src.env_n0 = env * N; src.self = j;
    orca::Lines L; L.base = scratch.data(); L.stride = 1;
    const orca::ObstacleWorld W = orca::global_world_with_cull(a, env);
    const float2 p = orca::v2(spv[(size_t)j].x, spv[(size_t)j].y), v = orca::v2(spv[(size_t)j].z, spv[(size_t)j].w);
    orca::agent_orca_lines<K>(q, table != nullptr, src, W, orca::obstacles_may_be_near(W, p), L, K + ORCA_MAX_OBST_LINES,
                              0xffffffffu, p, v, o, (size_t)g);
  }
}
}  // namespace

extern "C" {

// a: orca::StepArgs with HOST pointers (pos, vel, world; nd_sq = the largest neighborDist squared when a
// table is given, as orca_agent_lines sets it); table: orca_set_agent_params' [E*N][2] records or NULL.
// lines [E*N][max_lines][4], cnt [E*N], obst_cnt [E*N] or NULL.  K as orca_agent_lines picks it.
int emul_agent_lines(const orca::StepArgs* a, const float4* table, int grid, int max_lines, float* lines, int* cnt,
                     int* obst_cnt) {
  orca::LinesOut o;
  o.lines = reinterpret_cast<float4*>(lines);
  o.cnt = cnt;
  o.obst_cnt = obst_cnt;
  o.max_lines = max_lines;
  const int k = a->k;
  if (k > 16) return -1;
  if (grid) {
    if (k <= 5) run_grid<5>(*a, table, o);
    else if (k <= 10) run_grid<10>(*a, table, o);
    else run_grid<16>(*a, table, o);
  } else {
    if (k <= 5) run_tile<5>(*a, table, o);
    else if (k <= 10) run_tile<10>(*a, table, o);
    else run_tile<16>(*a, table, o);
  }
  return 0;
}

void emul_lines_counters(long long* out, int reset) {
  std::memcpy(out, g_orca_counters, sizeof(g_orca_counters));
  if (reset) std::memset(g_orca_counters, 0, sizeof(g_orca_counters));
}

int emul_lines_stepargs_size() { return (int)sizeof(orca::StepArgs); }

}  // extern "C"
