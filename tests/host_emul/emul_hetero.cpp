// emul_hetero.cpp -- TEST-ONLY host emulation of the step with per-agent ORCA parameters.
//
// The HETERO instantiation of the library's own per-agent device code (agent_step_body in
// csrc/orca_step_small.cuh with the orca_set_agent_params table), compiled with g++ and run
// serially over a batch, through the tile source (as emul.cpp's run_k, radii staged per env like
// the tile kernel does) and the grid source (as emul.cpp's run_grid_k, radii gathered by original
// id like the grid kernel does).  It lets the CPU suite check the heterogeneous logic against the
// oracle without a GPU; the package never loads it.
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

static inline void sincosf_(float x, float* s, float* c) { *s = sinf(x); *c = cosf(x); }
#define sincosf sincosf_
#include "../../collision_avoidance_b200/csrc/obstacle_world.h"
#include "../../collision_avoidance_b200/csrc/orca_step_small.cuh"
#include "../../collision_avoidance_b200/csrc/orca_grid.cuh"

namespace {
template <int K, class Src>
void body(const orca::StepArgs& a, const float4* table, int policy, int env, int la, int g, float2 p, float2 v, int estep,
          const Src& src, const orca::Lines& L) {
  switch (policy) {
    case 0: orca::agent_step_body<K, false, 0, true>(a, env, la, g, p, v, estep, src, L, 0xffffffffu, table); break;
    case 1: orca::agent_step_body<K, false, 1, true>(a, env, la, g, p, v, estep, src, L, 0xffffffffu, table); break;
    case 2: orca::agent_step_body<K, false, 2, true>(a, env, la, g, p, v, estep, src, L, 0xffffffffu, table); break;
    default: orca::agent_step_body<K, false, 3, true>(a, env, la, g, p, v, estep, src, L, 0xffffffffu, table); break;
  }
}

template <int K>
void run_tile(const orca::StepArgs& a, const float4* table, int policy) {
  const int E = a.E, N = a.N;
  std::vector<float2> spos((size_t)N), svel((size_t)N);
  std::vector<float> srad((size_t)N);
  std::vector<float4> lines((size_t)(K + ORCA_MAX_OBST_LINES));
  for (int e = 0; e < E; ++e) {
    for (int i = 0; i < N; ++i) {
      spos[(size_t)i] = a.pos[(size_t)e * N + i];
      svel[(size_t)i] = a.vel[(size_t)e * N + i];
      srad[(size_t)i] = table[2 * ((size_t)e * N + i)].x;
    }
    const int estep = a.env_step ? a.env_step[e] : 0;
    // host twin of build_tile_grid: ids inside a cell in descending id order (any order is legal)
    std::vector<unsigned short> cell_start(orca::kTileCells + 1, 0);
    std::vector<unsigned char> sorted((size_t)N);
    std::vector<int> cell_of((size_t)N);
    const bool tile_grid = a.tile_grid_inv_cell > 0.f;
    if (tile_grid) {
      float ox = INFINITY, oy = INFINITY;
      for (int i = 0; i < N; ++i) { ox = std::fmin(ox, spos[(size_t)i].x); oy = std::fmin(oy, spos[(size_t)i].y); }
      std::vector<int> cnt(orca::kTileCells, 0);
      for (int i = 0; i < N; ++i) {
        int cx = (int)floorf((spos[(size_t)i].x - ox) * a.tile_grid_inv_cell);
        int cy = (int)floorf((spos[(size_t)i].y - oy) * a.tile_grid_inv_cell);
        cx = cx < 0 ? 0 : (cx >= orca::kTileGrid ? orca::kTileGrid - 1 : cx);
        cy = cy < 0 ? 0 : (cy >= orca::kTileGrid ? orca::kTileGrid - 1 : cy);
        cell_of[(size_t)i] = cy * orca::kTileGrid + cx;
        cnt[cell_of[(size_t)i]]++;
      }
      for (int c = 0; c < orca::kTileCells; ++c) cell_start[c + 1] = (unsigned short)(cell_start[c] + cnt[c]);
      std::vector<int> fill(orca::kTileCells, 0);
      for (int i = N - 1; i >= 0; --i) sorted[cell_start[cell_of[(size_t)i]] + fill[cell_of[(size_t)i]]++] = (unsigned char)i;
    }
    for (int i = 0; i < N; ++i) {
      orca::Lines L;
      L.base = lines.data();
      L.stride = 1;
      const int g = e * N + i;
      orca::TileSource src;
      src.env_pos = spos.data();
      src.env_vel = svel.data();
      src.env_rad = srad.data();
      src.n = N;
      src.self = i;
      src.full_range_sq = table[2 * (size_t)g + 1].x;
      if (tile_grid) {
        src.cell_start = cell_start.data();
        src.sorted = sorted.data();
        src.cx = cell_of[(size_t)i] % orca::kTileGrid;
        src.cy = cell_of[(size_t)i] / orca::kTileGrid;
      }
      body<K>(a, table, policy, e, i, g, spos[(size_t)i], svel[(size_t)i], estep, src, L);
    }
  }
}

template <int K>
void run_grid(const orca::StepArgs& a0, const float4* table, int policy) {
  orca::StepArgs a = a0;
  a.grid_path = 1;
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
  std::vector<float2> spos((size_t)T), svel((size_t)T);
  std::vector<float4> spv((size_t)T);
  for (int j = 0; j < T; ++j) {
    spos[(size_t)j] = a.pos[sidx[(size_t)j]];
    svel[(size_t)j] = a.vel[sidx[(size_t)j]];
    spv[(size_t)j].x = spos[(size_t)j].x; spv[(size_t)j].y = spos[(size_t)j].y;
    spv[(size_t)j].z = svel[(size_t)j].x; spv[(size_t)j].w = svel[(size_t)j].y;
  }
  std::vector<int> estep0((size_t)E, 0);
  if (a.env_step) for (int e = 0; e < E; ++e) estep0[(size_t)e] = a.env_step[e];
  std::vector<float4> lines((size_t)(K + ORCA_MAX_OBST_LINES));
  for (int j = 0; j < T; ++j) {
    const int g = sidx[(size_t)j], env = g / N, la = g - env * N;
    orca::GridSource src;
    src.spv = spv.data(); src.orig = sidx.data(); src.cell_start = start.data(); src.params = table;
    src.full_range_sq = table[2 * (size_t)g + 1].x;
    src.gp = gp; src.env = env; src.env_n0 = env * N; src.self = j;
    orca::Lines L; L.base = lines.data(); L.stride = 1;
    body<K>(a, table, policy, env, la, g, spos[(size_t)j], svel[(size_t)j], estep0[(size_t)env], src, L);
  }
  if (a.env_step && !a.neighbors_only) for (int e = 0; e < E; ++e) a.env_step[e] += 1;
}
}  // namespace

extern "C" {

// a: orca::StepArgs with HOST pointers (nd_sq = the largest neighborDist squared, as launch_step sets
// it); table: the [E*N][2] float4 records of orca_set_agent_params.  K as orca_api.cu's launch_step.
int emul_hetero_step(const orca::StepArgs* a, const float4* table, int policy, int grid) {
  const int k = a->k;
  if (k > 16) return -1;
  if (grid) {
    if (k <= 5) run_grid<5>(*a, table, policy);
    else if (k <= 10) run_grid<10>(*a, table, policy);
    else run_grid<16>(*a, table, policy);
  } else {
    if (k <= 5) run_tile<5>(*a, table, policy);
    else if (k <= 10) run_tile<10>(*a, table, policy);
    else run_tile<16>(*a, table, policy);
  }
  return 0;
}

int emul_hetero_stepargs_size() { return (int)sizeof(orca::StepArgs); }

}  // extern "C"
