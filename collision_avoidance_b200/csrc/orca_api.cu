// orca_api.cu -- C ABI (include/orca_b200.h) over the sm_100a kernels.
//
// Build (see collision_avoidance_b200/build.py):
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -fmad=false \
//        -Xcompiler -fPIC,-ffp-contract=off -shared -o liborca_b200.so orca_api.cu
// -fmad=false is part of the contract: see orca_core.cuh.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/orca_b200.h"
#include "obstacle_world.h"
#include "orca_core.cuh"
#include "orca_grid.cuh"
#include "orca_lines.cuh"
#include "orca_obs.cuh"
#include "orca_policy.cuh"
#include "orca_policy_tc.cuh"
#include "orca_roadmap.cuh"
#include "orca_step_small.cuh"

namespace {

thread_local std::string g_last_error;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

#define CUDA_TRY(expr)                                                                          \
  do {                                                                                          \
    cudaError_t e_ = (expr);                                                                    \
    if (e_ != cudaSuccess) return fail(ORCA_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e_)); \
  } while (0)

// Switches to the handle's device for the duration of a call and restores the caller's device
// afterwards (the caller -- torch -- must not find its current device changed).
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  explicit DeviceGuard(int device) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != device) switched = (cudaSetDevice(device) == cudaSuccess);
  }
  ~DeviceGuard() {
    if (switched) cudaSetDevice(prev);
  }
};

}  // namespace

// orca_step_host pipelining: at most this many env chunks; batches below kHostChunkAgents are not cut
constexpr int kHostChunksMax = 16;
constexpr long long kHostChunkAgents = 65536;

// what a captured orca_step_host graph depends on
struct HostGraphKey {
  const void* pos;
  const void* vel;
  const void* aux;
  int policy, flags, steps, chunks;
  bool operator==(const HostGraphKey& o) const {
    return pos == o.pos && vel == o.vel && aux == o.aux && policy == o.policy && flags == o.flags &&
           steps == o.steps && chunks == o.chunks;
  }
};

struct OrcaSim {
  OrcaParams p{};
  int device = 0;
  int E = 0, N = 0;
  int grid_min_agents = 257;  // worlds with at least this many agents use the uniform-grid pipeline
  // obstacle world(s)
  std::vector<orca_host::ObstacleTables> worlds;  // 1 (shared) or E
  bool per_env = false;
  float4* d_vert_pd = nullptr;
  int4* d_vert_link = nullptr;
  int4* d_bsp = nullptr;
  float4* d_bsp_seg = nullptr;
  int* d_env_nodes = nullptr;
  uint32_t* d_cull_rows = nullptr;  // obstacle-free maps (obstacle_world.h: build_cull_map), 32 words per world
  float4* d_cull_geo = nullptr;
  int shared_nodes = 0;
  int vert_stride = 0;
  // staging for the *_host entry points
  float2* d_pos = nullptr;
  float2* d_vel = nullptr;
  float2* d_aux = nullptr;
  bool host_state_valid = false;  // d_pos / d_vel hold a state uploaded by an orca_step_host(upload_state = 1) call
  const void* host_aux_src = nullptr;  // host buffer whose content d_aux currently mirrors (ORCA_HOST_AUX_UNCHANGED)
  cudaStream_t host_streams[kHostChunksMax] = {};
  cudaEvent_t host_fork = nullptr;
  cudaEvent_t host_join[kHostChunksMax] = {};
  HostGraphKey host_graph_key{};
  cudaGraphExec_t host_graph_exec = nullptr;  // the captured upload | step | download fan-out
  int64_t host_graph_launches = 0;             // kernel launches one replay performs
  // route choice of steady-state orca_step_host calls (see there)
  HostGraphKey tune_key{};
  int tune_calls = 0;
  double tune_ms[2] = {0.0, 0.0};  // [direct, staged]
  float* d_nbr_hint = nullptr;  // [E*N] per-agent starting threshold of the neighbor search (see agent_front)
  // per-agent parameters (orca_set_agent_params): [E*N][2] records (orca::AgentParams, packed), or
  // nullptr (uniform), and the largest neighbor distance and obstacle range (tho * vmax + r) among them
  float4* d_agent_params = nullptr;
  float max_nd = 0.f, max_orange = 0.f;
  float cull_range = 0.f;  // obstacle range the obstacle-free maps were built for
  // roadmap (orca_set_roadmap): the caller's vertices are kept on the host so that orca_set_obstacles
  // can rebuild the edges and distances; rm_R == 0 means no roadmap
  std::vector<float> rm_host_xy;  // [1 or E][R][2]
  int rm_R = 0, rm_G = 0;
  bool rm_per_env = false;
  float rm_radius = 0.f;
  int rm_tables = 0;                // table sets on the device: E when the obstacles or the roadmap are per env, else 1
  float2* d_rm_xy = nullptr;
  uint32_t* d_rm_adj = nullptr;
  float* d_rm_dist = nullptr;
  // uniform-grid scratch (large worlds)
  orca::GridScratch grid;
  // ... of orca_agent_lines: a set of its own, so that the query never writes what a step reads
  orca::GridScratch lines_grid;
  int64_t launches = 0;
};

namespace {

void free_obstacles(OrcaSim* s) {
  if (s->host_graph_exec) {  // the captured host step has the old tables baked into its kernel arguments
    cudaGraphExecDestroy(s->host_graph_exec);
    s->host_graph_exec = nullptr;
  }
  cudaFree(s->d_vert_pd);
  cudaFree(s->d_vert_link);
  cudaFree(s->d_bsp);
  cudaFree(s->d_bsp_seg);
  cudaFree(s->d_env_nodes);
  cudaFree(s->d_cull_rows);
  cudaFree(s->d_cull_geo);
  s->d_cull_rows = nullptr;
  s->d_cull_geo = nullptr;
  s->d_vert_pd = nullptr;
  s->d_vert_link = nullptr;
  s->d_bsp = nullptr;
  s->d_bsp_seg = nullptr;
  s->d_env_nodes = nullptr;
  s->shared_nodes = 0;
  s->vert_stride = 0;
  s->worlds.clear();
}

int pick_k(int k) {
  if (k <= 5) return 5;
  if (k <= 10) return 10;
  if (k <= 16) return 16;
  return -1;
}

void fill_common(const OrcaSim* s, orca::StepArgs* a) {
  std::memset(a, 0, sizeof(*a));
  a->E = s->E;
  a->N = s->N;
  a->k = s->p.max_neighbors;
  a->dt = s->p.time_step;
  a->inv_dt = 1.0f / s->p.time_step;
  a->nd_sq = s->p.neighbor_dist * s->p.neighbor_dist;
  a->inv_th = 1.0f / s->p.time_horizon;
  a->inv_tho = 1.0f / s->p.time_horizon_obst;
  a->radius = s->p.radius;
  a->vmax = s->p.max_speed;
  const float orange = s->p.time_horizon_obst * s->p.max_speed + s->p.radius;
  a->obst_range_sq = orange * orange;
  a->vert_pd = s->d_vert_pd;
  a->vert_link = s->d_vert_link;
  a->bsp = s->d_bsp;
  a->bsp_seg = s->d_bsp_seg;
  a->env_nodes = s->per_env ? s->d_env_nodes : nullptr;
  a->shared_nodes = s->shared_nodes;
  a->vert_stride = s->per_env ? s->vert_stride : 0;
  a->world_verts = s->vert_stride;
  a->world_slots = 0;
  a->cull_rows = s->d_cull_rows;
  a->cull_geo = s->d_cull_geo;
}

template <int K, bool KFULL, int POLICY, int OL, bool HETERO = false>
int launch_small_kpo(OrcaSim* s, const orca::StepArgs& a, cudaStream_t st) {
  const int N = s->N;
  // 256-thread blocks: whole envs per block (256 / N of them); measured faster than 128 / 64 / 32
  // because the block-level LP3 queue gets denser (DESIGN.md section 5)
  int tpb = 256;
  if (const char* e = std::getenv("ORCA_B200_TPB")) {  // dev knob: block size of the tile kernel
    const int v = std::atoi(e);
    if (v >= N && v <= 256 && v % 32 == 0) tpb = v;
  }
  orca::StepArgs args = a;
  args.envs_per_block = tpb / N;
  const int blocks = (a.E - a.env_base + args.envs_per_block - 1) / args.envs_per_block;
  // obstacle tables staged in shared memory when they are small (<= 256 vertex slots = 16 KB)
  const int slots = s->per_env ? args.envs_per_block * s->vert_stride : s->vert_stride;
  args.world_slots = (slots > 0 && slots <= 256) ? slots : 0;
  // worlds of more than 32 agents: candidates come from an in-block uniform grid (cell = neighborDist + 0.1 %)
  args.tile_grid_inv_cell = 0.f;
  // (per-agent parameters: the largest neighborDist of the table)
  const float nd = HETERO ? s->max_nd : s->p.neighbor_dist;
  if (N > 32 && nd > 0.f && std::getenv("ORCA_B200_NO_TILE_GRID") == nullptr)
    args.tile_grid_inv_cell = 1.0f / (nd * 1.001f);
  size_t smem = orca::step_smem_bytes(K, tpb, true, args.world_slots, OL, HETERO);
  auto kern = orca::step_small_kernel<K, KFULL, POLICY, OL, HETERO>;
  // function attributes are per device: one flag per (instantiation, device)
  // (distinct handles may be driven from distinct threads: atomic flags; setting the attribute twice is harmless)
  static std::atomic<bool> attr_set[orca::kMaxDevices];
  if (s->device >= orca::kMaxDevices || !attr_set[s->device].load(std::memory_order_acquire)) {
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)orca::step_smem_bytes(K, 256, true, 256, OL, HETERO)));
    // the whole unified L1 as shared memory: the resident-block count is what this kernel lives on
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    if (s->device < orca::kMaxDevices) attr_set[s->device].store(true, std::memory_order_release);
  }
  if (const char* e = std::getenv("ORCA_B200_SMEM_PAD")) {  // dev knob: extra shared memory = fewer resident blocks (occupancy experiments)
    const long v = std::atol(e);
    if (v > 0 && smem + (size_t)v <= 227 * 1024) {
      smem += (size_t)v;
      CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
  }
  kern<<<blocks, tpb, smem, st>>>(args, HETERO ? s->d_agent_params : nullptr);
  CUDA_TRY(cudaGetLastError());
  s->launches += 1;
  return ORCA_OK;
}

template <int K, bool KFULL, int POLICY>
int launch_small_kp(OrcaSim* s, const orca::StepArgs& a, cudaStream_t st) {
  // a world of at most 4 processed vertices (none, or one wall) gives an agent at most 2 obstacle lines:
  // the K + 2 slot kernel, four blocks per SM (see step_small_kernel).  Instantiated for K = 10 (the ALAN
  // shells' maxNeighbors: BASELINE configs 2 and 3) only.
  // (worlds of more than 32 agents search through the candidate buffer, which lives in the line slots:
  // with 12 instead of 16 of them the smaller buffer costs more than the fourth block gains -- measured
  // 509 vs 501 us for 50-agent crowds, 497 vs 492 us for 256-agent crowds)
  if (K == 10 && s->vert_stride <= 4 && s->N <= 32 && std::getenv("ORCA_B200_NO_SLIM_KERNEL") == nullptr)
    return launch_small_kpo<10, true, POLICY, 2>(s, a, st);
  return launch_small_kpo<K, KFULL, POLICY, ORCA_MAX_OBST_LINES>(s, a, st);
}

template <int K, bool KFULL>
int launch_small_k(OrcaSim* s, const orca::StepArgs& a, int policy, cudaStream_t st) {
  switch (policy) {
    case ORCA_POLICY_EXTERNAL:
      return launch_small_kp<K, KFULL, orca::POLICY_EXTERNAL>(s, a, st);
    case ORCA_POLICY_GOAL:
      return launch_small_kp<K, KFULL, orca::POLICY_GOAL>(s, a, st);
    case ORCA_POLICY_RL:
      return launch_small_kp<K, KFULL, orca::POLICY_RL>(s, a, st);
    case ORCA_POLICY_ALAN:
      return launch_small_kp<K, KFULL, orca::POLICY_ALAN>(s, a, st);
    default:
      return fail(ORCA_ERR_INVALID, "unknown policy %d", policy);
  }
}

// Per-agent parameters: the HETERO variants of the full tile kernel and of the grid kernel, K from the
// handle's maxNeighbors (the width of the neighbor-list rows), lists of KFULL = false (per-agent k <= K).
template <int K, int POLICY>
int launch_hetero_kp(OrcaSim* s, const orca::StepArgs& a, cudaStream_t st) {
  if (s->N >= s->grid_min_agents)
    return orca::launch_grid_kpo<K, false, POLICY, ORCA_MAX_OBST_LINES, true>(s->grid, a, st, &s->launches, &g_last_error,
                                                                              s->d_agent_params);
  return launch_small_kpo<K, false, POLICY, ORCA_MAX_OBST_LINES, true>(s, a, st);
}

template <int K>
int launch_hetero_k(OrcaSim* s, const orca::StepArgs& a, int policy, cudaStream_t st) {
  switch (policy) {
    case ORCA_POLICY_EXTERNAL:
      return launch_hetero_kp<K, orca::POLICY_EXTERNAL>(s, a, st);
    case ORCA_POLICY_GOAL:
      return launch_hetero_kp<K, orca::POLICY_GOAL>(s, a, st);
    case ORCA_POLICY_RL:
      return launch_hetero_kp<K, orca::POLICY_RL>(s, a, st);
    case ORCA_POLICY_ALAN:
      return launch_hetero_kp<K, orca::POLICY_ALAN>(s, a, st);
    default:
      return fail(ORCA_ERR_INVALID, "unknown policy %d", policy);
  }
}

int launch_step(OrcaSim* s, const orca::StepArgs& a0, int policy, cudaStream_t st) {
  orca::StepArgs a = a0;
  // searches that run on a shrinking threshold (worlds of more than 32 agents) start from last step's
  // k-th neighbor distance; the parity hook orca_neighbors stays stateless
  if (s->d_nbr_hint != nullptr && !a.neighbors_only && std::getenv("ORCA_B200_NO_NBR_HINT") == nullptr) {
    a.nbr_hint = s->d_nbr_hint;  // allocated by orca_create (never inside a launch: the host path captures graphs)
    a.hint_slack = 2.5f * s->p.max_speed * s->p.time_step + 1e-4f;
  }
  if (s->d_agent_params != nullptr) {
    a.nd_sq = s->max_nd * s->max_nd;  // what the kernels still read of it: the cell size of the uniform grid
    const int K = pick_k(s->p.max_neighbors);
    if (K == 5) return launch_hetero_k<5>(s, a, policy, st);
    if (K == 10) return launch_hetero_k<10>(s, a, policy, st);
    return launch_hetero_k<16>(s, a, policy, st);
  }
  if (s->N >= s->grid_min_agents) {
    return orca::launch_grid_step(s->grid, a, policy, st, &s->launches, &g_last_error);
  }
  const int k = s->p.max_neighbors;
  if (k == 5) return launch_small_k<5, true>(s, a, policy, st);
  if (k == 10) return launch_small_k<10, true>(s, a, policy, st);
  if (k <= 16) return launch_small_k<16, false>(s, a, policy, st);
  return fail(ORCA_ERR_UNSUPPORTED, "max_neighbors=%d > 16 is not supported", k);
}

// The largest obstacle range (timeHorizonObst * maxSpeed + radius) of any agent of the handle.
float obstacle_range(const OrcaSim* s) {
  if (s->d_agent_params != nullptr) return s->max_orange;
  return s->p.time_horizon_obst * s->p.max_speed + s->p.radius;
}

// Obstacle-free maps of the current obstacle worlds for the current obstacle range: where no edge can
// come within that range, the step skips the BSP walk.
int build_cull_maps(OrcaSim* s) {
  cudaFree(s->d_cull_rows);
  cudaFree(s->d_cull_geo);
  s->d_cull_rows = nullptr;
  s->d_cull_geo = nullptr;
  if (s->vert_stride == 0 || std::getenv("ORCA_B200_NO_OBST_CULL") != nullptr) return ORCA_OK;
  const float orange = obstacle_range(s);
  const size_t n_worlds = s->worlds.size();
  std::vector<uint32_t> rows(n_worlds * orca_host::kCullGrid);
  std::vector<float4> geo(n_worlds);
  for (size_t w = 0; w < n_worlds; ++w) {
    const orca_host::CullMap M = orca_host::build_cull_map(s->worlds[w], orange);
    std::memcpy(&rows[w * orca_host::kCullGrid], M.rows, sizeof(M.rows));
    geo[w] = make_float4(M.x0, M.y0, M.inv_cx, M.inv_cy);
  }
  CUDA_TRY(cudaMalloc(&s->d_cull_rows, rows.size() * sizeof(uint32_t)));
  CUDA_TRY(cudaMalloc(&s->d_cull_geo, geo.size() * sizeof(float4)));
  CUDA_TRY(cudaMemcpy(s->d_cull_rows, rows.data(), rows.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(s->d_cull_geo, geo.data(), geo.size() * sizeof(float4), cudaMemcpyHostToDevice));
  s->cull_range = orange;
  return ORCA_OK;
}

orca::BspTables bsp_tables(const OrcaSim* s) {
  orca::BspTables T;
  T.bsp = s->d_bsp;
  T.bsp_seg = s->d_bsp_seg;
  T.env_nodes = s->per_env ? s->d_env_nodes : nullptr;
  T.shared_nodes = s->shared_nodes;
  T.vert_stride = s->per_env ? s->vert_stride : 0;
  return T;
}

orca::RoadmapArgs roadmap_args(const OrcaSim* s) {
  orca::RoadmapArgs a;
  a.bsp = bsp_tables(s);
  a.W = s->rm_tables;
  a.R = s->rm_R;
  a.G = s->rm_G;
  a.words = (s->rm_R + 31) / 32;
  a.xy_per_table = s->rm_per_env ? 1 : 0;
  a.obst_per_table = (s->per_env && s->vert_stride > 0) ? 1 : 0;
  a.radius = s->rm_radius;
  a.xy = s->d_rm_xy;
  a.adj = s->d_rm_adj;
  a.dist = s->d_rm_dist;
  return a;
}

void free_roadmap_tables(OrcaSim* s) {
  cudaFree(s->d_rm_xy);
  cudaFree(s->d_rm_adj);
  cudaFree(s->d_rm_dist);
  s->d_rm_xy = nullptr;
  s->d_rm_adj = nullptr;
  s->d_rm_dist = nullptr;
  s->rm_tables = 0;
}

// Edges and goal distances of the kept roadmap over the current obstacle worlds (Roadmap.cpp
// buildRoadmap), computed on the device; synchronises.
int build_roadmap(OrcaSim* s) {
  free_roadmap_tables(s);
  if (s->rm_R == 0) return ORCA_OK;
  const int R = s->rm_R, G = s->rm_G, words = (R + 31) / 32;
  const int W = (s->rm_per_env || s->per_env) ? s->E : 1;
  const size_t xy_rows = s->rm_per_env ? (size_t)s->E : 1;
  CUDA_TRY(cudaMalloc(&s->d_rm_xy, xy_rows * R * sizeof(float2)));
  CUDA_TRY(cudaMalloc(&s->d_rm_adj, (size_t)W * R * words * sizeof(uint32_t)));
  CUDA_TRY(cudaMalloc(&s->d_rm_dist, (size_t)W * G * R * sizeof(float)));
  CUDA_TRY(cudaMemcpy(s->d_rm_xy, s->rm_host_xy.data(), xy_rows * R * sizeof(float2), cudaMemcpyHostToDevice));
  s->rm_tables = W;
  const orca::RoadmapArgs a = roadmap_args(s);
  const long long threads = (long long)W * R * words * 32;
  orca::roadmap_edges_kernel<<<(unsigned)((threads + 255) / 256), 256>>>(a);
  CUDA_TRY(cudaGetLastError());
  // one thread per vertex (R <= 512); shared memory: vertices, adjacency, distances
  const int tpb = std::max(32, (R + 31) / 32 * 32);
  const size_t smem = (size_t)R * sizeof(float2) + (size_t)R * words * sizeof(uint32_t) + (size_t)R * sizeof(float);
  orca::roadmap_dist_kernel<<<(unsigned)((long long)W * G), tpb, smem>>>(a);
  CUDA_TRY(cudaGetLastError());
  s->launches += 2;
  CUDA_TRY(cudaDeviceSynchronize());
  return ORCA_OK;
}

int ensure_host_staging(OrcaSim* s) {
  if (s->d_pos != nullptr) return ORCA_OK;
  const size_t bytes = (size_t)s->E * s->N * sizeof(float2);
  CUDA_TRY(cudaMalloc(&s->d_pos, bytes));
  CUDA_TRY(cudaMalloc(&s->d_vel, bytes));
  CUDA_TRY(cudaMalloc(&s->d_aux, bytes));
  for (int c = 0; c < kHostChunksMax; ++c) {
    CUDA_TRY(cudaStreamCreateWithFlags(&s->host_streams[c], cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&s->host_join[c], cudaEventDisableTiming));
  }
  CUDA_TRY(cudaEventCreateWithFlags(&s->host_fork, cudaEventDisableTiming));
  return ORCA_OK;
}

template <int K>
int launch_agent_lines(OrcaSim* s, const orca::StepArgs& a, const orca::LinesOut& o, cudaStream_t st) {
  const float4* params = s->d_agent_params;
  if (s->N >= s->grid_min_agents) {
    // G1-G4 into the query's own grid scratch, without the step-counter bump: nothing a step reads
    // (the step's scratch, the neighbor-search hint, the step counters) is written, so the call needs
    // no ordering against steps -- only against whatever writes pos / vel, and against other
    // orca_agent_lines calls on the handle (they share this scratch)
    orca::GridScratch& G = s->lines_grid;
    const int rc = orca::grid_prep(G, a, 0, st, &g_last_error);
    if (rc != 0) return rc;
    const int T = s->E * s->N;
    const int tpb = orca::kLinesGridThreads;
    const size_t smem = (size_t)(K + ORCA_MAX_OBST_LINES) * tpb * sizeof(float4);
    auto kern = orca::agent_lines_grid_kernel<K>;
    static std::atomic<bool> attr_set[orca::kMaxDevices];  // function attributes are per device
    if (s->device >= orca::kMaxDevices || !attr_set[s->device].load(std::memory_order_acquire)) {
      CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      if (s->device < orca::kMaxDevices) attr_set[s->device].store(true, std::memory_order_release);
    }
    kern<<<(T + tpb - 1) / tpb, tpb, smem, st>>>(a, G.sorted_pv, G.sorted_idx, G.cell_start, G.params, params, o);
    CUDA_TRY(cudaGetLastError());
    s->launches += orca::kGridLaunchesPerStep;
    return ORCA_OK;
  }
  const int tpb = orca::kLinesTileThreads;
  orca::StepArgs args = a;
  args.envs_per_block = tpb / s->N;
  const int blocks = (s->E + args.envs_per_block - 1) / args.envs_per_block;
  const size_t smem = orca::lines_tile_smem_bytes(tpb);
  auto kern = orca::agent_lines_tile_kernel<K>;
  static std::atomic<bool> attr_set[orca::kMaxDevices];
  if (s->device >= orca::kMaxDevices || !attr_set[s->device].load(std::memory_order_acquire)) {
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (s->device < orca::kMaxDevices) attr_set[s->device].store(true, std::memory_order_release);
  }
  kern<<<blocks, tpb, smem, st>>>(args, params, o);
  CUDA_TRY(cudaGetLastError());
  s->launches += 1;
  return ORCA_OK;
}

}  // namespace

extern "C" {

int orca_abi_version(void) { return ORCA_B200_ABI_VERSION; }
const char* orca_last_error(void) { return g_last_error.c_str(); }

int orca_create(const OrcaParams* params, int device, int num_envs, int agents_per_env, OrcaSim** out) {
  if (params == nullptr || out == nullptr) return fail(ORCA_ERR_INVALID, "null argument");
  if (num_envs <= 0 || agents_per_env <= 0) return fail(ORCA_ERR_INVALID, "num_envs and agents_per_env must be > 0");
  if ((long long)num_envs * agents_per_env > (1ll << 30)) return fail(ORCA_ERR_UNSUPPORTED, "more than 2^30 agents");
  if (!(params->time_step > 0.f) || !(params->time_horizon > 0.f) || !(params->time_horizon_obst > 0.f))
    return fail(ORCA_ERR_INVALID, "time_step / time_horizon / time_horizon_obst must be > 0");
  if (params->max_neighbors < 0) return fail(ORCA_ERR_INVALID, "max_neighbors must be >= 0");
  if (pick_k(params->max_neighbors) < 0)
    return fail(ORCA_ERR_UNSUPPORTED, "max_neighbors=%d > 16 is not supported", params->max_neighbors);
  int ndev = 0;
  CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(ORCA_ERR_INVALID, "device %d out of range (%d visible)", device, ndev);
  DeviceGuard guard(device);
  OrcaSim* s = new OrcaSim();
  s->p = *params;
  s->device = device;
  s->E = num_envs;
  s->N = agents_per_env;
  // tuning knob (DESIGN.md section 5): the shared-memory tile path covers at most 256 agents per env
  if (const char* e = std::getenv("ORCA_B200_GRID_MIN_AGENTS")) {
    const int v = std::atoi(e);
    if (v >= 1 && v <= 257) s->grid_min_agents = v;
  }
  if (s->N > 32) {  // starting thresholds of the threshold searches (agent_front); 0x7f7f7f7f = 3.4e38: no hint yet
    const size_t n = (size_t)s->E * s->N;
    if (cudaMalloc(&s->d_nbr_hint, n * sizeof(float)) != cudaSuccess || cudaMemset(s->d_nbr_hint, 0x7f, n * sizeof(float)) != cudaSuccess) {
      const int rc = fail(ORCA_ERR_CUDA, "allocating the neighbor-search scratch failed: %s", cudaGetErrorString(cudaGetLastError()));
      cudaFree(s->d_nbr_hint);
      delete s;
      return rc;
    }
  }
  *out = s;
  return ORCA_OK;
}

int orca_destroy(OrcaSim* s) {
  if (s == nullptr) return ORCA_OK;
  DeviceGuard guard(s->device);
  free_obstacles(s);
  free_roadmap_tables(s);
  cudaFree(s->d_pos);
  cudaFree(s->d_vel);
  cudaFree(s->d_aux);
  cudaFree(s->d_nbr_hint);
  cudaFree(s->d_agent_params);
  if (s->host_graph_exec) cudaGraphExecDestroy(s->host_graph_exec);
  for (int c = 0; c < kHostChunksMax; ++c) {
    if (s->host_streams[c]) cudaStreamDestroy(s->host_streams[c]);
    if (s->host_join[c]) cudaEventDestroy(s->host_join[c]);
  }
  if (s->host_fork) cudaEventDestroy(s->host_fork);
  orca::grid_free(s->grid);
  orca::grid_free(s->lines_grid);
  delete s;
  return ORCA_OK;
}

int orca_get_params(const OrcaSim* s, OrcaParams* out, int* num_envs, int* agents_per_env) {
  if (s == nullptr) return fail(ORCA_ERR_INVALID, "null handle");
  if (out) *out = s->p;
  if (num_envs) *num_envs = s->E;
  if (agents_per_env) *agents_per_env = s->N;
  return ORCA_OK;
}

int orca_set_obstacles(OrcaSim* s, const float* xy, const int32_t* poly_sizes, int num_polys,
                       const int32_t* polys_per_env) {
  if (s == nullptr) return fail(ORCA_ERR_INVALID, "null handle");
  if (num_polys < 0 || (num_polys > 0 && (xy == nullptr || poly_sizes == nullptr)))
    return fail(ORCA_ERR_INVALID, "bad polygon arguments");
  DeviceGuard guard(s->device);
  free_obstacles(s);
  s->per_env = (polys_per_env != nullptr);
  const int n_worlds = s->per_env ? s->E : 1;
  s->worlds.resize((size_t)n_worlds);
  int poly = 0;
  size_t off = 0;
  for (int w = 0; w < n_worlds; ++w) {
    const int np = s->per_env ? polys_per_env[w] : num_polys;
    if (np < 0 || poly + np > num_polys) return fail(ORCA_ERR_INVALID, "polys_per_env does not match num_polys");
    for (int q = 0; q < np; ++q, ++poly) {
      if (orca_host::add_polygon(s->worlds[(size_t)w], xy + 2 * off, poly_sizes[poly]) < 0) {
        free_obstacles(s);
        return fail(ORCA_ERR_INVALID, "polygon %d has fewer than 2 vertices", poly);
      }
      off += (size_t)poly_sizes[poly];
    }
    orca_host::process(s->worlds[(size_t)w]);
    if (s->worlds[(size_t)w].depth > ORCA_MAX_BSP_DEPTH - 1) {
      free_obstacles(s);
      return fail(ORCA_ERR_UNSUPPORTED, "obstacle BSP depth %d exceeds %d", s->worlds[(size_t)w].depth,
                  ORCA_MAX_BSP_DEPTH - 1);
    }
  }
  if (poly != num_polys) return fail(ORCA_ERR_INVALID, "polys_per_env does not cover all polygons");
  int stride = 0;
  for (const auto& T : s->worlds) stride = T.num_vertices() > stride ? T.num_vertices() : stride;
  if (stride == 0) return build_roadmap(s);  // no obstacles at all
  std::vector<float4> pd((size_t)n_worlds * stride), seg((size_t)n_worlds * stride);
  std::vector<int4> link((size_t)n_worlds * stride), bsp((size_t)n_worlds * stride);
  std::vector<int> nodes((size_t)n_worlds);
  for (int w = 0; w < n_worlds; ++w) {
    const auto& T = s->worlds[(size_t)w];
    nodes[(size_t)w] = T.num_nodes();
    for (int v = 0; v < stride; ++v) {
      const size_t o = (size_t)w * stride + v;
      if (v < T.num_vertices()) {
        pd[o] = make_float4(T.px[v], T.py[v], T.ux[v], T.uy[v]);
        link[o] = make_int4(T.next[v], T.prev[v], T.convex[v], 0);
      } else {
        pd[o] = make_float4(0, 0, 1, 0);
        link[o] = make_int4(0, 0, 0, 0);
      }
      if (v < T.num_nodes()) {
        const int e1 = T.node_vertex[v], e2 = T.next[e1];
        bsp[o] = make_int4(e1, T.node_left[v], T.node_right[v], 0);
        seg[o] = make_float4(T.px[e1], T.py[e1], T.px[e2], T.py[e2]);
      } else {
        bsp[o] = make_int4(0, -1, -1, 0);
        seg[o] = make_float4(0, 0, 1, 0);
      }
    }
  }
  CUDA_TRY(cudaMalloc(&s->d_vert_pd, pd.size() * sizeof(float4)));
  CUDA_TRY(cudaMalloc(&s->d_vert_link, link.size() * sizeof(int4)));
  CUDA_TRY(cudaMalloc(&s->d_bsp, bsp.size() * sizeof(int4)));
  CUDA_TRY(cudaMalloc(&s->d_bsp_seg, seg.size() * sizeof(float4)));
  CUDA_TRY(cudaMemcpy(s->d_bsp_seg, seg.data(), seg.size() * sizeof(float4), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(s->d_vert_pd, pd.data(), pd.size() * sizeof(float4), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(s->d_vert_link, link.data(), link.size() * sizeof(int4), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(s->d_bsp, bsp.data(), bsp.size() * sizeof(int4), cudaMemcpyHostToDevice));
  if (s->per_env) {
    CUDA_TRY(cudaMalloc(&s->d_env_nodes, nodes.size() * sizeof(int)));
    CUDA_TRY(cudaMemcpy(s->d_env_nodes, nodes.data(), nodes.size() * sizeof(int), cudaMemcpyHostToDevice));
  }
  s->shared_nodes = s->per_env ? 0 : nodes[0];
  s->vert_stride = stride;
  const int rc = build_cull_maps(s);
  if (rc != ORCA_OK) return rc;
  return build_roadmap(s);  // the roadmap's edges and distances depend on the obstacles
}

int orca_set_agent_params(OrcaSim* s, const float* neighbor_dist, const int32_t* max_neighbors, const float* time_horizon,
                          const float* time_horizon_obst, const float* radius, const float* max_speed) {
  if (s == nullptr) return fail(ORCA_ERR_INVALID, "null handle");
  const bool any = neighbor_dist || max_neighbors || time_horizon || time_horizon_obst || radius || max_speed;
  const size_t n = (size_t)s->E * s->N;
  std::vector<float4> table;
  float max_nd = 0.f, max_orange = 0.f;
  if (any) {
    table.resize(2 * n);
    for (size_t i = 0; i < n; ++i) {
      const float nd = neighbor_dist ? neighbor_dist[i] : s->p.neighbor_dist;
      const int k = max_neighbors ? max_neighbors[i] : s->p.max_neighbors;
      const float th = time_horizon ? time_horizon[i] : s->p.time_horizon;
      const float tho = time_horizon_obst ? time_horizon_obst[i] : s->p.time_horizon_obst;
      const float r = radius ? radius[i] : s->p.radius;
      const float vmax = max_speed ? max_speed[i] : s->p.max_speed;
      if (!std::isfinite(nd) || !std::isfinite(th) || !std::isfinite(tho) || !std::isfinite(r) || !std::isfinite(vmax))
        return fail(ORCA_ERR_INVALID, "agent %zu: parameters must be finite", i);
      if (!(th > 0.f) || !(tho > 0.f)) return fail(ORCA_ERR_INVALID, "agent %zu: time_horizon and time_horizon_obst must be > 0", i);
      if (!(nd >= 0.f) || !(r >= 0.f) || !(vmax >= 0.f))
        return fail(ORCA_ERR_INVALID, "agent %zu: neighbor_dist, radius and max_speed must be >= 0", i);
      if (k < 0 || k > s->p.max_neighbors)
        return fail(ORCA_ERR_INVALID, "agent %zu: max_neighbors %d outside [0, %d] (the handle's max_neighbors)", i, k,
                    s->p.max_neighbors);
      // the expressions of fill_common: a table of the handle's values gives the uniform results bit for bit
      const float orange = tho * vmax + r;
      table[2 * i] = make_float4(r, vmax, 1.0f / th, 1.0f / tho);
      table[2 * i + 1] = make_float4(nd * nd, orange * orange, orca::bits_to_float(k), 0.f);
      max_nd = std::max(max_nd, nd);
      max_orange = std::max(max_orange, orange);
    }
  }
  DeviceGuard guard(s->device);
  CUDA_TRY(cudaDeviceSynchronize());  // steps in flight may still read the old table
  if (s->host_graph_exec) {  // the captured host step has the old table baked into its kernel arguments
    cudaGraphExecDestroy(s->host_graph_exec);
    s->host_graph_exec = nullptr;
  }
  cudaFree(s->d_agent_params);
  s->d_agent_params = nullptr;
  if (any) {
    CUDA_TRY(cudaMalloc(&s->d_agent_params, table.size() * sizeof(float4)));
    CUDA_TRY(cudaMemcpy(s->d_agent_params, table.data(), table.size() * sizeof(float4), cudaMemcpyHostToDevice));
    s->max_nd = max_nd;
    s->max_orange = max_orange;
  }
  // the obstacle-free maps must cover the largest obstacle range of any agent
  if (s->vert_stride > 0 && obstacle_range(s) != s->cull_range) return build_cull_maps(s);
  return ORCA_OK;
}

int orca_obstacle_vertex_count(const OrcaSim* s, int env) {
  if (s == nullptr) return fail(ORCA_ERR_INVALID, "null handle");
  if (s->worlds.empty()) return 0;
  const size_t w = s->per_env ? (size_t)env : 0;
  if (w >= s->worlds.size()) return fail(ORCA_ERR_INVALID, "env %d out of range", env);
  return s->worlds[w].num_vertices();
}

int orca_get_obstacle_vertices(const OrcaSim* s, int env, float* xy_out, int32_t* next_out, int32_t* prev_out,
                               int32_t* convex_out) {
  if (s == nullptr) return fail(ORCA_ERR_INVALID, "null handle");
  if (s->worlds.empty()) return ORCA_OK;
  const size_t w = s->per_env ? (size_t)env : 0;
  if (w >= s->worlds.size()) return fail(ORCA_ERR_INVALID, "env %d out of range", env);
  const auto& T = s->worlds[w];
  for (int v = 0; v < T.num_vertices(); ++v) {
    if (xy_out) {
      xy_out[2 * v] = T.px[(size_t)v];
      xy_out[2 * v + 1] = T.py[(size_t)v];
    }
    if (next_out) next_out[v] = T.next[(size_t)v];
    if (prev_out) prev_out[v] = T.prev[(size_t)v];
    if (convex_out) convex_out[v] = T.convex[(size_t)v];
  }
  return ORCA_OK;
}

int orca_query_visibility(OrcaSim* s, const float* q1_dev, const float* q2_dev, const float* radius_dev, float radius,
                          int queries_per_env, uint8_t* visible_dev, void* stream) {
  if (s == nullptr) return fail(ORCA_ERR_INVALID, "null handle");
  if (queries_per_env < 0) return fail(ORCA_ERR_INVALID, "queries_per_env must be >= 0");
  if (queries_per_env == 0) return ORCA_OK;
  if (q1_dev == nullptr || q2_dev == nullptr || visible_dev == nullptr)
    return fail(ORCA_ERR_INVALID, "orca_query_visibility: null pointer argument");
  if (radius_dev == nullptr && !(std::isfinite(radius) && radius >= 0.f))
    return fail(ORCA_ERR_INVALID, "radius must be finite and >= 0");
  const long long total = (long long)s->E * queries_per_env;
  if (total >= (1ll << 38)) return fail(ORCA_ERR_UNSUPPORTED, "E * queries_per_env must be below 2^38");
  DeviceGuard guard(s->device);
  orca::visibility_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      bsp_tables(s), s->E, queries_per_env, reinterpret_cast<const float2*>(q1_dev), reinterpret_cast<const float2*>(q2_dev),
      radius_dev, radius, visible_dev);
  CUDA_TRY(cudaGetLastError());
  s->launches += 1;
  return ORCA_OK;
}

int orca_set_roadmap(OrcaSim* s, const float* xy, int num_vertices, int num_goals, int per_env, float radius) {
  if (s == nullptr) return fail(ORCA_ERR_INVALID, "null handle");
  if (num_vertices < 0) return fail(ORCA_ERR_INVALID, "num_vertices must be >= 0");
  std::vector<float> host;
  if (num_vertices > 0) {
    if (num_vertices > orca::kRoadmapMaxVertices)
      return fail(ORCA_ERR_UNSUPPORTED, "a roadmap has at most %d vertices (got %d)", orca::kRoadmapMaxVertices, num_vertices);
    if (num_goals < 1 || num_goals > num_vertices)
      return fail(ORCA_ERR_UNSUPPORTED, "num_goals must be in [1, num_vertices] (got %d of %d)", num_goals, num_vertices);
    if (xy == nullptr) return fail(ORCA_ERR_INVALID, "null vertex array");
    if (!(std::isfinite(radius) && radius >= 0.f)) return fail(ORCA_ERR_INVALID, "radius must be finite and >= 0");
    host.assign(xy, xy + (size_t)(per_env ? s->E : 1) * num_vertices * 2);
    for (size_t i = 0; i < host.size(); ++i)
      if (!std::isfinite(host[i])) return fail(ORCA_ERR_INVALID, "roadmap vertex coordinates must be finite");
  }
  DeviceGuard guard(s->device);
  CUDA_TRY(cudaDeviceSynchronize());  // preferred-velocity launches in flight may still read the old tables
  s->rm_host_xy.swap(host);
  s->rm_R = num_vertices;
  s->rm_G = num_vertices > 0 ? num_goals : 0;
  s->rm_per_env = num_vertices > 0 && per_env != 0;
  s->rm_radius = radius;
  const int rc = build_roadmap(s);
  if (rc != ORCA_OK) {
    s->rm_R = 0;  // no half-built roadmap
    free_roadmap_tables(s);
  }
  return rc;
}

int orca_get_roadmap(const OrcaSim* s, int env, uint32_t* adjacency_out, float* dist_out) {
  if (s == nullptr) return fail(ORCA_ERR_INVALID, "null handle");
  if (s->rm_R == 0) return fail(ORCA_ERR_STATE, "no roadmap is set");
  if (env < 0 || env >= s->E) return fail(ORCA_ERR_INVALID, "env %d out of range", env);
  DeviceGuard guard(s->device);
  const size_t t = s->rm_tables > 1 ? (size_t)env : 0;
  const size_t words = (size_t)(s->rm_R + 31) / 32;
  if (adjacency_out != nullptr)
    CUDA_TRY(cudaMemcpy(adjacency_out, s->d_rm_adj + t * s->rm_R * words, (size_t)s->rm_R * words * sizeof(uint32_t),
                        cudaMemcpyDeviceToHost));
  if (dist_out != nullptr)
    CUDA_TRY(cudaMemcpy(dist_out, s->d_rm_dist + t * s->rm_G * s->rm_R, (size_t)s->rm_G * s->rm_R * sizeof(float),
                        cudaMemcpyDeviceToHost));
  return ORCA_OK;
}

int orca_roadmap_pref_velocity(OrcaSim* s, const float* pos_dev, const int32_t* goal_vertex_dev, float* pref_dev,
                               int32_t* vertex_out_dev, void* stream) {
  if (s == nullptr) return fail(ORCA_ERR_INVALID, "null handle");
  if (s->rm_R == 0) return fail(ORCA_ERR_STATE, "orca_roadmap_pref_velocity before orca_set_roadmap");
  if (pos_dev == nullptr || goal_vertex_dev == nullptr || pref_dev == nullptr)
    return fail(ORCA_ERR_INVALID, "orca_roadmap_pref_velocity: null pointer argument");
  DeviceGuard guard(s->device);
  const orca::RoadmapArgs a = roadmap_args(s);
  const long long total = (long long)s->E * s->N;
  const unsigned blocks = (unsigned)((total + 127) / 128);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const float2* pos = reinterpret_cast<const float2*>(pos_dev);
  float2* pref = reinterpret_cast<float2*>(pref_dev);
  orca::roadmap_pref_kernel<<<blocks, 128, 0, st>>>(a, s->E, s->N, pos, goal_vertex_dev, s->d_agent_params, s->p.radius,
                                                    pref, vertex_out_dev);
  CUDA_TRY(cudaGetLastError());
  s->launches += 1;
  return ORCA_OK;
}

int orca_step(OrcaSim* s, float* pos_dev, float* vel_dev, const float* pref_dev, void* stream) {
  if (s == nullptr) return fail(ORCA_ERR_INVALID, "null handle");
  if (pos_dev == nullptr || vel_dev == nullptr || pref_dev == nullptr) return fail(ORCA_ERR_INVALID, "null state pointer");
  DeviceGuard guard(s->device);
  orca::StepArgs a;
  fill_common(s, &a);
  a.pos = reinterpret_cast<float2*>(pos_dev);
  a.vel = reinterpret_cast<float2*>(vel_dev);
  a.pref = reinterpret_cast<const float2*>(pref_dev);
  return launch_step(s, a, ORCA_POLICY_EXTERNAL, static_cast<cudaStream_t>(stream));
}

int orca_env_step(OrcaSim* s, const OrcaEnvStepArgs* in, void* stream) {
  if (s == nullptr || in == nullptr) return fail(ORCA_ERR_INVALID, "null argument");
  if (in->struct_size != sizeof(OrcaEnvStepArgs))
    return fail(ORCA_ERR_INVALID, "OrcaEnvStepArgs size mismatch (%u vs %zu): ABI skew", in->struct_size,
                sizeof(OrcaEnvStepArgs));
  if (in->pos_dev == nullptr || in->vel_dev == nullptr) return fail(ORCA_ERR_INVALID, "pos_dev / vel_dev required");
  if (in->policy == ORCA_POLICY_EXTERNAL && in->pref_dev == nullptr)
    return fail(ORCA_ERR_INVALID, "EXTERNAL policy needs pref_dev");
  if (in->policy != ORCA_POLICY_EXTERNAL && in->goal_dev == nullptr)
    return fail(ORCA_ERR_INVALID, "goal-directed policies need goal_dev");
  if (in->policy == ORCA_POLICY_RL && in->action_theta_dev == nullptr)
    return fail(ORCA_ERR_INVALID, "RL policy needs action_theta_dev");
  if (in->policy == ORCA_POLICY_ALAN) {
    if (in->alan_weights_dev == nullptr || in->alan_actions_dev == nullptr)
      return fail(ORCA_ERR_INVALID, "ALAN policy needs alan_weights_dev and alan_actions_dev");
    if (in->alan_num_actions < 1 || in->alan_num_actions > ORCA_MAX_ACTIONS)
      return fail(ORCA_ERR_UNSUPPORTED, "alan_num_actions must be in [1, %d]", ORCA_MAX_ACTIONS);
    if (!(in->alan_temp > 0.f)) return fail(ORCA_ERR_INVALID, "alan_temp must be > 0");
    if (in->alan_actions_env_stride < 0 || (in->alan_actions_env_stride > 0 && in->alan_actions_env_stride < in->alan_num_actions))
      return fail(ORCA_ERR_INVALID, "alan_actions_env_stride must be 0 or >= alan_num_actions");
    // the step counter drives the Philox counter AND the weight-window reset: without it every step
    // would repeat step 0 (same draw, no reset) -- refuse instead of misbehaving silently
    if (in->env_step_dev == nullptr) return fail(ORCA_ERR_INVALID, "ALAN policy needs env_step_dev");
  }
  if (in->arrival_time_dev != nullptr && in->env_step_dev == nullptr)
    return fail(ORCA_ERR_INVALID, "arrival_time_dev needs env_step_dev (arrival time = step * time_step)");
  if (in->done_mode < ORCA_DONE_NONE || in->done_mode > ORCA_DONE_GOAL_RADIUS_DEFERRED)
    return fail(ORCA_ERR_INVALID, "unknown done_mode %d", in->done_mode);
  if (in->done_mode != ORCA_DONE_NONE) {
    if (in->agent_done_dev == nullptr) return fail(ORCA_ERR_INVALID, "done_mode needs agent_done_dev");
    if (in->goal_dev == nullptr) return fail(ORCA_ERR_INVALID, "done_mode needs goal_dev");
  }
  if (in->nbr_idx_dev != nullptr && in->nbr_cnt_dev == nullptr) return fail(ORCA_ERR_INVALID, "nbr_idx_dev needs nbr_cnt_dev");
  if (in->obst_nbr_idx_dev != nullptr && in->obst_nbr_cnt_dev == nullptr)
    return fail(ORCA_ERR_INVALID, "obst_nbr_idx_dev needs obst_nbr_cnt_dev");
  DeviceGuard guard(s->device);
  orca::StepArgs a;
  fill_common(s, &a);
  a.pos = reinterpret_cast<float2*>(in->pos_dev);
  a.vel = reinterpret_cast<float2*>(in->vel_dev);
  a.pref = reinterpret_cast<const float2*>(in->pref_dev);
  a.goal = reinterpret_cast<float2*>(in->goal_dev);
  a.goal2 = reinterpret_cast<const float2*>(in->goal2_dev);
  a.action_theta = in->action_theta_dev;
  a.rl_scale = in->rl_reward_scale;
  a.done_x = in->done_x_threshold;
  a.alan_w = in->alan_weights_dev;
  a.alan_actions = reinterpret_cast<const float2*>(in->alan_actions_dev);
  a.alan_action_out = in->alan_action_out_dev;
  a.alan_uniform_in = in->alan_uniform_in_dev;
  a.A = in->alan_num_actions;
  a.alan_window = in->alan_window_steps;
  a.alan_gamma = in->alan_gamma;
  a.alan_inv_temp = (in->policy == ORCA_POLICY_ALAN) ? 1.0f / in->alan_temp : 0.f;
  a.seed = in->rng_seed;
  a.alan_A_env = in->alan_num_actions_env_dev;
  a.alan_env_stride = in->alan_actions_env_stride;
  a.reward = in->reward_dev;
  a.done = in->agent_done_dev;
  a.arrival = in->arrival_time_dev;
  a.env_step = in->env_step_dev;
  a.env_done_cnt = in->env_done_cnt_dev;
  a.done_mode = in->done_mode;
  a.nbr_idx = in->nbr_idx_dev;
  a.nbr_cnt = in->nbr_cnt_dev;
  a.onbr_idx = in->obst_nbr_idx_dev;
  a.onbr_cnt = in->obst_nbr_cnt_dev;
  a.stats = reinterpret_cast<unsigned long long*>(in->stats_dev);
  return launch_step(s, a, in->policy, static_cast<cudaStream_t>(stream));
}

int orca_env_step_many(OrcaSim* s, const OrcaEnvStepArgs* in, int steps, void* stream) {
  if (steps < 1) return fail(ORCA_ERR_INVALID, "steps must be >= 1");
  if (in != nullptr && in->alan_uniform_in_dev != nullptr && steps > 1)
    return fail(ORCA_ERR_INVALID, "externally supplied uniforms cover a single step");
  for (int t = 0; t < steps; ++t) {
    const int rc = orca_env_step(s, in, stream);
    if (rc != ORCA_OK) return rc;
  }
  return ORCA_OK;
}

int orca_neighbors(OrcaSim* s, const float* pos_dev, int32_t* nbr_idx_dev, float* nbr_distsq_dev, int32_t* nbr_cnt_dev,
                   int32_t* obst_nbr_idx_dev, int32_t* obst_nbr_cnt_dev, void* stream) {
  if (s == nullptr) return fail(ORCA_ERR_INVALID, "null handle");
  if (pos_dev == nullptr || nbr_idx_dev == nullptr || nbr_cnt_dev == nullptr)
    return fail(ORCA_ERR_INVALID, "pos_dev, nbr_idx_dev and nbr_cnt_dev are required");
  if (obst_nbr_idx_dev != nullptr && obst_nbr_cnt_dev == nullptr) return fail(ORCA_ERR_INVALID, "obst_nbr_idx_dev needs obst_nbr_cnt_dev");
  DeviceGuard guard(s->device);
  orca::StepArgs a;
  fill_common(s, &a);
  // the search only reads positions; velocities alias them and nothing is written back
  a.pos = reinterpret_cast<float2*>(const_cast<float*>(pos_dev));
  a.vel = a.pos;
  a.pref = a.pos;
  a.nbr_idx = nbr_idx_dev;
  a.nbr_dsq = nbr_distsq_dev;
  a.nbr_cnt = nbr_cnt_dev;
  a.onbr_idx = obst_nbr_idx_dev;
  a.onbr_cnt = obst_nbr_cnt_dev;
  a.neighbors_only = 1;
  return launch_step(s, a, ORCA_POLICY_EXTERNAL, static_cast<cudaStream_t>(stream));
}

int orca_agent_lines(OrcaSim* s, const float* pos_dev, const float* vel_dev, int max_lines, float* lines_dev,
                     int32_t* line_cnt_dev, int32_t* obst_line_cnt_dev, void* stream) {
  if (s == nullptr) return fail(ORCA_ERR_INVALID, "null handle");
  if (pos_dev == nullptr || vel_dev == nullptr || line_cnt_dev == nullptr)
    return fail(ORCA_ERR_INVALID, "orca_agent_lines: pos_dev, vel_dev and line_cnt_dev are required");
  if (max_lines < 0) return fail(ORCA_ERR_INVALID, "max_lines must be >= 0");
  if (max_lines > 0 && lines_dev == nullptr) return fail(ORCA_ERR_INVALID, "orca_agent_lines: lines_dev is required when max_lines > 0");
  DeviceGuard guard(s->device);
  orca::StepArgs a;
  fill_common(s, &a);  // no nbr_hint, env_step or stats: nothing a later step reads is written
  a.pos = reinterpret_cast<float2*>(const_cast<float*>(pos_dev));
  a.vel = reinterpret_cast<float2*>(const_cast<float*>(vel_dev));
  a.neighbors_only = 1;
  if (s->d_agent_params != nullptr) a.nd_sq = s->max_nd * s->max_nd;  // the grid's cell size, as in launch_step
  orca::LinesOut o;
  o.lines = reinterpret_cast<float4*>(lines_dev);
  o.cnt = line_cnt_dev;
  o.obst_cnt = obst_line_cnt_dev;
  o.max_lines = max_lines;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int K = pick_k(s->p.max_neighbors);
  if (K == 5) return launch_agent_lines<5>(s, a, o, st);
  if (K == 10) return launch_agent_lines<10>(s, a, o, st);
  return launch_agent_lines<16>(s, a, o, st);
}

int orca_observe(OrcaSim* s, const float* pos_dev, const float* vel_dev, const float* goal_dev, const int32_t* nbr_idx_dev,
                 const int32_t* nbr_cnt_dev, const int32_t* obst_nbr_idx_dev, const int32_t* obst_nbr_cnt_dev, int laser_num,
                 int circle_approx_num, float* obs_dev, void* stream) {
  if (s == nullptr) return fail(ORCA_ERR_INVALID, "null handle");
  if (!pos_dev || !vel_dev || !goal_dev || !nbr_idx_dev || !nbr_cnt_dev || !obst_nbr_idx_dev || !obst_nbr_cnt_dev || !obs_dev)
    return fail(ORCA_ERR_INVALID, "orca_observe: null pointer argument");
  if (laser_num < 1 || laser_num > ORCA_MAX_LASER) return fail(ORCA_ERR_UNSUPPORTED, "laser_num must be in [1, %d]", ORCA_MAX_LASER);
  if (circle_approx_num < 3 || circle_approx_num > ORCA_MAX_CIRCLE_APPROX)
    return fail(ORCA_ERR_UNSUPPORTED, "circle_approx_num must be in [3, %d]", ORCA_MAX_CIRCLE_APPROX);
  DeviceGuard guard(s->device);
  orca::ObsArgs a;
  std::memset(&a, 0, sizeof(a));
  a.E = s->E;
  a.N = s->N;
  a.k = s->p.max_neighbors > 0 ? s->p.max_neighbors : 1;
  a.R = laser_num;
  a.C = circle_approx_num;
  a.pos = reinterpret_cast<const float2*>(pos_dev);
  a.vel = reinterpret_cast<const float2*>(vel_dev);
  a.goal = reinterpret_cast<const float2*>(goal_dev);
  a.nbr_idx = nbr_idx_dev;
  a.nbr_cnt = nbr_cnt_dev;
  a.onbr_idx = obst_nbr_idx_dev;
  a.onbr_cnt = obst_nbr_cnt_dev;
  a.vert_pd = s->d_vert_pd;
  a.vert_link = s->d_vert_link;
  a.vert_stride = s->per_env ? s->vert_stride : 0;
  a.obs = reinterpret_cast<float4*>(obs_dev);
  // tables in float64 like the reference (env:321-350), rounded once to float32
  const double two_pi = 6.283185307179586476925286766559;
  for (int i = 0; i < laser_num; ++i) {
    const double th = i * (two_pi / laser_num);
    a.ray_end[i] = make_float2((float)((double)s->p.neighbor_dist * std::cos(th)), (float)(-(double)s->p.neighbor_dist * std::sin(th)));
  }
  for (int i = 0; i < circle_approx_num; ++i) {
    const double th = i * (two_pi / circle_approx_num);
    a.poly[i] = make_float2((float)((double)s->p.radius * std::cos(th)), (float)(-(double)s->p.radius * std::sin(th)));
  }
  const long long total = (long long)s->E * s->N * laser_num;
  if (total >= (1ll << 31)) return fail(ORCA_ERR_UNSUPPORTED, "orca_observe: E * N * laser_num must be below 2^31");
  const bool paired = orca::obs_table_is_antipodal(a);  // ray i + R / 2 = -ray i: one lane culls for both
  const orca::ObsPlan plan = orca::obs_plan(a, paired);
  const size_t smem = (size_t)plan.warp_bytes * orca::kObsWarps;
  {
    static std::atomic<bool> attr_set[orca::kMaxDevices];  // function attributes are per device
    if (s->device >= orca::kMaxDevices || !attr_set[s->device].load(std::memory_order_acquire)) {
      CUDA_TRY(cudaFuncSetAttribute(orca::observe_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
      CUDA_TRY(cudaFuncSetAttribute(orca::observe_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
      if (s->device < orca::kMaxDevices) attr_set[s->device].store(true, std::memory_order_release);
    }
  }
  const long long per_block = (long long)plan.A * orca::kObsWarps;  // whole agents per warp: their rays share staged data
  const long long blocks = ((long long)s->E * s->N + per_block - 1) / per_block;
  if (paired)
    orca::observe_kernel<true><<<(unsigned)blocks, orca::kObsThreads, smem, static_cast<cudaStream_t>(stream)>>>(a, plan);
  else
    orca::observe_kernel<false><<<(unsigned)blocks, orca::kObsThreads, smem, static_cast<cudaStream_t>(stream)>>>(a, plan);
  CUDA_TRY(cudaGetLastError());
  s->launches += 1;
  return ORCA_OK;
}

}  // extern "C"

namespace {
// One orca_step_host call over the route asked for: direct (kernel reads / writes the mapped host
// buffers) when `allow_direct` and the buffers are mapped, else staged copies.
int step_host_route(OrcaSim* s, float* pos_host, float* vel_host, const float* pref_or_goal_host, int policy,
                    int flags, int steps, bool allow_direct) {
  if (s == nullptr) return fail(ORCA_ERR_INVALID, "null handle");
  const int upload_state = (flags & ORCA_HOST_UPLOAD_STATE) ? 1 : 0;
  if (pos_host == nullptr || pref_or_goal_host == nullptr) return fail(ORCA_ERR_INVALID, "null host buffer");
  if (vel_host == nullptr && upload_state) return fail(ORCA_ERR_INVALID, "uploading the state needs vel_host");
  if (policy != ORCA_POLICY_EXTERNAL && policy != ORCA_POLICY_GOAL)
    return fail(ORCA_ERR_INVALID, "orca_step_host supports the EXTERNAL and GOAL policies");
  if (steps < 1) return fail(ORCA_ERR_INVALID, "steps must be >= 1");
  if (!upload_state && !s->host_state_valid)
    return fail(ORCA_ERR_STATE, "orca_step_host(upload_state = 0) before any call uploaded the state");
  DeviceGuard guard(s->device);
  int rc = ensure_host_staging(s);
  if (rc != ORCA_OK) return rc;
  if (upload_state) s->host_state_valid = true;
  // ORCA_HOST_AUX_UNCHANGED: the caller promises that the goal / pref buffer holds what it held at the
  // previous call with the same pointer; its device copy is reused and nothing is read from the host
  const bool aux_cached = (flags & ORCA_HOST_AUX_UNCHANGED) != 0 && s->host_aux_src == pref_or_goal_host;
  const bool want_vel = vel_host != nullptr;
  // ---- direct path: the host buffers are pinned and mapped -------------------------------------
  // The step kernel itself reads the goals / preferred velocities from the caller's buffer and
  // writes the new positions and velocities into the caller's buffers (as well as into the
  // device-resident state) over PCIe while it computes: no staging copies, no copy-engine
  // start-up per chunk, the transfers overlap the arithmetic warp by warp.  One launch per step.
  const bool tile_path = s->N < s->grid_min_agents;
  if (tile_path && allow_direct) {
    void *m_pos = nullptr, *m_vel = nullptr, *m_aux = nullptr;
    const bool mapped = cudaHostGetDevicePointer(&m_pos, pos_host, 0) == cudaSuccess &&
                        (!want_vel || cudaHostGetDevicePointer(&m_vel, vel_host, 0) == cudaSuccess) &&
                        cudaHostGetDevicePointer(&m_aux, const_cast<float*>(pref_or_goal_host), 0) == cudaSuccess;
    if (!mapped) {
      cudaGetLastError();  // pageable buffers: clear the error, take the staged path below
    } else {
      const size_t bytes = (size_t)s->E * s->N * sizeof(float2);
      cudaStream_t st = s->host_streams[0];
      if (upload_state) {
        CUDA_TRY(cudaMemcpyAsync(s->d_pos, pos_host, bytes, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(s->d_vel, vel_host, bytes, cudaMemcpyHostToDevice, st));
      }
      orca::StepArgs a;
      fill_common(s, &a);
      a.pos = s->d_pos;
      a.vel = s->d_vel;
      const float2* aux = static_cast<const float2*>(m_aux);
      if (aux_cached) {
        aux = s->d_aux;
      } else if (steps > 1 || (flags & ORCA_HOST_AUX_UNCHANGED)) {  // read every step / reused by later calls: bring it over once
        CUDA_TRY(cudaMemcpyAsync(s->d_aux, pref_or_goal_host, bytes, cudaMemcpyHostToDevice, st));
        aux = s->d_aux;
        s->host_aux_src = pref_or_goal_host;
      } else {
        s->host_aux_src = nullptr;
      }
      if (policy == ORCA_POLICY_EXTERNAL)
        a.pref = aux;
      else
        a.goal = const_cast<float2*>(aux);
      for (int t = 0; t < steps; ++t) {
        if (t == steps - 1) {
          a.pos_mirror = static_cast<float2*>(m_pos);
          a.vel_mirror = want_vel ? static_cast<float2*>(m_vel) : nullptr;
        }
        rc = launch_step(s, a, policy, st);
        if (rc != ORCA_OK) return rc;
      }
      CUDA_TRY(cudaStreamSynchronize(st));
      return ORCA_OK;
    }
  }
  // ---- staged path (pageable host buffers, or the uniform-grid pipeline) -----------------------
  // Envs are independent, so the batch is cut into contiguous env chunks, each on its own
  // stream: upload -> step(s) -> download.  Chunk c's kernel runs while chunk c+1 uploads and
  // chunk c-1 downloads (the two copy engines and the SMs all busy); the call costs about the
  // slowest of the three stages instead of their sum.  The uniform-grid path (one huge env)
  // cannot be cut and goes through as a single chunk.
  //
  // The whole fan-out (4 calls per chunk) is captured once into a CUDA graph keyed by the
  // buffers and arguments, and replayed with a single launch on later calls: issued call by
  // call, the CPU cost of ~16-64 runtime calls was as long as the transfers themselves.
  //
  // Chunks are NOT equal: what the call cannot hide is the first chunk's upload + step (nothing
  // to download yet) while the downloads want to be few and large (a 0.5 MB copy reaches 47 GB/s
  // here, 4 MB 55 GB/s).  So the first chunk is small and the sizes grow: weights 1 : 3 : 6 : 6.
  int chunks = 1;
  if (tile_path) {
    const long long agents = (long long)s->E * s->N;
    chunks = agents >= kHostChunkAgents * 4 ? 4 : (agents >= kHostChunkAgents ? 2 : 1);
    if (const char* e = std::getenv("ORCA_B200_HOST_CHUNKS")) {  // dev knob
      const int v = std::atoi(e);
      if (v >= 1 && v <= kHostChunksMax) chunks = v;
    }
    chunks = std::min(chunks, s->E);
  }
  // env boundaries from cumulative weights 1, 3, 6, 6, 6, ...
  int bound[kHostChunksMax + 1];
  {
    long long wsum = 0, acc = 0;
    for (int c = 0; c < chunks; ++c) wsum += (c == 0 ? 1 : (c == 1 ? 3 : 6));
    bound[0] = 0;
    for (int c = 0; c < chunks; ++c) {
      acc += (c == 0 ? 1 : (c == 1 ? 3 : 6));
      bound[c + 1] = (int)((long long)s->E * acc / wsum);
    }
    for (int c = 1; c <= chunks; ++c) bound[c] = std::max(bound[c], std::min(s->E, bound[c - 1] + 1));  // no empty chunk
    bound[chunks] = s->E;
  }
  HostGraphKey key{pos_host, vel_host, pref_or_goal_host, policy, flags | (aux_cached ? 0x100 : 0), steps, chunks};
  const bool use_graph = tile_path && std::getenv("ORCA_B200_HOST_NO_GRAPH") == nullptr;
  if (use_graph && s->host_graph_exec != nullptr && !(key == s->host_graph_key)) {
    cudaGraphExecDestroy(s->host_graph_exec);
    s->host_graph_exec = nullptr;
  }
  cudaStream_t root = s->host_streams[0];
  if (!use_graph || s->host_graph_exec == nullptr) {
    if (use_graph) {
      CUDA_TRY(cudaStreamBeginCapture(root, cudaStreamCaptureModeThreadLocal));
      CUDA_TRY(cudaEventRecord(s->host_fork, root));
      for (int c = 1; c < chunks; ++c) CUDA_TRY(cudaStreamWaitEvent(s->host_streams[c], s->host_fork, 0));
    }
    orca::StepArgs a;
    fill_common(s, &a);
    a.pos = s->d_pos;
    a.vel = s->d_vel;
    if (policy == ORCA_POLICY_EXTERNAL)
      a.pref = s->d_aux;
    else
      a.goal = s->d_aux;
    const int64_t launches_before = s->launches;
    rc = ORCA_OK;
    cudaError_t ce = cudaSuccess;
    for (int c = 0; c < chunks && rc == ORCA_OK && ce == cudaSuccess; ++c) {
      const int e0 = bound[c], e1 = bound[c + 1];
      const size_t off = (size_t)e0 * s->N;  // in agents (= float2 elements = 2 floats)
      const size_t bytes = (size_t)(e1 - e0) * s->N * sizeof(float2);
      cudaStream_t st = s->host_streams[c];
      if (upload_state) {
        ce = cudaMemcpyAsync(s->d_pos + off, pos_host + 2 * off, bytes, cudaMemcpyHostToDevice, st);
        if (ce == cudaSuccess) ce = cudaMemcpyAsync(s->d_vel + off, vel_host + 2 * off, bytes, cudaMemcpyHostToDevice, st);
      }
      if (ce == cudaSuccess && !aux_cached)
        ce = cudaMemcpyAsync(s->d_aux + off, pref_or_goal_host + 2 * off, bytes, cudaMemcpyHostToDevice, st);
      orca::StepArgs ac = a;
      ac.env_base = e0;
      ac.E = e1;
      for (int t = 0; t < steps && rc == ORCA_OK && ce == cudaSuccess; ++t) rc = launch_step(s, ac, policy, st);
      if (ce == cudaSuccess) ce = cudaMemcpyAsync(pos_host + 2 * off, s->d_pos + off, bytes, cudaMemcpyDeviceToHost, st);
      if (ce == cudaSuccess && want_vel) ce = cudaMemcpyAsync(vel_host + 2 * off, s->d_vel + off, bytes, cudaMemcpyDeviceToHost, st);
      if (use_graph && c > 0 && ce == cudaSuccess) {
        ce = cudaEventRecord(s->host_join[c], st);
        if (ce == cudaSuccess) ce = cudaStreamWaitEvent(root, s->host_join[c], 0);
      }
    }
    if (use_graph) {
      cudaGraph_t graph = nullptr;
      const cudaError_t ee = cudaStreamEndCapture(root, &graph);  // always end the capture
      if (rc != ORCA_OK) {
        if (graph) cudaGraphDestroy(graph);
        return rc;
      }
      if (ce != cudaSuccess || ee != cudaSuccess) {
        if (graph) cudaGraphDestroy(graph);
        return fail(ORCA_ERR_CUDA, "capturing the host-step graph failed: %s", cudaGetErrorString(ce != cudaSuccess ? ce : ee));
      }
      const cudaError_t ie = cudaGraphInstantiate(&s->host_graph_exec, graph, 0);
      cudaGraphDestroy(graph);
      if (ie != cudaSuccess) {
        s->host_graph_exec = nullptr;
        return fail(ORCA_ERR_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ie));
      }
      s->host_graph_key = key;
      s->host_graph_launches = s->launches - launches_before;
      s->launches = launches_before;  // nothing ran yet: capture only recorded the launches
    } else {
      if (rc != ORCA_OK) return rc;
      if (ce != cudaSuccess) return fail(ORCA_ERR_CUDA, "host step failed: %s", cudaGetErrorString(ce));
      for (int c = 0; c < chunks; ++c) CUDA_TRY(cudaStreamSynchronize(s->host_streams[c]));
      s->host_aux_src = pref_or_goal_host;
      return ORCA_OK;
    }
  }
  CUDA_TRY(cudaGraphLaunch(s->host_graph_exec, root));
  s->launches += s->host_graph_launches;
  CUDA_TRY(cudaStreamSynchronize(root));
  s->host_aux_src = pref_or_goal_host;  // the staged route always leaves a device copy of it behind
  return ORCA_OK;
}

}  // namespace

extern "C" {

int orca_step_host_ex(OrcaSim* s, float* pos_host, float* vel_host, const float* pref_or_goal_host, int policy, int flags,
                      int steps) {
  if (s == nullptr) return fail(ORCA_ERR_INVALID, "null handle");
  if (flags & ~(ORCA_HOST_UPLOAD_STATE | ORCA_HOST_AUX_UNCHANGED)) return fail(ORCA_ERR_INVALID, "unknown host-step flags 0x%x", flags);
  const bool may_direct = std::getenv("ORCA_B200_HOST_NO_MAPPED") == nullptr;
  // Which route is faster depends on the host (PCIe write efficiency of GPU stores vs copy-engine
  // bursts; measured 0.39 vs 0.45 ms on one box, 0.51 vs 0.45 ms on another).  Both give the same
  // bits, so steady-state calls (same buffers, one step, no state upload) time each route three
  // times and keep the faster one.
  const bool steady = may_direct && !(flags & ORCA_HOST_UPLOAD_STATE) && steps == 1 &&
                      std::getenv("ORCA_B200_HOST_NO_AUTOTUNE") == nullptr;
  if (!steady) return step_host_route(s, pos_host, vel_host, pref_or_goal_host, policy, flags, steps, may_direct);
  HostGraphKey key{pos_host, vel_host, pref_or_goal_host, policy, flags, 1, 0};
  if (!(key == s->tune_key)) {
    s->tune_key = key;
    s->tune_calls = 0;
    s->tune_ms[0] = s->tune_ms[1] = 0.0;
  }
  // calls 0-4: direct, calls 5-9: staged; the first call of each route warms it up (graph capture,
  // first touch), the fastest of the other four is the route's time
  constexpr int kTunePerRoute = 5;  // one warm-up call + the fastest of four (the host link of a shared box is noisy)
  bool direct;
  if (s->tune_calls < 2 * kTunePerRoute) {
    direct = s->tune_calls < kTunePerRoute;
  } else {
    direct = s->tune_ms[0] <= s->tune_ms[1];
  }
  const auto t0 = std::chrono::steady_clock::now();
  const int rc = step_host_route(s, pos_host, vel_host, pref_or_goal_host, policy, flags, steps, direct);
  if (s->tune_calls < 2 * kTunePerRoute) {
    const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    const int route = s->tune_calls / kTunePerRoute, nth = s->tune_calls % kTunePerRoute;
    if (nth == 1) s->tune_ms[route] = ms;
    if (nth >= 2) s->tune_ms[route] = std::min(s->tune_ms[route], ms);
    s->tune_calls += 1;
    if (s->tune_calls == 2 * kTunePerRoute && std::getenv("ORCA_B200_HOST_TRACE") != nullptr)
      std::fprintf(stderr, "orca_step_host: direct %.3f ms, staged %.3f ms -> %s\n", s->tune_ms[0], s->tune_ms[1],
                   s->tune_ms[0] <= s->tune_ms[1] ? "direct" : "staged");
  }
  return rc;
}

int orca_step_host(OrcaSim* s, float* pos_host, float* vel_host, const float* pref_or_goal_host, int policy,
                   int upload_state, int steps) {
  if (vel_host == nullptr) return fail(ORCA_ERR_INVALID, "null host buffer");
  return orca_step_host_ex(s, pos_host, vel_host, pref_or_goal_host, policy, upload_state ? ORCA_HOST_UPLOAD_STATE : 0, steps);
}

}  // extern "C"

namespace {
int policy_mlp_common(OrcaSim* s, const float* obs_dev, int64_t rows, const OrcaMlpWeights* w, float* out_dev, void* stream,
                      bool tensor_cores) {
  if (s == nullptr) return fail(ORCA_ERR_INVALID, "null handle");
  if (w == nullptr || obs_dev == nullptr || out_dev == nullptr) return fail(ORCA_ERR_INVALID, "orca_policy_mlp: null pointer argument");
  if (w->struct_size != sizeof(OrcaMlpWeights)) return fail(ORCA_ERR_INVALID, "OrcaMlpWeights.struct_size mismatch");
  if (w->w1_dev == nullptr || w->b1_dev == nullptr || w->w2_dev == nullptr || w->b2_dev == nullptr || w->w3_dev == nullptr ||
      w->b3_dev == nullptr)
    return fail(ORCA_ERR_INVALID, "orca_policy_mlp: null weight pointer");
  if (w->in_dim != orca::kMlpIn || w->hidden_dim != orca::kMlpHidden)
    return fail(ORCA_ERR_UNSUPPORTED, "policy network must be %d -> %d -> %d -> out (got in=%d hidden=%d)", orca::kMlpIn,
                orca::kMlpHidden, orca::kMlpHidden, w->in_dim, w->hidden_dim);
  if (w->out_dim < 1 || w->out_dim > orca::kMlpMaxOut)
    return fail(ORCA_ERR_UNSUPPORTED, "policy outputs must be in [1, %d]", orca::kMlpMaxOut);
  if (rows < 0) return fail(ORCA_ERR_INVALID, "rows must be >= 0");
  if (rows == 0) return ORCA_OK;
  if ((reinterpret_cast<uintptr_t>(obs_dev) | reinterpret_cast<uintptr_t>(w->w1_dev) | reinterpret_cast<uintptr_t>(w->w2_dev)) & 15)
    return fail(ORCA_ERR_INVALID, "obs_dev, w1_dev and w2_dev must be 16-byte aligned");
  DeviceGuard guard(s->device);
  orca::MlpArgs a;
  a.obs = obs_dev;
  a.rows = rows;
  a.w1 = w->w1_dev;
  a.b1 = w->b1_dev;
  a.w2 = w->w2_dev;
  a.b2 = w->b2_dev;
  a.w3 = w->w3_dev;
  a.b3 = w->b3_dev;
  a.n_out = w->out_dim;
  a.out = out_dev;
  static std::atomic<bool> attr_set[orca::kMaxDevices];  // function attributes are per device
  int sm_count = 0;
  CUDA_TRY(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, s->device));
  if (s->device >= orca::kMaxDevices || !attr_set[s->device].load(std::memory_order_acquire)) {
    CUDA_TRY(cudaFuncSetAttribute(orca::policy_mlp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)orca::mlp_smem_bytes()));
    CUDA_TRY(cudaFuncSetAttribute(orca::policy_mlp_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)orca::mlp_tc_smem_bytes()));
    if (s->device < orca::kMaxDevices) attr_set[s->device].store(true, std::memory_order_release);
  }
  if (tensor_cores) {
    const long long tiles = (rows + orca::kTcTile - 1) / orca::kTcTile;
    // persistent: one CTA per SM (195 KB of shared memory), two tile pipelines per CTA
    const int blocks = (int)std::min<long long>((tiles + orca::kTcGroups - 1) / orca::kTcGroups, sm_count);
    orca::policy_mlp_tc_kernel<<<blocks, orca::kTcThreads, orca::mlp_tc_smem_bytes(), static_cast<cudaStream_t>(stream)>>>(a);
  } else {
    const long long tiles = (rows + orca::kMlpTile - 1) / orca::kMlpTile;
    const int blocks = (int)std::min<long long>(tiles, 2ll * sm_count);  // persistent: 2 resident blocks per SM
    orca::policy_mlp_kernel<<<blocks, orca::kMlpThreads, orca::mlp_smem_bytes(), static_cast<cudaStream_t>(stream)>>>(a);
  }
  CUDA_TRY(cudaGetLastError());
  s->launches += 1;
  return ORCA_OK;
}
}  // namespace

extern "C" {

int orca_policy_mlp(OrcaSim* s, const float* obs_dev, int64_t rows, const OrcaMlpWeights* w, float* out_dev, void* stream) {
  return policy_mlp_common(s, obs_dev, rows, w, out_dev, stream, true);
}
int orca_policy_mlp_fp32(OrcaSim* s, const float* obs_dev, int64_t rows, const OrcaMlpWeights* w, float* out_dev, void* stream) {
  return policy_mlp_common(s, obs_dev, rows, w, out_dev, stream, false);
}

int64_t orca_launch_count(const OrcaSim* s) { return s ? s->launches : 0; }

}  // extern "C"
