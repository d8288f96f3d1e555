// lp_harness.cu -- TEST-ONLY device harness of the library's linear programs (csrc/orca_core.cuh).
//
// Each lane of a block takes one LP programme (or none), keeps its lines in a column of shared
// memory as the step kernels do (line i of lane t at [i * blockDim + t]), and runs lp2 followed,
// where LP2 failed, by lp3 or by lp3_stored with its projected programme in a second shared
// column.  Warps mix short and long programmes and lanes without one, so the ORCA_ANY vote loops
// run with lanes of every kind.  Built by tests/test_gpu_lp3_harness.py with the library's flags.
#include <cuda_runtime.h>

#include "../../collision_avoidance_b200/csrc/orca_core.cuh"

namespace {
constexpr int kMaxLines = 22;  // K = 16 agent lines + ORCA_MAX_OBST_LINES

// lines [P][kMaxLines] float4, meta[P] = n | n_obst << 8, radius[P], pref[P]; lane_prog[T]: programme of
// each lane, -1 = none.  out[T], fail[T]: result and LP2 fail index of each lane that has a programme.
__global__ void lp_harness_kernel(const float4* __restrict__ lines, const int* __restrict__ meta,
                                  const float* __restrict__ radius, const float2* __restrict__ pref,
                                  const int* __restrict__ lane_prog, int T, int variant, float2* out, int* fail_out) {
  extern __shared__ float4 smem[];
  const int tid = threadIdx.x, stride = blockDim.x;
  const int g = blockIdx.x * blockDim.x + tid;
  const int p = g < T ? lane_prog[g] : -1;
  const bool has = p >= 0;
  const int m = has ? meta[p] : 0;
  const int n = m & 0xff, n_obst = (m >> 8) & 0xff;
  orca::Lines L;
  L.base = smem + tid;
  L.stride = stride;
  orca::Lines P;
  P.base = smem + kMaxLines * stride + tid;
  P.stride = stride;
  for (int i = 0; i < n; ++i) L.base[i * stride] = lines[(size_t)p * kMaxLines + i];
  const float r = has ? radius[p] : 1.f;
  float2 res = orca::v2(0.f, 0.f);
  const int fail = orca::lp2(0xffffffffu, has, L, n, r, has ? pref[p] : orca::v2(0.f, 0.f), false, res);
  const bool need = has && fail < n;
  if (variant == 1)
    orca::lp3_stored(0xffffffffu, need, L, n, n_obst, fail, r, P, res);
  else
    orca::lp3(0xffffffffu, need, L, n, n_obst, fail, r, res);
  if (has) {
    out[g] = res;
    fail_out[g] = fail;
  }
}
}  // namespace

extern "C" int lp_harness_run(const void* lines, const void* meta, const void* radius, const void* pref,
                              const void* lane_prog, int T, int variant, int tpb, void* out, void* fail_out) {
  const size_t smem = (size_t)2 * kMaxLines * tpb * sizeof(float4);
  lp_harness_kernel<<<(T + tpb - 1) / tpb, tpb, smem>>>(
      static_cast<const float4*>(lines), static_cast<const int*>(meta), static_cast<const float*>(radius),
      static_cast<const float2*>(pref), static_cast<const int*>(lane_prog), T, variant, static_cast<float2*>(out),
      static_cast<int*>(fail_out));
  if (cudaGetLastError() != cudaSuccess) return -1;
  return cudaDeviceSynchronize() == cudaSuccess ? 0 : -2;
}

extern "C" int lp_harness_max_lines() { return kMaxLines; }
