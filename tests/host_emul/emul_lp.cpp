// emul_lp.cpp -- TEST-ONLY host build of the library's linear programs (csrc/orca_core.cuh).
//
// lp2 followed, when it fails, by lp3 or by lp3_stored -- the two LP3 forms the step kernels run
// (block_lp3 stores the projected programme of a round in a borrowed column, or recomputes it on
// access) -- compiled with g++ -ffp-contract=off so that the CPU suite compares them with the
// oracle bit for bit without a GPU.  Built with ORCA_EMUL_COUNT: g_orca_counters counts the LP
// branches (slot list at the top of orca_core.cuh).  The package never loads this library.
#include <cstring>
#include <vector>

#include "../../collision_avoidance_b200/csrc/orca_core.cuh"

long long g_orca_counters[16];

extern "C" {

// lines [n][4] = (point.xy, dir.xy), obstacle lines first; variant 0: lp3, 1: lp3_stored with a host
// array as the programme store.  out[2] = the new velocity; returns LP2's fail index (n on success),
// as oracle.rvo2_oracle.solve_lp does.
int emul_solve(const float* lines, int n, int n_obst, float radius, float pref_x, float pref_y, int variant,
               float* out) {
  std::vector<float4> buf(static_cast<size_t>(n > 0 ? n : 1));
  std::memcpy(buf.data(), lines, sizeof(float4) * static_cast<size_t>(n));
  orca::Lines L;
  L.base = buf.data();
  L.stride = 1;
  float2 res = orca::v2(0.f, 0.f);
  const int fail = orca::lp2(0xffffffffu, true, L, n, radius, orca::v2(pref_x, pref_y), false, res);
  if (fail < n) {
    if (variant == 1) {
      std::vector<float4> store(buf.size());
      orca::Lines P;
      P.base = store.data();
      P.stride = 1;
      orca::lp3_stored(0xffffffffu, true, L, n, n_obst, fail, radius, P, res);
    } else {
      orca::lp3(0xffffffffu, true, L, n, n_obst, fail, radius, res);
    }
  }
  out[0] = res.x;
  out[1] = res.y;
  return fail;
}

void emul_lp_counters(long long* out, int reset) {
  std::memcpy(out, g_orca_counters, sizeof(g_orca_counters));
  if (reset) std::memset(g_orca_counters, 0, sizeof(g_orca_counters));
}

}  // extern "C"
