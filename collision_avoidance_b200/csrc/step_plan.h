// step_plan.h -- which step kernel a handle runs: tile or uniform grid, and step_small_kernel /
// step_grid_kernel's (K, KFULL, OL, HETERO).  Plain values, so g++ compiles it without CUDA.
#pragma once

#include "../../include/orca_b200.h"

namespace orca_host {

// Neighbor-list width K for maxNeighbors k; -1 above 16 (orca_create refuses the handle).
inline int pick_k(int k) {
  if (k <= 5) return 5;
  if (k <= 10) return 10;
  if (k <= 16) return 16;
  return -1;
}

struct StepPlanInputs {
  int N;                // agents per env
  int max_neighbors;    // the handle's maxNeighbors k (<= 16)
  int grid_min_agents;  // worlds of at least this many agents run the uniform-grid pipeline
  int vert_stride;      // vertex slots of the largest obstacle world (0: no obstacles)
  bool per_env;         // one obstacle world per env
  bool hetero;          // per-agent parameters (orca_set_agent_params)
  bool no_slim;         // never the K + 2 kernel (ORCA_B200_NO_SLIM_KERNEL)
};

struct StepPlan {
  bool grid;    // uniform-grid pipeline (step_grid_kernel), else the tile (step_small_kernel)
  int K;        // neighbor-list width
  bool kfull;   // the handle's k equals K (the acceptance threshold is the last slot)
  int ol;       // obstacle-line slots per agent: ORCA_MAX_OBST_LINES, or 2 (the slim kernel)
  bool hetero;  // per-agent parameters
};

// Uneven on purpose; kernels are instantiated for exactly what this returns:
// - uniform k = 5 and k = 10 run K = k with KFULL lists; any other k, 0-4 included, runs K = 16;
// - per-agent parameters run K = pick_k(k) (k = 3 runs K = 5), never KFULL, never slim;
// - slim (OL = 2, uniform k = 10): at most 4 obstacle vertices (none, or one wall) give an agent at
//   most 2 obstacle lines.  The tile takes it up to 32 agents only: larger worlds keep their candidate
//   buffer in the line slots, and 12 instead of 16 slots cost more than the fourth resident block
//   gains (509 vs 501 us for 50-agent crowds, 497 vs 492 us for 256).  The grid has no N bound
//   (ORCA_B200_GRID_MIN_AGENTS can move small worlds onto it), but takes per-env worlds only when
//   they have no vertices.
inline StepPlan step_plan(const StepPlanInputs& in) {
  StepPlan p;
  p.grid = in.N >= in.grid_min_agents;
  p.hetero = in.hetero;
  p.ol = ORCA_MAX_OBST_LINES;
  const int k = in.max_neighbors;
  if (in.hetero) {
    p.K = pick_k(k);
    p.kfull = false;
    return p;
  }
  p.kfull = (k == 5 || k == 10);
  p.K = p.kfull ? k : 16;
  if (k == 10 && in.vert_stride <= 4 && !in.no_slim && (p.grid ? !in.per_env || in.vert_stride == 0 : in.N <= 32))
    p.ol = 2;
  return p;
}

}  // namespace orca_host
