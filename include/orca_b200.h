/* orca_b200.h -- C ABI of the B200-native batched ORCA simulator.
 *
 * This is the drop-in boundary for the reference's `rvo2.PyRVOSimulator` usage
 * (SURVEY.md section 8b).  Each entry point cites the reference call site(s) it
 * replaces; `INTEGRATION.md` shows the ctypes binding a maintainer would add.
 *
 * Conventions
 *   - plain C types only: pointers, ints, floats.  No torch types.
 *   - every function returns 0 on success and a negative OrcaStatus on error;
 *     `orca_last_error()` returns a thread-local message for the last failure.
 *   - `*_dev` pointers are CUDA device pointers on the handle's device; the caller
 *     owns them (torch tensors in the Python layer).  `stream` is a cudaStream_t
 *     cast to void* (NULL = legacy default stream).  Nothing synchronises the host
 *     unless the function name ends in `_host`.
 *   - arrays are structure-of-arrays, env-major: agent (e, a) lives at index
 *     e * agents_per_env + a; 2-vectors are interleaved (x, y) float pairs.
 *   - a handle is not re-entrant; distinct handles may be used from distinct threads.
 */
#ifndef ORCA_B200_H_
#define ORCA_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ORCA_B200_ABI_VERSION 2

typedef enum OrcaStatus {
  ORCA_OK = 0,
  ORCA_ERR_INVALID = -1,     /* bad argument (-> ValueError in the Python layer) */
  ORCA_ERR_CUDA = -2,        /* CUDA runtime failure (-> RuntimeError) */
  ORCA_ERR_UNSUPPORTED = -3, /* shape outside what the kernels cover */
  ORCA_ERR_STATE = -4        /* call order violated (e.g. step before create) */
} OrcaStatus;

/* Simulator-wide agent parameters: the 7 scalars of
 * rvo2.PyRVOSimulator(timeStep, neighborDist, maxNeighbors, timeHorizon,
 * timeHorizonObst, radius, maxSpeed)  -- ALAN_true.py:22-28, collision_avoidence_env.py:62-68,
 * and of addAgent(...) -- collision_avoidence_env.py:126-133, ALAN_true.py:461-468.
 * They are every agent's parameters unless orca_set_agent_params gives agents their own. */
typedef struct OrcaParams {
  float time_step;
  float neighbor_dist;
  int32_t max_neighbors;
  float time_horizon;
  float time_horizon_obst;
  float radius;
  float max_speed;
} OrcaParams;

typedef struct OrcaSim OrcaSim; /* opaque; one per (device, batch shape) */

/* How the preferred velocity of a step is produced. */
typedef enum OrcaPolicy {
  ORCA_POLICY_EXTERNAL = 0, /* pref_dev given: plain setAgentPrefVelocity + doStep */
  ORCA_POLICY_GOAL = 1,     /* unit vector to goal: orca_step, ALAN_true.py:631-633,483-495;
                               collision_avoidence_env.py:447-449,151-162 */
  ORCA_POLICY_RL = 2,       /* goal direction rotated by action angle: env.step :371-383 */
  ORCA_POLICY_ALAN = 3      /* softmax bandit over an action table: online_step ALAN_true.py:576-598 */
} OrcaPolicy;

/* Which done test runs after the integration. */
typedef enum OrcaDoneMode {
  ORCA_DONE_NONE = 0,
  ORCA_DONE_GOAL_RADIUS = 1, /* |pos - goal| < 2*radius -> record time, goal <- goal2 : ALAN_true.py:547-566 */
  ORCA_DONE_X_BELOW = 2,     /* pos.x < x_threshold    -> goal <- goal2              : collision_avoidence_env.py:352-365 */
  /* GOAL_RADIUS in the order of run_sim(mode=0) (ALAN_true.py:116-120,631-633): orca_step computes the
   * preferred velocity of the NEXT doStep before done_test swaps the target, so the step right after an
   * arrival still aims at the old goal.  agent_done holds 2 for that one step ("swap pending"), then 1. */
  ORCA_DONE_GOAL_RADIUS_DEFERRED = 3
} OrcaDoneMode;

/* Slots of the device statistics vector (uint64 counters / float64 sums, 8 bytes each). */
enum {
  ORCA_STAT_AGENT_STEPS = 0,  /* u64: agents advanced by one step */
  ORCA_STAT_FINISHED = 1,     /* u64: agents that reached their goal */
  ORCA_STAT_COLLISIONS = 2,   /* u64: (agent, neighbor) pairs with distSq <= (2r)^2 (RVO2's collision branch) */
  ORCA_STAT_LP3_CALLS = 3,    /* u64: agents whose LP2 was infeasible */
  ORCA_STAT_OVERFLOW = 4,     /* u64: agent-steps that exceeded even the uncapped path's capacity (64 obstacle edges /
                               * lines per agent): a constraint was dropped; impossible for worlds of <= 64 vertices */
  ORCA_STAT_SUM_ARRIVAL = 5,  /* f64: sum of arrival times  (TTime, ALAN_true.py:125-131) */
  ORCA_STAT_SUM_ARRIVAL2 = 6, /* f64: sum of squared arrival times */
  ORCA_STAT_SUM_REWARD = 7,   /* f64: sum of the per-agent rewards (RL and ALAN policies) */
  ORCA_STAT_COUNT = 8
};

/* Arguments of one fused environment step.  Unused pointers are NULL. */
typedef struct OrcaEnvStepArgs {
  uint32_t struct_size; /* = sizeof(OrcaEnvStepArgs), ABI guard */
  int32_t policy;       /* OrcaPolicy */
  int32_t done_mode;    /* OrcaDoneMode */
  int32_t _pad0;

  /* simulator state, in/out: getAgentPosition/getAgentVelocity/setAgentPosition
   * (collision_avoidence_env.py:157,237,394,479; ALAN_true.py:490,553,613) */
  float* pos_dev; /* [E*N][2] */
  float* vel_dev; /* [E*N][2] */

  const float* pref_dev; /* [E*N][2] EXTERNAL policy: setAgentPrefVelocity (env :383, ALAN :598) */
  float* goal_dev;       /* [E*N][2] in/out; world["targets_pos"] (env :94, ALAN :314-317) */
  const float* goal2_dev; /* [E*N][2] secondary goal taken on arrival (ALAN :561-562, env :361) */

  const float* action_theta_dev; /* [E*N] RL policy: action['agent_i'] (env :373) */
  float rl_reward_scale;         /* 0.3 at env :396 */
  float done_x_threshold;        /* 2.0 at env :359 */

  /* ALAN bandit (ALAN_true.py:569-628) */
  float* alan_weights_dev;          /* [E*N][A] in/out: world["action_weights"] */
  const float* alan_actions_dev;    /* [A][2]  unit vectors: online_actions (ALAN :31-38, *.act files) */
  uint8_t* alan_action_out_dev;     /* [E*N] chosen action id, optional */
  const float* alan_uniform_in_dev; /* [E*N] optional: externally supplied U[0,1) draws (parity tests) */
  int32_t alan_num_actions;         /* A <= 16 (row length of alan_weights_dev; max over envs) */
  int32_t alan_window_steps;        /* steps between global weight resets: 121 for dt=1/60, window 2 s (SURVEY Q7) */
  float alan_gamma;                 /* 0.6 (ALAN :47) */
  float alan_temp;                  /* 0.2 (ALAN :49) */
  uint64_t rng_seed;                /* Philox key; counter = (global agent id, env step) */
  /* per-env action sets (batched action-space search, Train_ALAN_action_space.py:55-67): when
   * alan_actions_env_stride > 0, env e reads its table at alan_actions_dev + e*stride*2 floats and
   * uses alan_num_actions_env_dev[e] (<= alan_num_actions) of its entries */
  const int32_t* alan_num_actions_env_dev; /* [E] or NULL */
  int32_t alan_actions_env_stride;         /* actions per env slot, 0 = one shared table */
  int32_t _pad1;

  /* per-step outputs */
  float* reward_dev;         /* [E*N] optional */
  uint8_t* agent_done_dev;   /* [E*N] in/out, required when done_mode != NONE */
  float* arrival_time_dev;   /* [E*N] in/out optional: agents_time (ALAN :559) */
  int32_t* env_step_dev;     /* [E] in/out step counter (step_count, ALAN :117, env :408).  REQUIRED with
                              * ORCA_POLICY_ALAN (Philox counter, weight-window reset) and whenever
                              * arrival_time_dev is given (arrival time = step * dt): ORCA_ERR_INVALID otherwise */
  int32_t* env_done_cnt_dev; /* [E] in/out number of done agents; env done <=> == N */

  /* neighbor lists of THIS step (pre-update positions, SURVEY Q3), optional:
   * getAgentNumAgentNeighbors/getAgentAgentNeighbor, ...ObstacleNeighbor (env :246-252,283-289,305-312) */
  int32_t* nbr_idx_dev;      /* [E*N][max_neighbors] env-local agent ids, ascending distance */
  int32_t* nbr_cnt_dev;      /* [E*N] */
  int32_t* obst_nbr_idx_dev; /* [E*N][ORCA_MAX_OBST_NEIGHBORS] obstacle vertex ids */
  int32_t* obst_nbr_cnt_dev; /* [E*N] */

  uint64_t* stats_dev; /* [ORCA_STAT_COUNT] accumulated, optional */
} OrcaEnvStepArgs;

#define ORCA_MAX_OBST_NEIGHBORS 16 /* width of the obstacle neighbor-list OUTPUT (the 16 nearest edges) */
#define ORCA_MAX_OBST_LINES 6      /* obstacle ORCA lines of the fast path; agents with more (or with more than 16
                                    * obstacle neighbors) are redone by the uncapped path (64 of each) -- RVO2 has
                                    * no cap (insertObstacleNeighbor), and neither has the step */
#define ORCA_MAX_ACTIONS 16

/* ---- lifecycle ---------------------------------------------------------------- */
int orca_abi_version(void);
const char* orca_last_error(void);

/* Replaces `rvo2.PyRVOSimulator(...)` + the N `addAgent` calls of one world, for a
 * batch of `num_envs` independent worlds of `agents_per_env` agents each
 * (collision_avoidence_env.py:62-68,126-133; ALAN_true.py:22-28,461-468). */
int orca_create(const OrcaParams* params, int device, int num_envs, int agents_per_env, OrcaSim** out);
int orca_destroy(OrcaSim* sim);
int orca_get_params(const OrcaSim* sim, OrcaParams* out, int* num_envs, int* agents_per_env);

/* Per-agent ORCA parameters: RVO2's addAgent(pos, neighborDist, maxNeighbors, timeHorizon,
 * timeHorizonObst, radius, maxSpeed, velocity) and its setAgent{NeighborDist,MaxNeighbors,
 * TimeHorizon,TimeHorizonObst,Radius,MaxSpeed}.  HOST arrays of E*N entries, env-major.
 * A NULL array means every agent takes the handle's OrcaParams value.  All six NULL returns the
 * handle to uniform parameters.  The values are copied; the call synchronises (a setup call,
 * like orca_set_obstacles).  ORCA_ERR_INVALID unless every value is finite, time_horizon and
 * time_horizon_obst > 0, neighbor_dist, radius, max_speed >= 0 and 0 <= max_neighbors <=
 * OrcaParams.max_neighbors (which stays the row width of the neighbor-list outputs).
 * Handle-wide whatever the table holds: the time step, the 2 * radius of the done test and
 * orca_observe (its neighbor octagons use OrcaParams.radius, its rays OrcaParams.neighbor_dist). */
int orca_set_agent_params(OrcaSim* sim, const float* neighbor_dist, const int32_t* max_neighbors,
                          const float* time_horizon, const float* time_horizon_obst,
                          const float* radius, const float* max_speed);

/* ---- obstacles -------------------------------------------------------------------
 * Replaces addObstacle(...) x P + processObstacles() (collision_avoidence_env.py:118-123,145;
 * ALAN_true.py:196-210,476).  `xy` holds all polygon vertices back to back, `poly_sizes[p]`
 * vertices each.  With `polys_per_env == NULL` the world is shared by every env; otherwise
 * env e owns the next `polys_per_env[e]` polygons.  The obstacle BSP is built on the host
 * exactly once (it may split edges and append vertices, SURVEY A.3) and uploaded. */
int orca_set_obstacles(OrcaSim* sim, const float* xy, const int32_t* poly_sizes, int num_polys,
                       const int32_t* polys_per_env);
/* Post-processing vertex table of env `env` (0 when shared):
 * getObstacleVertex / getNextObstacleVertexNo (env :148,208,307-311; ALAN :479,530). */
int orca_obstacle_vertex_count(const OrcaSim* sim, int env);
int orca_get_obstacle_vertices(const OrcaSim* sim, int env, float* xy_out, int32_t* next_out, int32_t* prev_out,
                               int32_t* convex_out);

/* ---- line of sight and roadmap navigation -------------------------------------------
 * Replaces RVO2's RVOSimulator::queryVisibility(point1, point2, radius): can a disc of `radius` move
 * along the segment q1 -> q2 without crossing an obstacle edge?  The obstacle BSP of each query's
 * env answers, bit for bit as RVO2's recursion does.  q1_dev, q2_dev: [E][Q][2]; radius_dev: [E][Q],
 * or NULL for the scalar `radius` (finite, >= 0) everywhere.  visible_dev: [E][Q] bytes of 0 / 1.
 * Every query is visible when no obstacles are set.  Asynchronous on `stream`. */
int orca_query_visibility(OrcaSim* sim, const float* q1_dev, const float* q2_dev, const float* radius_dev,
                          float radius, int queries_per_env, uint8_t* visible_dev, void* stream);
/* Replaces the roadmap of RVO2's obstacle example (examples/Roadmap.cpp buildRoadmap): HOST `xy` of
 * [W][R][2] roadmap vertices, W = 1 (shared) or W = E when `per_env` is set; the first `num_goals`
 * vertices of each world are its goals.  Edge u -> v exists when queryVisibility(p_u, p_v, radius)
 * (not symmetric in general); distToGoal[g][v] is Dijkstra's over those edges, weights |p_v - p_u|,
 * 9e9f when unreachable.  Edges and distances are computed on the device for every obstacle world
 * (per env when the obstacles or the roadmap are) and recomputed by orca_set_obstacles.  A setup
 * call: it synchronises.  num_vertices == 0 removes the roadmap.  ORCA_ERR_UNSUPPORTED unless
 * R <= 512 and 1 <= num_goals <= R; ORCA_ERR_INVALID for non-finite vertices or a radius that is
 * not finite and >= 0. */
int orca_set_roadmap(OrcaSim* sim, const float* xy, int num_vertices, int num_goals, int per_env, float radius);
/* The roadmap tables of env `env`: adjacency as R rows of ceil(R / 32) words (row u bit v = edge
 * u -> v), distances as [G][R].  Either output may be NULL.  Synchronises.  ORCA_ERR_STATE without a
 * roadmap. */
int orca_get_roadmap(const OrcaSim* sim, int env, uint32_t* adjacency_out, float* dist_out);
/* Replaces Roadmap.cpp setPreferredVelocities (without its random perturbation) for every agent:
 * among the roadmap vertices j with |p_j - pos| + distToGoal[goal][j] < 9e9f that are visible from
 * the agent's position for its radius (the per-agent radius when orca_set_agent_params set one), the
 * lowest index of smallest cost; pref = normalize(p_j - pos), or normalize(p_goal - pos) when the agent
 * stands on a vertex other than its goal, (0, 0) on its goal or when no vertex qualifies.
 * pos_dev [E*N][2], goal_vertex_dev [E*N] (goal ids in [0, num_goals); any other id gives pref (0, 0)
 * and vertex -1), pref_dev [E*N][2] out, vertex_out_dev [E*N] out or NULL.  ORCA_ERR_STATE without a
 * roadmap.  Asynchronous on `stream`. */
int orca_roadmap_pref_velocity(OrcaSim* sim, const float* pos_dev, const int32_t* goal_vertex_dev,
                               float* pref_dev, int32_t* vertex_out_dev, void* stream);

/* ---- stepping ---------------------------------------------------------------------
 * orca_step: setAgentPrefVelocity x N + doStep (env :383-385, ALAN :598-601), batched. */
int orca_step(OrcaSim* sim, float* pos_dev, float* vel_dev, const float* pref_dev, void* stream);
/* Fused environment step: policy + doStep + reward + done test + bandit update. */
int orca_env_step(OrcaSim* sim, const OrcaEnvStepArgs* args, void* stream);
/* `steps` fused environment steps back to back on `stream` without returning to the host in
 * between (run_sim's inner loop, ALAN_true.py:113-121): the launches are issued from C, which removes the
 * per-step Python / ctypes cost (the launches themselves are asynchronous either way).  Same arguments as
 * orca_env_step.  Worlds whose env_done_cnt had reached agents_per_env when a step began keep being
 * stepped, but no longer count into stats_dev (agent steps, collisions, LP3 calls, reward sum). */
int orca_env_step_many(OrcaSim* sim, const OrcaEnvStepArgs* args, int steps, void* stream);
/* Parity hook: neighbor search only.  nbr_distsq_dev optional. */
int orca_neighbors(OrcaSim* sim, const float* pos_dev, int32_t* nbr_idx_dev, float* nbr_distsq_dev,
                   int32_t* nbr_cnt_dev, int32_t* obst_nbr_idx_dev, int32_t* obst_nbr_cnt_dev, void* stream);

/* The ORCA half-planes every agent would solve in a step from (pos, vel): RVO2's
 * getAgentNumORCALines / getAgentORCALine.  Obstacle lines first (RVO2's order, covered edges
 * skipped), then one line per agent neighbor in ascending (distSq, id); each line is (point.x, point.y,
 * direction.x, direction.y), bit for bit what the next orca_step / orca_env_step from this state
 * solves (the preferred velocity plays no part).  lines_dev [E*N][max_lines][4]; rows past max_lines
 * are not written, counts are always complete.  line_cnt_dev [E*N] (-1: beyond the uncapped capacity,
 * ORCA_SLOW_MAX_OBST obstacle lines), obst_line_cnt_dev [E*N] or NULL.  max_lines = 0 gives counts
 * only.  Writes nothing a step reads (no neighbor-search hint, step counter, statistic or step scratch):
 * on worlds of more than 256 agents it sorts (pos, vel) into a grid scratch of its own (allocated at the
 * first such call, about 36 B per agent plus the cells).  Asynchronous on `stream`: order it after
 * whatever writes pos_dev / vel_dev, and order two orca_agent_lines calls on one handle (they share that
 * scratch). */
int orca_agent_lines(OrcaSim* sim, const float* pos_dev, const float* vel_dev, int max_lines, float* lines_dev,
                     int32_t* line_cnt_dev, int32_t* obst_line_cnt_dev, void* stream);

/* Laser-scan observation of every agent: Collision_Avoidance_Env._get_obs + utils.comp_laser
 * (collision_avoidence_env.py:231-350 ; utils.py:5-113).  `laser_num` rays of length
 * neighbor_dist per agent, neighbors approximated by `circle_approx_num`-gons of the agent
 * radius; neighbor lists as written by orca_env_step / orca_neighbors.  obs_dev is
 * [E*N][laser_num][4] = (hit.x, hit.y, vel.x, vel.y) in the goal-aligned frame. */
int orca_observe(OrcaSim* sim, const float* pos_dev, const float* vel_dev, const float* goal_dev,
                 const int32_t* nbr_idx_dev, const int32_t* nbr_cnt_dev, const int32_t* obst_nbr_idx_dev,
                 const int32_t* obst_nbr_cnt_dev, int laser_num, int circle_approx_num, float* obs_dev, void* stream);

/* Weights of the shared policy network (run_rllib.py:35-52, CustomModel1: fc1 64->64 ReLU,
 * fc2 64->64 ReLU, fc_out 64->out_dim linear).  Matrices are [in][out] row-major (the layout of
 * slim.fully_connected's `weights`), float32, device pointers; w1_dev and w2_dev 16-byte aligned. */
typedef struct OrcaMlpWeights {
  uint32_t struct_size; /* = sizeof(OrcaMlpWeights) */
  int32_t in_dim;       /* 64: laser_num(16) * 4 */
  int32_t hidden_dim;   /* 64 */
  int32_t out_dim;      /* 1..8 (PPO on the env's Box(1) action space: mean, log-std) */
  const float* w1_dev;
  const float* b1_dev;
  const float* w2_dev;
  const float* b2_dev;
  const float* w3_dev;
  const float* b3_dev;
} OrcaMlpWeights;

/* Forward pass of that network for `rows` observation rows ([rows][64], e.g. the buffer
 * orca_observe wrote for E*N agents): out_dev[rows][out_dim].  Replaces the per-env TensorFlow
 * evaluation inside RLlib's rollout workers (run_rllib.py:35-52,96-112) so that
 * observe -> policy -> orca_env_step stays on the device.  Asynchronous on `stream`.
 *   orca_policy_mlp       tcgen05 tensor cores, TF32 products split 3x (hi.hi + hi.lo + lo.hi),
 *                         FP32 accumulation in TMEM: FP32-level accuracy, bound by reading obs once;
 *   orca_policy_mlp_fp32  the same network on the FP32 pipes (fused multiply-adds), kept as the
 *                         reference point for the tensor-core kernel. */
int orca_policy_mlp(OrcaSim* sim, const float* obs_dev, int64_t rows, const OrcaMlpWeights* weights, float* out_dev,
                    void* stream);
int orca_policy_mlp_fp32(OrcaSim* sim, const float* obs_dev, int64_t rows, const OrcaMlpWeights* weights, float* out_dev,
                         void* stream);

/* Host-buffer variant of orca_step (the e2e path: what a PyRVOSimulator-style caller
 * pays): takes pref / goal (and, if `upload_state`, pos/vel) from host buffers, steps `steps`
 * times with the given policy (EXTERNAL or GOAL), leaves the new pos/vel in the host buffers,
 * synchronises.  Two routes, same results:
 *   - pinned (cudaHostAlloc / cudaHostRegister, i.e. mapped) buffers: the step kernel reads the
 *     input from and writes the new state into the caller's buffers itself, over PCIe, while it
 *     computes -- one launch, no staging copies;
 *   - pageable buffers, or the uniform-grid pipeline: staged copies, the batch cut into env
 *     chunks on separate streams (upload | step | download overlapped), replayed from a CUDA
 *     graph while the arguments stay the same. */
int orca_step_host(OrcaSim* sim, float* pos_host, float* vel_host, const float* pref_or_goal_host, int policy,
                   int upload_state, int steps);
/* The same with the per-step host traffic under the caller's control:
 *   ORCA_HOST_UPLOAD_STATE   take pos / vel from the host buffers first (= upload_state above)
 *   ORCA_HOST_AUX_UNCHANGED  the goal / pref buffer holds what it held at the previous call with the same
 *                            pointer: its device copy is reused, nothing is read from the host.  Goals are
 *                            static under ORCA_POLICY_GOAL, and the reference's orca_step loop
 *                            (ALAN_true.py:631-633) writes no per-step input either.
 * vel_host may be NULL: only the positions are written back -- all that loop reads per step
 * (getAgentPosition in update_pref_vel / done_test, ALAN_true.py:490,553).  Returns ORCA_ERR_STATE when the
 * state was never uploaded. */
#define ORCA_HOST_UPLOAD_STATE 1
#define ORCA_HOST_AUX_UNCHANGED 2
int orca_step_host_ex(OrcaSim* sim, float* pos_host, float* vel_host, const float* pref_or_goal_host, int policy,
                      int flags, int steps);

/* Number of kernels launched through this handle so far (bench.py's gpu_launches). */
int64_t orca_launch_count(const OrcaSim* sim);

#ifdef __cplusplus
}
#endif
#endif /* ORCA_B200_H_ */
