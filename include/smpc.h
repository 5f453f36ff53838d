/*
 * smpc.h — C-ABI of libsmpc.so, the B200-native batched social-MPC solver.
 *
 * Drop-in boundary for the hot path of PIC4SeR/nav2_social_mpc_controller:
 *   bool Optimizer::optimize(...)            include/nav2_social_mpc_controller/optimizer.hpp:167-170
 *   void Optimizer::initialize(params)       include/nav2_social_mpc_controller/optimizer.hpp:152
 *   struct OptimizerParams                   include/nav2_social_mpc_controller/optimizer.hpp:59-101
 *   ceres::Solve(options_, &problem, &summary)   src/optimizer.cpp:381
 *
 * Everything here is POD: plain pointers, sizes and doubles. No exceptions, no
 * torch / STL types cross this boundary. All floating point is FP64 except
 * the costmap (u8) and the obstacle-distance grid (f32 + u32).
 *
 * Memory layouts (B = problems, S = optimised steps N_v, NB = parameter blocks,
 * A = agent columns per step, row-major, last index fastest):
 *   pose0      [B][3]            x, y, yaw of the first seed pose (yaw already tf2 round-tripped, SURVEY Q14)
 *   u0         [B][NB][2]        initial (v, w) of block b = seed velocity at TIME INDEX b (SURVEY Q1)
 *   path_xy    [B][2][S+1]       seed positions: row 0 = x, row 1 = y; step index fastest
 *   goal_yaw   [B]               yaw of the last seed pose (src/optimizer.cpp:298)
 *   agents     [B][A][6][S+1]    projected people: component c in (x, y, yaw, t, lv, av), step index fastest;
 *                                t == -1 marks an invalid (padded) agent (src/optimizer.cpp:468-474).
 *                                The reference shape AgentsTrajectories[step][agent][6]
 *                                (tools/type_definitions.hpp:6-9) is transposed so the S+1 steps a warp
 *                                reads are contiguous.
 *   has_people [B] u8            people.people.size() != 0 (src/optimizer.cpp:263)
 *   costmaps   [M][size_y][size_x] u8, Nav2 costmap bytes, row = y (src/optimizer.cpp:167-168)
 *   costmap_origin [M][2]        world origin of each map
 *   costmap_index  [B] i32       which of the M maps problem b reads (NULL: map b % M)
 */
#ifndef SMPC_H_
#define SMPC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMPC_ABI_VERSION 4
#define SMPC_MAX_BLOCKS 18 /* control_horizon 18 with parameter_block_length 1: the "36x36 class" */

/* Return codes of every entry point. Per-problem solver outcomes are NOT call
 * errors: they are reported in smpc_result.termination[] (mirrors
 * `return false` of Optimizer::optimize, src/optimizer.cpp:384-388). */
enum smpc_status {
  SMPC_OK = 0,
  SMPC_ERR_ARGUMENT = -1,
  SMPC_ERR_CUDA = -2,
  SMPC_ERR_UNSUPPORTED = -3,
  SMPC_ERR_IO = -4,
  SMPC_ERR_PARAM = -5 /* e.g. invalid linear_solver_type, src/optimizer.cpp:31-45 */
};

/* ceres::TerminationType as observed through Solver::Summary, plus the reason. */
enum smpc_termination {
  SMPC_CONVERGENCE_GRADIENT = 0,  /* gradient_max_norm <= gradient_tolerance */
  SMPC_CONVERGENCE_PARAMETER = 1, /* step_norm <= param_tol*(x_norm+param_tol) */
  SMPC_CONVERGENCE_FUNCTION = 2,  /* |cost_change| <= fn_tol*cost */
  SMPC_CONVERGENCE_RADIUS = 3,    /* trust region radius <= 1e-32 */
  SMPC_NO_CONVERGENCE = 4,        /* max_num_iterations reached */
  SMPC_FAILURE_INVALID_STEPS = 5, /* 5 consecutive invalid steps */
  SMPC_FAILURE_EVALUATION = 6     /* non-finite residual/Jacobian at an accepted point */
};

/* Mirrors OptimizerParams (optimizer.hpp:59-101) and the defaults declared in
 * OptimizerParams::get (src/optimizer.cpp:26-84). */
typedef struct smpc_params {
  char linear_solver_type[32]; /* validated against the 5-entry map, optimizer.hpp:71-77 */
  double param_tol;
  double fn_tol;
  double gradient_tol;
  int max_iterations;
  int debug;
  int control_horizon;
  int parameter_block_length;
  int discretization; /* read from yaml, never used (SURVEY §5) */
  double distance_w;
  double socialwork_w;
  double velocity_w;
  double angle_w;
  double agent_angle_w;
  double proxemics_w;
  double velocity_feasibility_w;
  double obstacle_w;
  double goal_align_w;
  float current_path_w;
  float current_cmds_w;
  float max_time;  /* trajectorizer.max_time */
  float time_step; /* trajectorizer.time_step (held as float in the reference, SURVEY Q15) */
  /* trajectorizer.* and top-level plugin parameters (path_trajectorizer.cpp:52-70, social_mpc_controller.cpp:59-65) */
  int omnidirectional;
  double traj_desired_linear_vel;
  double lookahead_dist;
  double max_angular_vel;
  double transform_tolerance;
  char base_frame[64];
  double desired_linear_vel;
  double fov_angle;
  /* Solver-behaviour switches that are not reference yaml (documented in DESIGN.md):
   * ceres_compat 200 = Ceres 2.0.0 loop (Ubuntu 22.04 / Humble), 220 = Ceres >= 2.1
   * (parameter / function tolerance only tested after a first successful step). */
  int ceres_compat;
  /* Deterministic stand-in for Solver::Options::max_solver_time_in_seconds (src/optimizer.cpp:131; Ceres tests it in
   * FinalizeIterationAndCheckIfMinimizerCanContinue, before the iteration cap): a solve that has spent this many
   * evaluations stops with NO_CONVERGENCE at its next iteration boundary. 0 = off (the wall clock of the reference is
   * not reproducible; parity runs keep it off). */
  int max_evaluations;
  /* Extension, not reference behaviour: 1 = the solve optimises omnidirectional (vx, vy, w) blocks (the reference's
   * update_state.hpp:46-61 is unicycle-only; only its trajectorizer has an omni branch). 0 = unicycle (v, w). */
  int omni_solve;
} smpc_params;

/* One batch of independent MPC problems, post-projection: exactly the arrays
 * the Ceres problem of src/optimizer.cpp:241-379 is assembled from. Pointers
 * are host pointers for smpc_solve_batch and device pointers for
 * smpc_solve_batch_device. */
typedef struct smpc_batch {
  int n_problems; /* B */
  int n_steps;    /* S = N_v = P_poses - 1: the longest horizon of the batch (see n_steps_each) and the array stride */
  int n_agents;   /* A: 3 in the reference (src/optimizer.cpp:468-479); any A >= 0 here */
  int n_costmaps; /* M */
  int size_x;
  int size_y;
  double resolution;
  double dt; /* (double)(float)time_step, SURVEY Q15 */
  const double* pose0;
  const double* u0;
  const double* path_xy;
  const double* goal_yaw;
  const double* agents;       /* may be NULL when n_agents == 0 */
  const uint8_t* has_people;  /* may be NULL: no problem has people. Ignored (treated as all zero) when n_agents == 0 or
                                 agents == NULL: the people critics have no agent columns to act on */
  const uint8_t* costmaps;
  const double* costmap_origin;
  const int32_t* costmap_index; /* may be NULL */
  /* Per-problem horizon S_b <= n_steps ([B] i32, may be NULL: every problem has n_steps steps). The trajectorizer
   * stops early near the goal (src/path_trajectorizer.cpp:152) and the optimizer sizes the problem from what it got
   * (src/optimizer.cpp:248-249), so the robots of a fleet have different S, ch, bl and block counts. Array strides stay
   * those of n_steps (rows are padded); problem b reads steps 0..S_b, uses the first ceil(ch_b/bl_b) blocks of its
   * u0 / u rows and does not write the rest of its output rows (smpc_solve_batch returns them zero-filled,
   * smpc_solve_batch_device leaves the caller's memory untouched). */
  const int32_t* n_steps_each;
  /* Scenario sharing (multi-start: many start points u0 of ONE scene). When scenario_index != NULL the arrays pose0,
   * path_xy, goal_yaw, agents, has_people, n_steps_each and costmap_index have n_scenarios rows instead of n_problems
   * and problem b reads row scenario_index[b] (costmap of row r without an index: r % M); u0 and every output stay per
   * problem. The scene of 1024 starts then crosses the bus once and stays in L2 instead of 1024 times. */
  const int32_t* scenario_index; /* [B] in [0, n_scenarios), or NULL */
  int n_scenarios;
} smpc_batch;

/* Per-problem outputs. Any pointer may be NULL (that output is skipped).
 *   u            [B][NB][2]   optimised block values (the Ceres parameter blocks after Solve)
 *   cmds         [B][S+1][2]  per-step (v, w) after hold-last fill and block expansion, src/optimizer.cpp:390-419
 *   path         [B][S+1][3]  Euler-rebuilt poses x, y, yaw, pose0 excluded, src/optimizer.cpp:420-446
 *   cost_initial [B]          Summary::initial_cost
 *   cost_final   [B]          Summary::final_cost (min over iteration costs)
 *   iterations   [B]          index of the last recorded TR iteration
 *   termination  [B]          enum smpc_termination
 *   usable       [B]          Summary::IsSolutionUsable(); 0 <=> optimize() would return false
 *   n_evals      [B][2]       {evaluations that built J^T J, evaluations that stopped at cost + J^T r (line-search
 *                             samples that failed the Armijo test)} (roofline numerator)
 */
typedef struct smpc_result {
  double* u;
  double* cmds;
  double* path;
  double* cost_initial;
  double* cost_final;
  int32_t* iterations;
  int32_t* termination;
  uint8_t* usable;
  int32_t* n_evals;
  /* Optional per-evaluation solver trace (diagnostics: tools/flip_log.py): trace [B][trace_rows][8] =
   * iteration, phase (1 init / 2 line-search sample / 3 full step), step size t, cost of the differentiated
   * evaluation, cost of the plain evaluation, aux (rejected sample: Armijo margin; candidate: relative decrease),
   * code (bit 0 Armijo ok, 1 became the candidate, 2 accepted, 3 terminated, bits 4.. termination), radius.
   * Rows beyond trace_rows are dropped; unused rows are left untouched. NULL = off. */
  double* trace;
  int trace_rows;
} smpc_result;

/* Normal-equation snapshot of one evaluation (first-slice / test entry):
 *   cost [B], grad [B][P], hess [B][P*(P+1)/2] (row-major lower triangle), P = 2*NB. */
typedef struct smpc_eval_out {
  double* cost; /* 1/2 sum r^2 as a DIFFERENTIATED evaluation (Jets) of the reference computes it */
  double* grad;
  double* hess;
  uint8_t* ok; /* 0 when a residual or Jacobian entry was non-finite */
  /* the same sum as a cost-only (double) evaluation computes it; differs from `cost` only under ceres_compat < 210
   * with people (ProxemicsCost evaluates differently under Ceres 2.0.0 Jets, DESIGN.md). May be NULL. */
  double* cost_plain;
} smpc_eval_out;

typedef struct smpc_handle smpc_handle;

/* ---- parameters ------------------------------------------------------- */
/* Fill with the defaults of OptimizerParams::get (src/optimizer.cpp:26-84). */
void smpc_params_default(smpc_params* p);
/* Parse `<plugin_name>:` subtree (e.g. "FollowPath") of a Nav2 params yaml:
 * trajectorizer.*, optimizer.*, optimizer.weights.* (src/optimizer.cpp:16-85). */
int smpc_params_from_yaml(const char* yaml_path, const char* plugin_name, smpc_params* p);
/* Derived sizes of the assembled problem (src/optimizer.cpp:248-249):
 * ch = min(control_horizon, S), bl = min(block_length, ch), NB = ceil(ch/bl),
 * n_bounded = ch/bl. Any out pointer may be NULL. */
int smpc_problem_dims(const smpc_params* p, int n_steps, int* ch, int* bl, int* n_blocks, int* n_bounded);

/* ---- handle ------------------------------------------------------------ */
/* One handle per caller thread and per GPU; calls on a handle are serialised.
 * Replaces Optimizer::initialize (src/optimizer.cpp:98-132). */
int smpc_create(const smpc_params* p, int device, smpc_handle** out);
void smpc_destroy(smpc_handle* h);
const char* smpc_last_error(void);
int smpc_abi_version(void);

/* ---- level-1 solve: replaces ceres::Solve at src/optimizer.cpp:381 ------ */
/* Host buffers in, host buffers out (H2D, kernels, D2H inside the call; returns when the results are in `out`). Copies
 * and solves are pipelined over two streams (batches with people: chunks of problems; people-free batches: per-problem
 * costmaps / large per-problem arrays stream into the running solve) when the caller's buffers are page-locked; pageable
 * buffers work too, without the overlap. Results do not depend on it. */
int smpc_solve_batch(smpc_handle* h, const smpc_batch* in, smpc_result* out);
/* Device buffers in/out; asynchronous on `stream` (a cudaStream_t, NULL = the handle's own stream). A handle owns ONE set
 * of work-queue counters and scratch buffers: a new solve may be enqueued only on the stream of the previous one, or
 * after that one has finished (use one handle per stream to overlap solves). */
int smpc_solve_batch_device(smpc_handle* h, const smpc_batch* in, smpc_result* out, void* stream);
/* Evaluate cost, J^T r and J^T J at given block values x [B][NB][2] (device pointers). */
int smpc_eval_batch_device(smpc_handle* h, const smpc_batch* in, const double* x, smpc_eval_out* out, void* stream);
/* Host-buffer convenience wrapper of the above (tests). */
int smpc_eval_batch(smpc_handle* h, const smpc_batch* in, const double* x, smpc_eval_out* out);

/* ---- level-2 entry: mirrors bool Optimizer::optimize(...) (optimizer.hpp:167-170) for ONE robot ------------------
 * One-robot fleet tick (smpc_optimize_batch with B = 1, 3 people columns): every stage runs on the GPU in the
 * reference's arithmetic order — people_to_status src/optimizer.cpp:454-482, format_to_optimize :484-551 with the
 * handle's device-resident previous path / cmds standing in for the TrajectoryMemory singleton
 * (trajectory_memory.hpp), project_people :554-671 + sfm.hpp, computeObstacle :673-728, the solve and the post-solve
 * expansion (level-1 kernel), the memory update :448-449. */
typedef struct smpc_obstacle_distance { /* obstacle_distance_msgs::msg::ObstacleDistance */
  uint32_t width;
  uint32_t height;
  float resolution;
  double origin_x;
  double origin_y;
  const float* distances;  /* [height*width] (unused by the reference beyond the emptiness check) */
  const uint32_t* indexes; /* [height*width] index of the nearest obstacle cell */
} smpc_obstacle_distance;

typedef struct smpc_optimize_io {
  /* in/out: seed path from the trajectorizer -> optimised path. poses [capacity][3] = x, y, yaw (tf2::getYaw of the
   * pose quaternion); n_poses is updated. cmds [capacity][2] = linear.x, angular.z; n_cmds is updated. */
  int capacity;
  int n_poses;
  double* poses;
  int n_cmds;
  double* cmds;
  /* in */
  int n_people;
  const double* people; /* [n_people][5] position.x, position.y, velocity.x, velocity.y, velocity.z (people_msgs) */
  double speed_v;       /* speed.linear.x */
  double speed_w;       /* speed.angular.z */
  float time_step;
  const uint8_t* costmap; /* Costmap2D::getCharMap() */
  int size_x;
  int size_y;
  double origin_x;
  double origin_y;
  double resolution;
  smpc_obstacle_distance od;
  /* out */
  int n_proj_steps;    /* P = number of poses optimised */
  double* people_proj; /* [capacity][3][6] AgentsTrajectories (may be NULL) */
  int optimized;       /* the bool optimize() returns */
  int termination;
  int iterations;
  double cost_initial;
  double cost_final;
} smpc_optimize_io;

/* Returns SMPC_OK when the call itself worked (io->optimized holds the reference's return value); the
 * std::runtime_error cases of computeObstacle (src/optimizer.cpp:676-713) map to SMPC_ERR_ARGUMENT.
 * Implemented as smpc_optimize_batch for one robot: every stage runs in the GPU kernels of the fleet tick. */
int smpc_optimize(smpc_handle* h, smpc_optimize_io* io);

/* ---- level-2 BATCH entry: bool Optimizer::optimize(...) for a fleet of robots, one call per controller tick ---------
 * Host buffers in and out; every stage is a kernel on the handle's stream: TrajectoryMemory seeding (:174-186),
 * people_to_status (:454-482), format_to_optimize (:484-551), project_people (:554-671 + sfm.hpp), the bounded TR-LM
 * solve with the post-solve expansion (:241-446) and the memory update (:448-449). Robots have their OWN horizon:
 * n_poses[b] is what the trajectorizer produced for robot b (it stops early near the goal,
 * src/path_trajectorizer.cpp:152) and the problem is sized from it (:248-249, :492-497). The warm-start memory
 * (previous path / cmds, one TrajectoryMemory per robot) and the costmaps / obstacle grids live on the device between
 * calls; no device allocation happens after the first tick of a fleet shape. smpc_reset_memory forgets the memory. */
typedef struct smpc_fleet_io {
  int n_robots;  /* B */
  int max_poses; /* row stride of poses / cmds / people_proj (>= every n_poses[b], e.g. trajectorizer max_steps + 1) */
  int n_agents;  /* A people columns per robot (the reference: 3; more than A people are truncated by the caller) */
  float time_step; /* <= 0: params.time_step */
  /* in */
  const int32_t* n_poses;  /* [B] seed poses per robot (cmds: n_poses - 1); < 2 -> optimized[b] = 0 (:158-162) */
  const double* people;    /* [B][A][5] position.x/y, velocity.x/y/z */
  const int32_t* n_people; /* [B] */
  const double* speed;     /* [B][2] linear.x, angular.z */
  const uint8_t* costmaps; /* [M][size_y][size_x] */
  const double* costmap_origin; /* [M][2] */
  const int32_t* costmap_index; /* [B] or NULL (robot b uses map b % M) */
  int n_costmaps, size_x, size_y;
  double resolution;
  const uint32_t* od_indexes; /* [Mo][od_height * od_width] nearest-obstacle cell index (ObstacleDistance.indexes) */
  const double* od_origin;    /* [Mo][2] */
  const int32_t* od_index;    /* [B] or NULL (robot b uses grid b % Mo) */
  int n_od_grids;
  uint32_t od_width, od_height;
  float od_resolution;
  /* Costmaps and obstacle grids are re-sent to the device only when maps_version differs from the previous call's
   * (Nav2 updates local costmaps far slower than the 20 Hz control loop); 0 = always re-send. */
  long long maps_version;
  /* in-out: seed -> result. A robot whose solve is not usable keeps its cmds and gets the cut + blended seed path
   * (what format_to_optimize leaves in `path`); inactive robots are untouched. */
  double* poses; /* [B][max_poses][3] x, y, yaw */
  double* cmds;  /* [B][max_poses][2] linear.x, angular.z */
  /* out */
  int32_t* n_out;     /* [B] poses / cmds valid after the call */
  uint8_t* optimized; /* [B] the bool Optimizer::optimize returns */
  int32_t* termination;    /* [B] may be NULL */
  int32_t* iterations;     /* [B] may be NULL */
  double* cost_initial;    /* [B] may be NULL */
  double* cost_final;      /* [B] may be NULL */
  int32_t* project_status; /* [B] may be NULL: 1 = a person left the obstacle grid (the reference throws
                              std::runtime_error there); such a robot is reported optimized = 0 and keeps its memory */
  double* people_proj;     /* [B][A][6][max_poses] may be NULL (level-1 agents layout) */
} smpc_fleet_io;
int smpc_optimize_batch(smpc_handle* h, smpc_fleet_io* io);
/* Forget the previous path / cmds (a fresh TrajectoryMemory). */
int smpc_reset_memory(smpc_handle* h);

/* ---- closed-loop episodes: N robots through their crowd scenes for T controller ticks, all on the GPU --------------
 * One tick of SocialMPCController::computeVelocityCommands per episode and tick, then the world moves:
 *   1. seed: the trajectorizer (smpc_trajectorize_batch_device) on the whole global path from the current pose, with
 *      max_steps = round(max_time / dt) and dt = time_step rounded to 6 decimals (the yaml double, SURVEY Q15). The
 *      reference's PathHandler prune and TF step are not modelled: the trajectorizer's own search picks the look-ahead
 *      point, so a path that comes back within lookahead_dist of itself is out of scope;
 *   2. people: constant velocity, x_k = x_0 + vx * (k * control_period) (same for y, velocities unchanged), then the
 *      FOV filter (smpc_fov_filter_batch_device) keeps n_agents columns; skipped when n_people == 0;
 *   3. optimize: the fleet tick's stages (as in smpc_optimize_batch) with n_poses = seed steps + 1 (0 once an episode is
 *      done), cmds = the seed's (linear.x, angular.z) and the measured speed; each call starts with fresh warm-start
 *      memory of its own and leaves that of smpc_optimize_batch / smpc_optimize untouched;
 *   4. command: row 0 of the fleet tick's cmds (the seed command when optimize() returned false);
 *   5. world step: unicycle forward Euler over control_period, yaw read back through setRPY / getYaw; the next measured
 *      speed is the command (ideal actuator). Metrics at time (k+1) * control_period against all people of the scene;
 *      the episode is done when the robot is within goal_tolerance of the last path pose.
 * The people do not react to the robot here (smpc_run_crowd_episodes below moves them under the social force model)
 * and the costmap does not roll with it; omnidirectional robots are not supported.
 * Host buffers in and out: one upload at the start, one download at the end, no host round trip per tick (the host
 * polls a 4-byte count of active episodes every 16 ticks and stops early when it reaches 0; results do not depend on
 * it). Returns SMPC_ERR_UNSUPPORTED for omni_solve or omnidirectional params, SMPC_ERR_ARGUMENT for invalid inputs;
 * both before anything is launched. */
typedef struct smpc_episode_io {
  int n_episodes;        /* B */
  int n_ticks;           /* T: controller ticks at most */
  int n_path;            /* N poses per global path (>= 2) */
  int n_people;          /* K: row stride of people (all people of a scene) */
  int n_agents;          /* A: people columns the optimizer keeps after the FOV filter (3 = the reference), 1..63 */
  double control_period; /* s per tick = 1 / controller_frequency (params yaml: 20 Hz -> 0.05) */
  double goal_tolerance; /* m, position-only goal check (Nav2 SimpleGoalChecker default 0.25); >= 0.2, the distance
                            to the path end within which the trajectorizer produces no seed (smaller: ARGUMENT) */
  const double* global_path;    /* [B][N][2], in the costmap frame */
  const double* pose;           /* [B][3] start pose x, y, yaw */
  const double* speed;          /* [B][2] measured (v, w) at tick 0 */
  const double* people;         /* [B][K][5] at t = 0: x, y, vx, vy, vz (people_msgs); may be NULL when K == 0 */
  const int32_t* n_people_each; /* [B] <= K; may be NULL when K == 0 */
  /* maps: same meaning as in smpc_fleet_io */
  const uint8_t* costmaps;      /* [M][size_y][size_x] */
  const double* costmap_origin; /* [M][2] */
  const int32_t* costmap_index; /* [B] or NULL (episode b uses map b % M) */
  int n_costmaps;
  int size_x;
  int size_y;
  double resolution;
  const uint32_t* od_indexes; /* [Mo][od_height * od_width] */
  const double* od_origin;    /* [Mo][2] */
  const int32_t* od_index;    /* [B] or NULL (episode b uses grid b % Mo) */
  int n_od_grids;
  uint32_t od_width;
  uint32_t od_height;
  float od_resolution;
  /* out, per episode (none may be NULL) */
  uint8_t* reached;             /* [B] 1 = within goal_tolerance of the last path pose */
  int32_t* ticks;               /* [B] ticks run: arrival tick + 1, or T */
  double* path_length;          /* [B] m driven */
  double* min_person_dist;      /* [B] m, +inf for a scene without people */
  int32_t* intimate_ticks;      /* [B] ticks with a person closer than 0.45 m */
  int32_t* personal_ticks;      /* [B] ticks with a person closer than 1.2 m */
  int32_t* collision_ticks;     /* [B] ticks on a costmap cell >= 253 (outside the map: 255) */
  int32_t* not_optimized_ticks; /* [B] ticks where optimize() returned false */
  double* cmd_variation;        /* [B] sum over k >= 1 of |v_k - v_k-1| + |w_k - w_k-1| */
  /* optional logs (NULL = off); rows after an episode is done repeat its final pose, cmd and optimized rows are 0 */
  double* pose_log;       /* [B][T+1][3] */
  double* cmd_log;        /* [B][T][2] */
  uint8_t* optimized_log; /* [B][T] */
} smpc_episode_io;
int smpc_run_episodes(smpc_handle* h, smpc_episode_io* io);

/* ---- closed-loop episodes with a reactive crowd ----------------------------------------------------------------------
 * smpc_run_episodes with people who walk to their own goals under the lightsfm social force model (sfm.hpp, with the
 * constants the controller's people projection uses) and react to the robot. io keeps its meaning; io->people holds
 * the state at t = 0, its velocity columns the initial velocities. Per tick k and episode still running, after the
 * fleet tick and before the world step, the crowd takes `substeps` synchronous updates of dt_s = control_period /
 * substeps. Agents: the people 0 .. n_people_each[b]-1 of the scene (all of them, not only those the FOV filter kept)
 * and the robot, which exerts force but is not moved by the model: at substep s it is at
 * x_k + (s dt_s) v_k (cos th_k, sin th_k) with velocity v_k (cos th_k, sin th_k), (v_k, w_k) = the command of tick k.
 * Forces on a person: toward its goal at its desired speed (braking -v / 0.5 once the goal is cleared), the nearest
 * obstacle cell of the episode's obstacle-distance grid at its current position (radius 0.5; none outside the grid),
 * and the pair force of every other person and of the robot. updatePosition (sfm.hpp:512-545): velocity capped at the
 * desired speed; the goal is cleared for good the first time an updated position is within 0.25 m of it; vz becomes
 * lightsfm's angular velocity. The FOV filter and the world step's metrics read the crowd's state (the controller at
 * tick k sees the people after k crowd ticks). Once an episode is done its people stand still.
 * Returns what smpc_run_episodes returns, plus SMPC_ERR_ARGUMENT for crowd == NULL, goals / desired_speed NULL while
 * n_people > 0, n_people > 63, substeps outside 1..64, a non-finite goal or a desired speed that is not finite and
 * > 0 for a person < n_people_each[b], or people_disturbance == NULL; all before anything is launched. */
typedef struct smpc_crowd_io {
  const double* goals;         /* [B][K][2] each person's goal, in the costmap frame */
  const double* desired_speed; /* [B][K] lightsfm desiredVelocity, m/s, > 0 */
  int substeps;                /* social-force updates per control period, 1..64 (dt_s = control_period / substeps) */
  double* people_disturbance;  /* [B] out: sum over ticks run, substeps and people of |F(robot -> person)| * dt_s */
  double* people_log;          /* [B][T+1][K][5] or NULL: x, y, vx, vy, vz at every tick (row 0 = the input); rows
                                  after an episode is done repeat its final row */
} smpc_crowd_io;
int smpc_run_crowd_episodes(smpc_handle* h, smpc_episode_io* io, const smpc_crowd_io* crowd);

/* ---- closed-loop episodes in shared scenes: several robots in one crowd -----------------------------------------------
 * smpc_run_crowd_episodes with the B robots grouped into S = B / R scenes of R = robots_per_scene consecutive robots
 * (robot r of scene s is episode s * R + r). The robots of a scene share one reactive crowd, one costmap and one
 * obstacle-distance grid, and each robot's controller sees the other robots of its scene as people.
 * Layout: io and crowd keep their fields. Per robot, B rows: global_path, pose, speed, every metric, pose_log, cmd_log,
 * optimized_log and people_disturbance. Per scene, S rows (a scene is stored once): io->people [S][K][5],
 * io->n_people_each [S], crowd->goals [S][K][2], crowd->desired_speed [S][K] and crowd->people_log [S][T+1][K][5].
 * costmap_index and od_index stay per robot and must be equal within a scene (with a NULL index array, robot b uses
 * map b % M, which must then be equal within a scene too).
 * What robot b sees at tick k: the FOV filter's input list holds the other R-1 robots of its scene first, in index
 * order, then the scene's people after k crowd steps. A robot enters as the person (x, y, v cos th, v sin th, w) with
 * its pose of tick k and its measured speed (v, w) of tick k (speed at k = 0, the previous command after that); a
 * robot whose episode is done stands at its final pose with zero velocity and stays visible. Robots go first because
 * the FOV filter keeps the first n_agents survivors: behind three people in view the robot most likely to be on a
 * collision course would drop out.
 * Crowd: one update per scene and substep with the K people and the R robots as agents (K + R <= 64). Each person feels
 * the pair force of every other person, then of robots 0 .. R-1 in order (R = 1: smpc_run_crowd_episodes exactly).
 * Robot r at substep s is at x_k + (s dt_s) v_k (cos th_k, sin th_k) for its own command; a finished robot stands
 * still. people_disturbance[b] sums |F(robot b -> person)| * dt_s while robot b runs. A scene's people move while any
 * robot of the scene runs; after that they stand still and their people_log rows repeat the final row.
 * World: robots do not push each other (no contact model); the person metrics stay against people only. Per robot
 * (scene->robot_min_dist, robot_intimate_ticks): the nearest other robot of the scene at (k+1) * control_period over
 * the ticks robot b ran (+inf for R = 1) and the ticks with another robot closer than 0.45 m.
 * Returns what smpc_run_crowd_episodes returns, plus SMPC_ERR_ARGUMENT for scene == NULL, robots_per_scene outside
 * 1..8, n_episodes not a multiple of it, n_people + robots_per_scene > 64, costmap_index or od_index differing within a
 * scene, or robot_min_dist / robot_intimate_ticks NULL; all before anything is launched. */
typedef struct smpc_scene_io {
  int robots_per_scene;          /* R, 1..8 */
  double* robot_min_dist;        /* [B] out: m, nearest other robot of the scene; +inf for R = 1 */
  int32_t* robot_intimate_ticks; /* [B] out: ticks with another robot of the scene closer than 0.45 m */
} smpc_scene_io;
int smpc_run_shared_episodes(smpc_handle* h, smpc_episode_io* io, const smpc_crowd_io* crowd,
                             const smpc_scene_io* scene);

/* ---- batched pre-solve stage on the GPU: project_people (src/optimizer.cpp:554-671 + sfm.hpp) -----------------
 * One warp per problem, lanes over agents, sequential over the horizon. Generalised from the reference's 3 people to
 * A columns. Inputs (device pointers): robot [B][S+1][6] = the robot AgentTrajectory of format_to_optimize
 * (x, y, yaw, t, lv, av), people_init [B][A][6] = people_to_status output (t == -1: padded), the obstacle-distance
 * grids od_indexes [M][height*width] (od_index [B] selects one, NULL: grid b % M). Output agents [B][A][6][S+1] in the
 * level-1 layout (valid people compacted to the front from step 1 on, like the reference), status [B]: 0 ok,
 * 1 = a person left the obstacle grid (the reference throws std::runtime_error there; its agents are marked invalid). */
typedef struct smpc_project_args {
  int n_problems;
  int n_steps;  /* S: robot has S+1 states */
  int n_agents; /* A <= 63 */
  int n_grids;  /* M */
  uint32_t od_width;
  uint32_t od_height;
  float od_resolution;
  float max_time;
  float time_step;
  const double* od_origin; /* [M][2] */
  const uint32_t* od_indexes;
  const int32_t* od_index; /* may be NULL */
  const double* robot;
  const double* people_init;
  double* agents;
  int32_t* status; /* may be NULL */
  const int32_t* n_steps_each; /* [B] per-problem horizon S_b <= n_steps (may be NULL); array strides stay n_steps + 1 */
} smpc_project_args;
int smpc_project_people_batch_device(smpc_handle* h, const smpc_project_args* a, void* stream);
/* Host-buffer wrapper (tests): same struct with host pointers. */
int smpc_project_people_batch(smpc_handle* h, const smpc_project_args* a);

/* ---- batched pre-solve stage on the GPU: format_to_optimize + unpacking (src/optimizer.cpp:484-551, :197-237) ----
 * One thread per (problem, pose). poses [B][n_poses][3] (x, y, yaw = tf2::getYaw), cmds [B][n_poses-1][2], speed [B][2];
 * prev_poses / prev_cmds: the previous tick's OUTPUT with n_prev_poses / n_prev_cmds entries per robot (NULL or 0 on
 * the first tick: previous = current, :177-181). The caller has already applied the max_time cut (:492-497).
 * Outputs: robot [B][n_poses][6] (input of project_people) and the level-1 arrays pose0 [B][3], u0 [B][NB][2],
 * path_xy [B][2][n_poses], goal_yaw [B]. All device pointers. */
typedef struct smpc_format_args {
  int n_problems;
  int n_poses;
  int n_prev_poses;
  int n_prev_cmds;
  int n_blocks;
  float time_step;
  float current_path_w;
  float current_cmds_w;
  const double* poses;
  const double* cmds;
  const double* speed;
  const double* prev_poses;
  const double* prev_cmds;
  double* robot;
  double* pose0;
  double* u0;
  double* path_xy;
  double* goal_yaw;
  /* Per-robot lengths (all may be NULL / 0 = uniform): n_poses_each [B] poses kept per robot (<= n_poses = the row
   * stride; < 2: the robot is inactive, its level-1 inputs are zeroed and has_people[b] cleared), n_prev_poses_each /
   * n_prev_cmds_each [B] entries of the robot's memory rows (strides n_prev_poses / n_prev_cmds), cmds_stride = row
   * stride of cmds (0: n_poses - 1), has_people [B] (may be NULL). */
  const int32_t* n_poses_each;
  const int32_t* n_prev_poses_each;
  const int32_t* n_prev_cmds_each;
  int cmds_stride;
  uint8_t* has_people;
} smpc_format_args;
int smpc_format_batch_device(smpc_handle* h, const smpc_format_args* a, void* stream);

/* ---- batched seed generation on the GPU: PathTrajectorizer::trajectorize (src/path_trajectorizer.cpp:120-288) ----
 * One warp per robot (the 32 lanes search the global path for the look-ahead point): pure-pursuit on its global path, diff-drive (curvature law, rotate in place beyond
 * 90 deg) or omnidirectional branch (:190-194), forward-Euler simulation with the DOUBLE time_step (SURVEY Q15), early
 * stop within 0.2 m of the goal. global_path [B][n_path][2] (path_index NULL) or [Mp][n_path][2] selected by
 * path_index [B]; pose [B][3]. Outputs poses [B][max_steps+1][3] (pose 0 = the robot pose, yaw round-tripped like
 * setRPY/getYaw), cmds [B][max_steps][3] = linear.x, linear.y, angular.z, n_steps [B] = steps actually produced
 * (entries beyond it are left untouched). Returns the reference's `false` (path with < 2 poses) as SMPC_ERR_ARGUMENT. */
typedef struct smpc_trajectorize_args {
  int n_problems;
  int n_path;
  int max_steps;
  int omnidirectional;
  double desired_linear_vel;
  double lookahead_dist;
  double max_angular_vel;
  double time_step;
  const double* global_path;
  const int32_t* path_index; /* may be NULL */
  const double* pose;
  double* poses;
  double* cmds;
  int32_t* n_steps;
} smpc_trajectorize_args;
int smpc_trajectorize_batch_device(smpc_handle* h, const smpc_trajectorize_args* a, void* stream);

/* people_to_status (src/optimizer.cpp:454-482) for a fleet: people_raw [B][A][5] = position.x/y, velocity.x/y/z,
 * n_people [B] (entries >= n_people[b] are padding; more than A people are truncated by the caller like :476-479).
 * Outputs people_init [B][A][6] and has_people [B] (u8). Device pointers. */
int smpc_people_to_status_device(smpc_handle* h, int n_problems, int n_agents, const double* people_raw,
                                 const int32_t* n_people, double* people_init, uint8_t* has_people, void* stream);
/* TrajectoryMemory update of a fleet tick (src/optimizer.cpp:448-449): where usable[b], prev_poses[b] <- path[b] and
 * prev_cmds[b] <- cmds[b] (n entries of 3 / 2 doubles each); other robots keep their memory. Device pointers. */
int smpc_memory_update_device(smpc_handle* h, int n_problems, int n, const uint8_t* usable, const double* path,
                              const double* cmds, double* prev_poses, double* prev_cmds, void* stream);

/* ---- in-library multi-GPU dispatch of the level-1 solve (SURVEY §8e) -------------------------------------------
 * One handle + one host thread per GPU; the host batch is cut into contiguous shards whose boundaries are multiples of
 * `granule` (multi-start: starts per robot, so a robot's arg-min never spans GPUs); every shard runs the ordinary
 * host-buffer pipeline and its results land in the caller's arrays at the shard's offset (the final host gather). No
 * collective, nothing on the solve path crosses GPUs. `devices` may name a GPU twice (two handles on it). */
typedef struct smpc_multi smpc_multi;
int smpc_multi_create(const smpc_params* p, int n_devices, const int* devices /* NULL: 0 .. n_devices-1 */, smpc_multi** out);
void smpc_multi_destroy(smpc_multi* m);
int smpc_multi_device_count(smpc_multi* m);
int smpc_solve_batch_multi(smpc_multi* m, const smpc_batch* in, smpc_result* out, int granule);
/* Diagnostics (no GPU needed): [lo, hi) of `shard` when n_problems are cut into n_shards at multiples of granule. */
int smpc_debug_shard_bounds(int n_problems, int n_shards, int shard, int granule, int* lo, int* hi);

/* ---- FOV people filter of SocialMPCController::computeVelocityCommands (src/social_mpc_controller.cpp:198-214) for a
 * fleet: a person survives when it lies inside the robot's costmap (Costmap2D::worldToMap) and its bearing is within
 * fov_angle of the robot's yaw (float roundings of the reference kept). Order-preserving; the first n_out_max
 * survivors are written, n_people_out [B] counts ALL survivors (people.people.size(), which decides has_people).
 * Device pointers. */
typedef struct smpc_fov_args {
  int n_robots;
  int n_in_max;  /* row stride of people_in */
  int n_out_max; /* row stride of people_out (3 for the reference's optimizer) */
  int n_costmaps, size_x, size_y;
  double resolution;
  double fov_angle;             /* FollowPath.fov_angle, default pi/4 (src/social_mpc_controller.cpp:60) */
  const double* people_in;      /* [B][n_in_max][5] position.x/y, velocity.x/y/z */
  const int32_t* n_people_in;   /* [B] */
  const double* pose;           /* [B][3] robot x, y, yaw */
  const double* costmap_origin; /* [M][2] */
  const int32_t* costmap_index; /* [B] or NULL (robot b uses map b % M) */
  double* people_out;           /* [B][n_out_max][5] */
  int32_t* n_people_out;        /* [B] */
} smpc_fov_args;
int smpc_fov_filter_batch_device(smpc_handle* h, const smpc_fov_args* a, void* stream);

/* Multi-start selection: per robot arg-min of cost_final over `n_starts`
 * consecutive problems (device pointers). best_index [R] i32 (global problem
 * index, -1 if no usable start), best_cost [R], best_u [R][NB][2]. */
int smpc_multistart_argmin_device(smpc_handle* h, int n_robots, int n_starts, int n_blocks, const double* cost_final,
                                  const uint8_t* usable, const double* u, int32_t* best_index, double* best_cost,
                                  double* best_u, void* stream);

/* Work mapping: lanes of a warp that cooperate on one problem (4, 8, 16, 32; 0 = choose from the batch size:
 * 32 for single solves / lowest latency, 4 for large batches / highest throughput). Results do not depend on it
 * beyond floating-point summation order. */
int smpc_set_group(smpc_handle* h, int lanes_per_problem);

/* Device-time (ms) of the solve kernel of the last *_device / host solve call,
 * measured with CUDA events on the launching stream; < 0 if unavailable.
 * Synchronises the stream. */
double smpc_last_kernel_ms(smpc_handle* h);
/* Number of kernels this library launched on the handle since creation. */
long long smpc_launch_count(smpc_handle* h);
/* Measured FP64 FMA throughput of this GPU (TFLOP/s, DFMA-saturating microbenchmark, best of 5): the roofline
 * denominator of the solve kernel ("of measured"; MEASURED_PEAKS.json carries no FP64 figure). */
int smpc_measure_fp64_peak(smpc_handle* h, double* tflops);
/* Diagnostics for unit tests (no GPU needed): the chunk plan smpc_solve_batch would use for a host batch of
 * `n_problems` on a GPU with `n_sm` SMs. has_people = agent columns and a has_people array are given;
 * maps_per_problem = one costmap per problem (no index, or an identity index); has_index = a non-identity
 * costmap_index; forced_chunks = the SMPC_CHUNKS override (0 = heuristic). Outputs: number of chunks and problems
 * per chunk (the last chunk holds the remainder). */
int smpc_debug_plan_chunks(int n_sm, int n_problems, int has_people, int n_costmaps, int maps_per_problem, int has_index,
                           int forced_chunks, int* n_chunks, int* chunk);
/* Diagnostics for unit tests: run the line-search interpolating-polynomial minimiser (Ceres polynomial.cc
 * restatement) on n host rows of (lo, hi, f0, g0, t1, f1, g1, t2, f2, g2); t2 <= 0 selects the 2-sample case. */
int smpc_debug_polymin(smpc_handle* h, int n, const double* rows, double* out);
/* Diagnostics for unit tests: the social-force loops' own elementary functions (csrc/smpc_math.cuh) on n host rows of
 * (a, b): kind 0 = exp_nonpos(a) (a <= 0), 1 = rsqrt_pos(a) (a > 0, normal), 2 = atan2_unit(a, b) (|(b, a)| ~ 1). */
int smpc_debug_math(smpc_handle* h, int kind, int n, const double* rows, double* out);

#ifdef __cplusplus
}
#endif
#endif /* SMPC_H_ */
