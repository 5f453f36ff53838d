// smpc_episode.cu — closed-loop episodes (smpc_run_episodes, smpc_run_crowd_episodes, smpc_run_shared_episodes,
// smpc_run_weighted_episodes, smpc_run_orca_episodes, smpc_run_perceived_episodes, smpc_run_tracked_episodes,
// smpc_run_local_costmap_episodes): B robots through their crowd scenes for up to T controller ticks, every tick
// enqueued on the handle's stream without a host round trip. One tick per episode is
//   trajectorizer (seed) -> tick prep (constant-velocity people at k * dt_c, seed repack, max_time cut) -> [scene view]
//   -> [perception, smpc_perception.cu, or tracked perception, smpc_tracker.cu] -> [local costmap build on build
//   ticks, smpc_local_costmap.cu] -> FOV filter -> fleet tick
//   (smpc_fleet_tick_enqueue) -> [reactive crowd step, smpc_crowd.cu, or ORCA crowd step, smpc_orca.cu] -> world step
//   (robot Euler step, metrics, goal check, logs) -> [robot-robot metrics].
// All entries share one loop: with a crowd the prep leaves the people alone, the FOV filter and the world step read
// the crowd's state, and the crowd step moves it from tick k to k + 1. Shared scenes (R robots per scene, one crowd per
// scene) add the scene view, which puts the other robots of the scene in front of the people the FOV filter sees, and
// the robot-robot metrics. The fleet tick runs on the handle's third fleet state, so episodes never touch the
// warm-start memory of smpc_optimize_batch or smpc_optimize.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/smpc.h"
#include "smpc_host_state.h"

namespace {

constexpr int kPollTicks = 16;  // ticks between two reads of the device count of active episodes
constexpr int kCrowdMaxAgents = 64;  // people + robots in the agent slots of smpc_crowd_step_kernel
constexpr int kMaxRobotsPerScene = 8;
constexpr int kPerceptionMaxRows = 64;  // two rows per lane of smpc_perception_kernel's warp
constexpr double kIntimate = 0.45;  // m, the intimate zone of the person metrics
// The trajectorizer produces no step within this distance of the path end (smpc_trajectorize_kernel,
// src/path_trajectorizer.cpp:152). A robot that close has no seed, so the fleet tick leaves it inactive and its
// command is zero: a goal tolerance below this distance could leave it standing short of the goal until T.
constexpr double kSeedGoalStop = 0.2;

struct EpisodePrep {
  int B, K, stride, max_steps, maxsize;
  double t;  // k * dt_c
  const int32_t* n_steps;   // [B] seed steps from the trajectorizer
  const double* seed_cmds;  // [B][max_steps][3] linear.x, linear.y, angular.z
  const uint8_t* active;    // [B]
  const double* people0;    // [B][K][5] at t = 0
  double* people;           // [B][K][5] at t
  double* poses;            // [B][stride][3] seed poses (rows beyond the seed are zeroed)
  double* cmds;             // [B][stride][2] (linear.x, angular.z), zero beyond the seed
  int32_t* n_in;
  int32_t* n_each;
  int32_t* s_each;
};

// One thread per (episode, row): the seed repack and the constant-velocity people of this tick, and the per-robot
// sizes of the fleet tick with the max_time cut of format_to_optimize (src/optimizer.cpp:492-497).
__global__ void smpc_episode_prep_kernel(EpisodePrep a) {
  const int rows = a.stride > a.K ? a.stride : a.K;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)a.B * rows) return;
  const int b = (int)(t / rows), i = (int)(t % rows);
  const int ns = a.n_steps[b];
  if (i < a.stride) {
    double* c = a.cmds + ((size_t)b * a.stride + i) * 2;
    if (i < ns) {
      const double* s = a.seed_cmds + ((size_t)b * a.max_steps + i) * 3;
      c[0] = s[0];
      c[1] = s[2];
    } else {
      c[0] = 0.0;
      c[1] = 0.0;
    }
    if (i > ns)
      for (int q = 0; q < 3; ++q) a.poses[((size_t)b * a.stride + i) * 3 + q] = 0.0;
  }
  if (i < a.K) {
    const double* p0 = a.people0 + ((size_t)b * a.K + i) * 5;
    double* p = a.people + ((size_t)b * a.K + i) * 5;
    p[0] = __dadd_rn(p0[0], __dmul_rn(p0[2], a.t));
    p[1] = __dadd_rn(p0[1], __dmul_rn(p0[3], a.t));
    p[2] = p0[2];
    p[3] = p0[3];
    p[4] = p0[4];
  }
  if (i == 0) {
    const int n = a.active[b] ? ns + 1 : 0;
    int cut = 0;
    if (n >= 2) cut = n > a.maxsize ? a.maxsize - 1 : n;  // >= 2: checked on the host before the first tick
    a.n_in[b] = n;
    a.n_each[b] = cut;
    a.s_each[b] = cut >= 2 ? cut - 1 : 1;
  }
}

struct EpisodeStep {
  int B, R, K, T, k, stride, n_path;  // R robots per scene: robot b sees the people of scene b / R
  double dt_c, goal_tol;
  const double* cmds;          // [B][stride][2] fleet tick output: row 0 is the command
  const uint8_t* optimized;    // [B]
  const double* people0;       // [B/R][K][5]
  const double* people_now;    // [B/R][K][5] people at (k+1) * dt_c (reactive crowd), or NULL: people0 at constant
                               // velocity
  const int32_t* n_people;     // [B/R] or NULL (K == 0)
  const double* global_path;   // [B][N][2]
  const uint8_t* maps;
  const double* map_org;
  const int32_t* map_index;    // may be NULL
  int n_costmaps, size_x, size_y;
  double resolution;
  double* pose;                // [B][3] in: x_k, out: x_k+1
  double* speed;               // [B][2] in: measured speed of tick k (= cmd_k-1 for k >= 1), out: cmd_k
  uint8_t* active;
  int* n_active;
  uint8_t* reached;
  int32_t* ticks;
  double* path_length;
  double* min_dist;
  int32_t* intimate;
  int32_t* personal;
  int32_t* collision;
  int32_t* not_optimized;
  double* cmd_variation;
  double* pose_log;            // [B][T+1][3] or NULL
  double* cmd_log;             // [B][T][2] or NULL
  uint8_t* optimized_log;      // [B][T] or NULL
};

__device__ __forceinline__ double hypot_rn(double dx, double dy) {  // no FMA contraction: numpy reproduces it bit for bit
  return sqrt(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
}

// One warp per episode, lanes over people. Robot: unicycle forward Euler over dt_c, yaw through setRPY / getYaw.
// Metrics at time (k+1) * dt_c against all people of the scene (not only those the FOV filter kept; no robots).
__global__ void __launch_bounds__(128) smpc_episode_step_kernel(EpisodeStep a) {
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (b >= a.B || !a.active[b]) return;  // warp-uniform
  const double v = a.cmds[(size_t)b * a.stride * 2], w = a.cmds[(size_t)b * a.stride * 2 + 1];
  const bool opt = a.optimized[b] != 0;
  const double x = a.pose[3 * b], y = a.pose[3 * b + 1], th = a.pose[3 * b + 2];
  double st, ct;
  sincos(th, &st, &ct);
  const double x1 = __dadd_rn(x, __dmul_rn(__dmul_rn(v, ct), a.dt_c));
  const double y1 = __dadd_rn(y, __dmul_rn(__dmul_rn(v, st), a.dt_c));
  const double th1 = __dadd_rn(th, __dmul_rn(w, a.dt_c));
  double sh, ch;
  sincos(th1 * 0.5, &sh, &ch);
  const double yaw1 = atan2(2.0 * (ch * sh), ch * ch - sh * sh);  // setRPY(0, 0, th1) read back by getYaw

  // nearest person at (k+1) * dt_c
  const double t1 = __dmul_rn((double)(a.k + 1), a.dt_c);
  const int sc = b / a.R;
  const int np = a.K > 0 ? a.n_people[sc] : 0;
  double dmin = INFINITY;
  for (int j = lane; j < np; j += 32) {
    double px, py;
    if (a.people_now) {
      px = a.people_now[((size_t)sc * a.K + j) * 5];
      py = a.people_now[((size_t)sc * a.K + j) * 5 + 1];
    } else {
      const double* p = a.people0 + ((size_t)sc * a.K + j) * 5;
      px = __dadd_rn(p[0], __dmul_rn(p[2], t1));
      py = __dadd_rn(p[1], __dmul_rn(p[3], t1));
    }
    dmin = fmin(dmin, hypot_rn(__dsub_rn(px, x1), __dsub_rn(py, y1)));
  }
  for (int off = 16; off > 0; off >>= 1) dmin = fmin(dmin, __shfl_xor_sync(0xffffffffu, dmin, off));
  if (lane != 0) return;

  // costmap cell under the robot (Costmap2D::worldToMap; outside the map reads as 255)
  const int mi = a.map_index ? a.map_index[b] : b % a.n_costmaps;
  const double ox = a.map_org[2 * mi], oy = a.map_org[2 * mi + 1];
  int cost = 255;
  if (x1 >= ox && y1 >= oy) {
    const unsigned mx = (unsigned)((x1 - ox) / a.resolution), my = (unsigned)((y1 - oy) / a.resolution);
    if (mx < (unsigned)a.size_x && my < (unsigned)a.size_y)
      cost = a.maps[((size_t)mi * a.size_y + my) * a.size_x + mx];
  }
  const double* goal = a.global_path + ((size_t)b * a.n_path + a.n_path - 1) * 2;
  const bool done = hypot_rn(__dsub_rn(x1, goal[0]), __dsub_rn(y1, goal[1])) <= a.goal_tol;
  const double step = hypot_rn(__dsub_rn(x1, x), __dsub_rn(y1, y));

  if (a.k == 0) {
    a.path_length[b] = step;
    a.min_dist[b] = dmin;
    a.intimate[b] = dmin < kIntimate;
    a.personal[b] = dmin < 1.2;
    a.collision[b] = cost >= 253;
    a.not_optimized[b] = !opt;
    a.cmd_variation[b] = 0.0;
    if (a.pose_log) {
      double* pl = a.pose_log + (size_t)b * (a.T + 1) * 3;
      pl[0] = x; pl[1] = y; pl[2] = th;
    }
  } else {
    a.path_length[b] = __dadd_rn(a.path_length[b], step);
    a.min_dist[b] = fmin(a.min_dist[b], dmin);
    a.intimate[b] += dmin < kIntimate;
    a.personal[b] += dmin < 1.2;
    a.collision[b] += cost >= 253;
    a.not_optimized[b] += !opt;
    const double dv = __dadd_rn(fabs(__dsub_rn(v, a.speed[2 * b])), fabs(__dsub_rn(w, a.speed[2 * b + 1])));
    a.cmd_variation[b] = __dadd_rn(a.cmd_variation[b], dv);
  }
  a.pose[3 * b] = x1;
  a.pose[3 * b + 1] = y1;
  a.pose[3 * b + 2] = yaw1;
  a.speed[2 * b] = v;  // ideal actuator
  a.speed[2 * b + 1] = w;
  if (a.pose_log) {
    double* pl = a.pose_log + ((size_t)b * (a.T + 1) + a.k + 1) * 3;
    pl[0] = x1; pl[1] = y1; pl[2] = yaw1;
  }
  if (a.cmd_log) {
    a.cmd_log[((size_t)b * a.T + a.k) * 2] = v;
    a.cmd_log[((size_t)b * a.T + a.k) * 2 + 1] = w;
  }
  if (a.optimized_log) a.optimized_log[(size_t)b * a.T + a.k] = opt;
  a.reached[b] = done;
  a.ticks[b] = a.k + 1;
  if (done) {
    a.active[b] = 0;
    atomicSub(a.n_active, 1);
  }
}

struct SceneView {
  int B, R, K, n_view;  // n_view = R - 1 + K rows per robot
  const uint8_t* active;    // [B]
  const double* pose;       // [B][3] x_k
  const double* speed;      // [B][2] measured speed of tick k
  const double* people;     // [B/R][K][5] the crowd after k steps
  const int32_t* n_people;  // [B/R] or NULL (K == 0)
  double* view;             // [B][n_view][5] the FOV filter's input
  int32_t* n_view_each;     // [B]
};

// One thread per (robot, row): rows 0 .. R-2 hold the other robots of the scene in index order as people
// (x, y, v cos th, v sin th, w) with the measured speed of tick k (zero once a robot is done), then the scene's people.
// Robots go first because the FOV filter keeps the first n_agents survivors.
__global__ void smpc_scene_view_kernel(SceneView a) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)a.B * a.n_view) return;
  const int b = (int)(t / a.n_view), i = (int)(t % a.n_view);
  const int sc = b / a.R, me = b % a.R;
  double* o = a.view + ((size_t)b * a.n_view + i) * 5;
  if (i < a.R - 1) {
    const int ob = sc * a.R + (i < me ? i : i + 1);
    const bool on = a.active[ob] != 0;
    const double v = on ? a.speed[2 * ob] : 0.0, w = on ? a.speed[2 * ob + 1] : 0.0;
    double st, ct;
    sincos(a.pose[3 * ob + 2], &st, &ct);
    o[0] = a.pose[3 * ob];
    o[1] = a.pose[3 * ob + 1];
    o[2] = __dmul_rn(v, ct);
    o[3] = __dmul_rn(v, st);
    o[4] = w;
  } else {
    const double* p = a.people + ((size_t)sc * a.K + (i - (a.R - 1))) * 5;
    for (int q = 0; q < 5; ++q) o[q] = p[q];
  }
  if (i == 0) a.n_view_each[b] = a.R - 1 + (a.K > 0 ? a.n_people[sc] : 0);
}

struct RobotMetrics {
  int B, R, k;
  const double* pose;    // [B][3] x_k+1 (after the world step)
  const int32_t* ticks;  // [B] == k + 1 for the robots that ran tick k
  double* min_dist;      // [B]
  int32_t* intimate;     // [B]
};

// One thread per robot that ran tick k: the nearest other robot of its scene at (k+1) * dt_c (finished robots stand
// at their final pose). +inf with one robot per scene.
__global__ void smpc_robot_metrics_kernel(RobotMetrics a) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= a.B || a.ticks[b] != a.k + 1) return;
  const int r0 = b - b % a.R;
  const double x = a.pose[3 * b], y = a.pose[3 * b + 1];
  double dmin = INFINITY;
  for (int o = r0; o < r0 + a.R; ++o)
    if (o != b) dmin = fmin(dmin, hypot_rn(__dsub_rn(a.pose[3 * o], x), __dsub_rn(a.pose[3 * o + 1], y)));
  if (a.k == 0) {
    a.min_dist[b] = dmin;
    a.intimate[b] = dmin < kIntimate;
  } else {
    a.min_dist[b] = fmin(a.min_dist[b], dmin);
    a.intimate[b] += dmin < kIntimate;
  }
}

// The loop of all entries; crowd == NULL: constant-velocity people (smpc_run_episodes); scene == NULL: one robot per
// scene (smpc_run_episodes, smpc_run_crowd_episodes).
// w != NULL: per-episode critic weights (smpc_run_weighted_episodes). orca != NULL (checked, crowd given): the crowd
// moves by ORCA (smpc_run_orca_episodes) instead of the social force model. pc != NULL (parameters checked): the
// perception stage cuts the FOV filter's input to what the sensor reports (smpc_run_perceived_episodes). tk != NULL
// (checked, pc given): a people tracker follows the sensor and the FOV filter reads its delayed published list
// (smpc_run_tracked_episodes). local != NULL (outputs checked): the FOV filter and the fleet tick read per-robot rolling
// windows that smpc_local_costmap_kernel rebuilds every update_period_ticks (smpc_run_local_costmap_episodes).
int run_episodes(smpc_handle* h, smpc_episode_io* io, const smpc_crowd_io* crowd, const smpc_scene_io* scene,
                 const char* name, const smpc_weight_sets* w = nullptr, const smpc_orca_params* orca = nullptr,
                 const smpc_perception* pc = nullptr, const smpc_tracker* tk = nullptr,
                 const smpc_local_costmap* local = nullptr) {
  auto fail_arg = [name](const char* msg) {
    return smpc_host_fail(SMPC_ERR_ARGUMENT, std::string(name) + ": " + msg);
  };
  if (!h || !io) return smpc_host_fail(SMPC_ERR_ARGUMENT, "NULL argument");
  const smpc_params* prm = smpc_handle_params(h);
  if (prm->omni_solve)
    return smpc_host_fail(SMPC_ERR_UNSUPPORTED, std::string(name) + ": the fleet tick has no omnidirectional solve");
  if (prm->omnidirectional)
    return smpc_host_fail(SMPC_ERR_UNSUPPORTED,
                          std::string(name) + ": the world step moves a unicycle, not an omnidirectional robot");
  const int B = io->n_episodes, T = io->n_ticks, N = io->n_path, K = io->n_people, A = io->n_agents;
  if (B < 0) return fail_arg("n_episodes < 0");
  if (N < 2) return fail_arg("n_path < 2");
  if (T < 1) return fail_arg("n_ticks < 1");
  if (A < 1 || A > 63) return fail_arg("n_agents outside 1..63");
  if (K < 0) return fail_arg("n_people < 0");
  if (!(io->control_period > 0.0)) return fail_arg("control_period <= 0");
  if (!(io->goal_tolerance >= kSeedGoalStop))
    return fail_arg("goal_tolerance below the trajectorizer's 0.2 m stop at the path end");
  if (!io->global_path || !io->pose || !io->speed || (K > 0 && (!io->people || !io->n_people_each)))
    return fail_arg("missing input");
  if (!io->costmaps || !io->costmap_origin || io->n_costmaps < 1 || io->size_x < 1 || io->size_y < 1 ||
      !(io->resolution > 0.0))
    return fail_arg("missing costmaps");
  if (!io->od_indexes || !io->od_origin || io->n_od_grids < 1 || io->od_width == 0 || io->od_height == 0 ||
      !(io->od_resolution > 0.0f))
    return fail_arg("missing obstacle-distance grids");
  if (!io->reached || !io->ticks || !io->path_length || !io->min_person_dist || !io->intimate_ticks ||
      !io->personal_ticks || !io->collision_ticks || !io->not_optimized_ticks || !io->cmd_variation)
    return fail_arg("missing output");
  const int R = scene ? scene->robots_per_scene : 1;
  if (R < 1 || R > kMaxRobotsPerScene) return fail_arg("robots_per_scene outside 1..8");
  if (B % R != 0) return fail_arg("n_episodes not a multiple of robots_per_scene");
  if (scene && (!scene->robot_min_dist || !scene->robot_intimate_ticks)) return fail_arg("missing output");
  if (w) {
    const int rc = smpc_check_weight_sets(w, B, name);
    if (rc != SMPC_OK) return rc;
  }
  const int S = B / R;  // scenes: people, n_people_each, goals, desired_speed and people_log have S rows
  for (int c = 0; c < S && K > 0; ++c)
    if (io->n_people_each[c] < 0 || io->n_people_each[c] > K) return fail_arg("n_people_each[b] outside 0..K");
  for (int b = 0; b < B; ++b) {
    if (io->costmap_index && (io->costmap_index[b] < 0 || io->costmap_index[b] >= io->n_costmaps))
      return fail_arg("costmap_index[b] outside 0..n_costmaps-1");
    if (io->od_index && (io->od_index[b] < 0 || io->od_index[b] >= io->n_od_grids))
      return fail_arg("od_index[b] outside 0..n_od_grids-1");
    const int r0 = b - b % R;  // the robots of a scene share its costmap and obstacle grid
    if ((io->costmap_index ? io->costmap_index[b] != io->costmap_index[r0] : b % io->n_costmaps != r0 % io->n_costmaps) ||
        (io->od_index ? io->od_index[b] != io->od_index[r0] : b % io->n_od_grids != r0 % io->n_od_grids))
      return fail_arg("costmap_index or od_index differs within a scene");
  }
  const bool reactive = crowd != nullptr;
  if (reactive) {
    if (K + R > kCrowdMaxAgents)
      return fail_arg("n_people + robots_per_scene above 64 (people and robots share one warp's 64 slots)");
    if (crowd->substeps < 1 || crowd->substeps > 64) return fail_arg("substeps outside 1..64");
    if (K > 0 && (!crowd->goals || !crowd->desired_speed)) return fail_arg("missing goals or desired speeds");
    if (!crowd->people_disturbance) return fail_arg("missing output");
    for (int b = 0; b < S && K > 0; ++b)
      for (int i = 0; i < io->n_people_each[b]; ++i) {
        const double* g = crowd->goals + ((size_t)b * K + i) * 2;
        const double vd = crowd->desired_speed[(size_t)b * K + i];
        if (!std::isfinite(g[0]) || !std::isfinite(g[1])) return fail_arg("non-finite goal");
        if (!std::isfinite(vd) || !(vd > 0.0)) return fail_arg("desired_speed not finite and > 0");
      }
  }
  const int n_list = scene ? R - 1 + K : K;  // rows of the FOV filter's input
  if (pc) {
    if (n_list > kPerceptionMaxRows) return fail_arg("the perceived list (R - 1 + n_people rows) above 64");
    for (int b = 0; b < B && pc->stream_index; ++b)
      if (pc->stream_index[b] < 0) return fail_arg("stream_index[b] < 0");
  }
  std::vector<uint8_t> stencil;
  int half = 0;
  if (local) {
    const int lrc = smpc_local_costmap_build_stencil(local, io->resolution, &stencil, &half, name);
    if (lrc != SMPC_OK) return lrc;
  }
  // the trajectorizer integrates with the yaml DOUBLE time_step (SURVEY Q15), as FleetOptimizer.trajectorize_batch
  const double traj_dt = std::round((double)prm->time_step * 1e6) / 1e6;
  const int max_steps = (int)std::round((double)prm->max_time / traj_dt);
  if (!(traj_dt > 0.0) || max_steps < 1) return fail_arg("max_time / time_step give no trajectorizer step");
  const int stride = max_steps + 1;
  const float timestep = prm->time_step, maxtime = prm->max_time;
  const int maxsize = (int)std::round(maxtime / timestep);
  if (stride > maxsize && maxsize - 1 < 2) return fail_arg("max_time / time_step leaves fewer than 2 poses");
  int nb = 0;
  int rc = smpc_problem_dims(prm, stride - 1, nullptr, nullptr, &nb, nullptr);
  if (rc != SMPC_OK) return rc;
  if (B == 0) return SMPC_OK;

  smpc_fleet_state* fs = smpc_handle_episodes(h);
  std::lock_guard<std::mutex> lk(fs->mu);
  SMPC_FLEET_CUDA(cudaSetDevice(smpc_handle_device(h)));
  cudaStream_t st = smpc_handle_stream(h);

  smpc_fleet_dev d{};
  d.B = B; d.stride = stride; d.A = A; d.nb = nb; d.time_step = timestep; d.max_time = maxtime;
  fs->forget();  // fresh warm-start memory for every call
  SMPC_FLEET_CUDA(smpc_fleet_memory(fs, &d, st));

  // ---- maps, uploaded once per call
  const size_t map_bytes = (size_t)io->n_costmaps * io->size_x * io->size_y;
  const size_t od_bytes = (size_t)io->n_od_grids * io->od_width * io->od_height * sizeof(uint32_t);
  const size_t Bz = B, Sz = S, Kz = K, BS = Bz * stride;
  const int n_view = scene ? R - 1 + K : 0;  // rows of a robot's scene view (0: the FOV filter reads the people)
  const bool fov = scene ? n_view > 0 : K > 0;
  const bool logs_pose = io->pose_log != nullptr, logs_cmd = io->cmd_log != nullptr, logs_opt = io->optimized_log != nullptr;
  const bool logs_people = reactive && crowd->people_log != nullptr;
  const bool perceive = pc && fov;  // K = 0 and R = 1: no list to perceive
  const bool logs_seen = perceive && pc->seen_log != nullptr;
  const size_t Lz = n_list;
  double* seen = nullptr, *seen_log = nullptr;
  int32_t *seen_n = nullptr, *unseen = nullptr, *stream_idx = nullptr, *n_seen_log = nullptr;
  const bool tracked = perceive && tk != nullptr;
  const size_t Mz = scene ? K + R : K, Dz = tracked ? tk->latency_ticks + 1 : 0;  // track slots, ring slots
  double *trk_x = nullptr, *trk_y = nullptr, *trk_vx = nullptr, *trk_vy = nullptr;
  double *trk_pp = nullptr, *trk_pv = nullptr, *trk_vv = nullptr, *ring = nullptr, *pos_err = nullptr, *vel_err = nullptr;
  int32_t *trk_hits = nullptr, *trk_misses = nullptr, *ring_n = nullptr, *ring_id = nullptr, *untracked = nullptr;
  int32_t *track_rows = nullptr, *id_log = nullptr;
  double *goals = nullptr, *vdes = nullptr, *disturbance = nullptr, *people_log = nullptr;
  double *view = nullptr, *robot_min = nullptr;
  int32_t *view_n = nullptr, *robot_intimate = nullptr;
  uint8_t* has_goal = nullptr;
  int32_t* n_people_dev = nullptr;
  double *gp, *pose, *people0, *people, *seed_cmds, *pose_log, *cmd_log, *path_length, *min_dist, *cmd_var;
  int32_t *map_index, *od_index, *n_steps, *fov_n, *ticks, *intimate, *personal, *collision, *not_opt;
  uint8_t *active, *reached, *opt_log, *maps;
  double *map_org, *od_org, *fov_people, *speed;
  uint32_t* od;
  int* n_active;
  double* weights = nullptr;
  int32_t* weight_set = nullptr;
  const int n_period = local ? local->update_period_ticks : 1, n_builds = (T + n_period - 1) / n_period;
  const size_t cells = local ? (size_t)local->size_x * local->size_y : 0;
  const bool logs_local = local && local->costmap_log != nullptr;
  uint8_t *windows = nullptr, *stencil_dev = nullptr, *window_log = nullptr;
  double *window_org = nullptr, *window_org_log = nullptr;
  int32_t* marked = nullptr;
  auto carve = [&](smpc_carve& c) {
    maps = c.take<uint8_t>(map_bytes);
    od = c.take<uint32_t>(od_bytes / 4);
    map_org = c.take<double>((size_t)io->n_costmaps * 2);
    od_org = c.take<double>((size_t)io->n_od_grids * 2);
    map_index = c.take<int32_t>(Bz);
    od_index = c.take<int32_t>(Bz);
    gp = c.take<double>(Bz * N * 2);
    pose = c.take<double>(Bz * 3);
    speed = c.take<double>(Bz * 2);
    people0 = c.take<double>(Sz * Kz * 5);
    people = c.take<double>(Sz * Kz * 5);
    n_people_dev = c.take<int32_t>(Sz);
    seed_cmds = c.take<double>(Bz * max_steps * 3);
    n_steps = c.take<int32_t>(Bz);
    fov_people = c.take<double>(Bz * A * 5);
    fov_n = c.take<int32_t>(Bz);
    d.poses = c.take<double>(BS * 3);
    d.cmds = c.take<double>(BS * 2);
    d.n_in = c.take<int32_t>(Bz);
    d.n_each = c.take<int32_t>(Bz);
    d.s_each = c.take<int32_t>(Bz);
    smpc_fleet_carve_stages(c, &d);
    active = c.take<uint8_t>(Bz);
    n_active = c.take<int>(1);
    reached = c.take<uint8_t>(Bz);
    ticks = c.take<int32_t>(Bz);
    path_length = c.take<double>(Bz);
    min_dist = c.take<double>(Bz);
    intimate = c.take<int32_t>(Bz);
    personal = c.take<int32_t>(Bz);
    collision = c.take<int32_t>(Bz);
    not_opt = c.take<int32_t>(Bz);
    cmd_var = c.take<double>(Bz);
    pose_log = c.take<double>(logs_pose ? Bz * (T + 1) * 3 : 0);
    cmd_log = c.take<double>(logs_cmd ? Bz * T * 2 : 0);
    opt_log = c.take<uint8_t>(logs_opt ? Bz * T : 0);
    if (reactive) {  // people holds the crowd's state of the current tick
      goals = c.take<double>(Sz * Kz * 2);
      vdes = c.take<double>(Sz * Kz);
      has_goal = c.take<uint8_t>(Sz * Kz);
      disturbance = c.take<double>(Bz);
      people_log = c.take<double>(logs_people ? Sz * (T + 1) * Kz * 5 : 0);
    }
    if (w) {
      weights = c.take<double>((size_t)w->n_sets * 9);
      weight_set = c.take<int32_t>(Bz);
    }
    if (scene) {
      view = c.take<double>(Bz * n_view * 5);
      view_n = c.take<int32_t>(Bz);
      robot_min = c.take<double>(Bz);
      robot_intimate = c.take<int32_t>(Bz);
    }
    if (perceive) {
      seen = c.take<double>(tracked ? 0 : Bz * Lz * 5);
      seen_n = c.take<int32_t>(tracked ? 0 : Bz);
      unseen = c.take<int32_t>(Bz);
      stream_idx = c.take<int32_t>(pc->stream_index ? Bz : 0);
      seen_log = c.take<double>(logs_seen ? Bz * T * Lz * 5 : 0);
      n_seen_log = c.take<int32_t>(logs_seen ? Bz * T : 0);
    }
    if (tracked) {
      trk_x = c.take<double>(Bz * Mz);
      trk_y = c.take<double>(Bz * Mz);
      trk_vx = c.take<double>(Bz * Mz);
      trk_vy = c.take<double>(Bz * Mz);
      trk_pp = c.take<double>(Bz * Mz);
      trk_pv = c.take<double>(Bz * Mz);
      trk_vv = c.take<double>(Bz * Mz);
      trk_hits = c.take<int32_t>(Bz * Mz);
      trk_misses = c.take<int32_t>(Bz * Mz);
      ring = c.take<double>(Dz * Bz * Lz * 5);
      ring_n = c.take<int32_t>(Dz * Bz);
      ring_id = c.take<int32_t>(Dz * Bz * Lz);
      untracked = c.take<int32_t>(Bz);
      track_rows = c.take<int32_t>(Bz);
      pos_err = c.take<double>(Bz);
      vel_err = c.take<double>(Bz);
      id_log = c.take<int32_t>(logs_seen ? Bz * T * Lz : 0);
    }
    if (local) {
      windows = c.take<uint8_t>(Bz * cells);
      window_org = c.take<double>(Bz * 2);
      stencil_dev = c.take<uint8_t>(stencil.size());
      marked = c.take<int32_t>(Bz);
      window_log = c.take<uint8_t>(logs_local ? Bz * n_builds * cells : 0);
      window_org_log = c.take<double>(logs_local ? Bz * n_builds * 2 : 0);
    }
  };
  size_t need = 0;
  {
    smpc_carve probe(nullptr);
    carve(probe);
    need = probe.off;
  }
  SMPC_FLEET_CUDA(fs->scratch.reserve(need));
  smpc_carve cs(fs->scratch.ptr);
  carve(cs);

  // ---- inputs up (the only host-to-device copies of the call)
  struct Up { void* dev; const void* host; size_t bytes; };
  const Up ups[] = {
      {maps, io->costmaps, map_bytes}, {od, io->od_indexes, od_bytes},
      {map_org, io->costmap_origin, (size_t)io->n_costmaps * 16}, {od_org, io->od_origin, (size_t)io->n_od_grids * 16},
      {map_index, io->costmap_index, Bz * 4}, {od_index, io->od_index, Bz * 4},
      {gp, io->global_path, Bz * N * 16}, {pose, io->pose, Bz * 24}, {speed, io->speed, Bz * 16},
      {people0, K > 0 ? io->people : nullptr, Sz * Kz * 40}, {n_people_dev, K > 0 ? io->n_people_each : nullptr, Sz * 4},
      {weights, w ? w->weights : nullptr, w ? (size_t)w->n_sets * 72 : 0}, {weight_set, w ? w->set_index : nullptr, Bz * 4},
      {stream_idx, perceive ? pc->stream_index : nullptr, Bz * 4},
      {stencil_dev, local ? stencil.data() : nullptr, stencil.size()},
  };
  for (const Up& u : ups)
    if (u.host && u.bytes) SMPC_FLEET_CUDA(cudaMemcpyAsync(u.dev, u.host, u.bytes, cudaMemcpyHostToDevice, st));
  if (reactive) {
    if (K > 0) {
      SMPC_FLEET_CUDA(cudaMemcpyAsync(people, io->people, Sz * Kz * 40, cudaMemcpyHostToDevice, st));
      SMPC_FLEET_CUDA(cudaMemcpyAsync(goals, crowd->goals, Sz * Kz * 16, cudaMemcpyHostToDevice, st));
      SMPC_FLEET_CUDA(cudaMemcpyAsync(vdes, crowd->desired_speed, Sz * Kz * 8, cudaMemcpyHostToDevice, st));
      SMPC_FLEET_CUDA(cudaMemsetAsync(has_goal, 1, Sz * Kz, st));
    }
    SMPC_FLEET_CUDA(cudaMemsetAsync(disturbance, 0, Bz * 8, st));
  }
  SMPC_FLEET_CUDA(cudaMemsetAsync(active, 1, Bz, st));
  SMPC_FLEET_CUDA(cudaMemsetAsync(fov_people, 0, Bz * A * 40, st));
  SMPC_FLEET_CUDA(cudaMemsetAsync(fov_n, 0, Bz * 4, st));  // K == 0: nobody to filter, n_people stays 0
  if (perceive) SMPC_FLEET_CUDA(cudaMemsetAsync(unseen, 0, Bz * 4, st));
  if (local) SMPC_FLEET_CUDA(cudaMemsetAsync(marked, 0, Bz * 4, st));
  if (tracked) {  // no tracks, and nothing published before tick 0
    SMPC_FLEET_CUDA(cudaMemsetAsync(trk_hits, 0, Bz * Mz * 4, st));
    SMPC_FLEET_CUDA(cudaMemsetAsync(trk_misses, 0, Bz * Mz * 4, st));
    for (double* p : {trk_x, trk_y, trk_vx, trk_vy, trk_pp, trk_pv, trk_vv})
      SMPC_FLEET_CUDA(cudaMemsetAsync(p, 0, Bz * Mz * 8, st));
    SMPC_FLEET_CUDA(cudaMemsetAsync(ring_n, 0, Dz * Bz * 4, st));
    SMPC_FLEET_CUDA(cudaMemsetAsync(untracked, 0, Bz * 4, st));
    SMPC_FLEET_CUDA(cudaMemsetAsync(track_rows, 0, Bz * 4, st));
    SMPC_FLEET_CUDA(cudaMemsetAsync(pos_err, 0, Bz * 8, st));
    SMPC_FLEET_CUDA(cudaMemsetAsync(vel_err, 0, Bz * 8, st));
  }
  SMPC_FLEET_CUDA(fs->pin_out.reserve(sizeof(int)));
  int* host_active = static_cast<int*>(fs->pin_out.ptr);
  *host_active = B;
  SMPC_FLEET_CUDA(cudaMemcpyAsync(n_active, host_active, sizeof(int), cudaMemcpyHostToDevice, st));

  d.n_costmaps = io->n_costmaps; d.size_x = io->size_x; d.size_y = io->size_y; d.resolution = io->resolution;
  d.maps = maps; d.map_org = map_org; d.map_index = io->costmap_index ? map_index : nullptr;
  d.n_od_grids = io->n_od_grids; d.od_width = io->od_width; d.od_height = io->od_height;
  d.od_resolution = io->od_resolution; d.od = od; d.od_org = od_org; d.od_index = io->od_index ? od_index : nullptr;
  d.people = fov_people; d.n_people = fov_n; d.speed = speed;
  d.weights = weights; d.weight_set = weight_set;

  smpc_trajectorize_args ta{};
  ta.n_problems = B; ta.n_path = N; ta.max_steps = max_steps; ta.omnidirectional = 0;
  ta.desired_linear_vel = prm->traj_desired_linear_vel; ta.lookahead_dist = prm->lookahead_dist;
  ta.max_angular_vel = prm->max_angular_vel; ta.time_step = traj_dt;
  ta.global_path = gp; ta.path_index = nullptr; ta.pose = pose; ta.poses = d.poses; ta.cmds = seed_cmds; ta.n_steps = n_steps;

  smpc_fov_args fa{};
  fa.n_robots = B; fa.n_in_max = scene ? n_view : K; fa.n_out_max = A; fa.n_costmaps = io->n_costmaps;
  fa.size_x = io->size_x; fa.size_y = io->size_y; fa.resolution = io->resolution; fa.fov_angle = prm->fov_angle;
  fa.people_in = scene ? view : people; fa.n_people_in = scene ? view_n : n_people_dev; fa.pose = pose;
  fa.costmap_origin = map_org;
  fa.costmap_index = d.map_index; fa.people_out = fov_people; fa.n_people_out = fov_n;

  smpc_perception_args pa{};
  if (perceive) {  // between the list and the FOV filter, which then reads what the sensor reports
    pa.B = B; pa.R = R; pa.K = K; pa.L = n_list; pa.T = T;
    pa.max_range = pc->max_range; pa.occluder_r2 = pc->occluder_radius * pc->occluder_radius;
    pa.detect_prob = pc->detect_prob; pa.pos_noise = pc->pos_noise; pa.vel_noise = pc->vel_noise;
    pa.occluding_cost = pc->occluding_cost; pa.seed = pc->seed;
    pa.active = active; pa.pose = pose; pa.list = fa.people_in; pa.n_list = fa.n_people_in;
    pa.stream_index = pc->stream_index ? stream_idx : nullptr;
    pa.maps = maps; pa.map_org = map_org; pa.map_index = d.map_index;
    pa.n_costmaps = io->n_costmaps; pa.size_x = io->size_x; pa.size_y = io->size_y; pa.resolution = io->resolution;
    pa.seen = seen; pa.n_seen = seen_n; pa.unseen = unseen;
    pa.seen_log = logs_seen ? seen_log : nullptr; pa.n_seen_log = logs_seen ? n_seen_log : nullptr;
    fa.people_in = seen; fa.n_people_in = seen_n;
  }
  smpc_tracker_args tka{};
  if (tracked) {  // the FOV filter reads a ring slot instead, switched every tick
    tka.p = pa;
    tka.p.seen = nullptr; tka.p.n_seen = nullptr;
    tka.M = (int)Mz; tka.confirm_hits = tk->confirm_hits; tka.max_coast = tk->max_coast_ticks;
    tka.dt = io->control_period; tka.accel_noise = tk->accel_noise; tka.meas_noise = tk->meas_noise;
    tka.init_vel_std = tk->init_vel_std;
    tka.px = trk_x; tka.py = trk_y; tka.vx = trk_vx; tka.vy = trk_vy;
    tka.p_pp = trk_pp; tka.p_pv = trk_pv; tka.p_vv = trk_vv; tka.hits = trk_hits; tka.misses = trk_misses;
    tka.untracked = untracked; tka.track_rows = track_rows; tka.pos_err = pos_err; tka.vel_err = vel_err;
    tka.id_log = logs_seen ? id_log : nullptr;
  }

  // with a crowd the prep moves nobody (K = 0 there): the crowd step does
  EpisodePrep pp{B, reactive ? 0 : K, stride, max_steps, maxsize, 0.0, n_steps, seed_cmds, active, people0, people, d.poses, d.cmds,
                 const_cast<int32_t*>(d.n_in), const_cast<int32_t*>(d.n_each), const_cast<int32_t*>(d.s_each)};
  EpisodeStep es{};
  es.B = B; es.R = R; es.K = K; es.T = T; es.stride = stride; es.n_path = N;
  es.dt_c = io->control_period; es.goal_tol = io->goal_tolerance;
  es.cmds = d.cmds; es.optimized = d.optimized; es.people0 = people0; es.n_people = K > 0 ? n_people_dev : nullptr;
  es.global_path = gp; es.maps = maps; es.map_org = map_org; es.map_index = d.map_index;
  es.n_costmaps = io->n_costmaps; es.size_x = io->size_x; es.size_y = io->size_y; es.resolution = io->resolution;
  es.pose = pose; es.speed = speed; es.active = active; es.n_active = n_active;
  es.reached = reached; es.ticks = ticks; es.path_length = path_length; es.min_dist = min_dist;
  es.intimate = intimate; es.personal = personal; es.collision = collision; es.not_optimized = not_opt;
  es.cmd_variation = cmd_var;
  es.people_now = reactive ? people : nullptr;
  es.pose_log = logs_pose ? pose_log : nullptr;
  es.cmd_log = logs_cmd ? cmd_log : nullptr;
  es.optimized_log = logs_opt ? opt_log : nullptr;

  smpc_crowd_step_args ca{};
  if (reactive) {
    ca.B = S; ca.R = R; ca.K = K; ca.T = T; ca.stride = stride; ca.substeps = crowd->substeps; ca.dt_c = io->control_period;
    ca.active = active; ca.n_people = n_people_dev; ca.pose = pose; ca.cmds = d.cmds; ca.goals = goals; ca.vdes = vdes;
    ca.has_goal = has_goal; ca.people = people; ca.disturbance = disturbance;
    ca.people_log = logs_people ? people_log : nullptr;
    ca.n_od_grids = io->n_od_grids; ca.od_width = io->od_width; ca.od_height = io->od_height;
    ca.od_resolution = io->od_resolution; ca.od = od; ca.od_org = od_org; ca.od_index = d.od_index;
  }

  smpc_local_costmap_args la{};
  if (local) {  // built from the true list, before perception; the FOV filter and the fleet tick read the windows
    la.B = B; la.sx = local->size_x; la.sy = local->size_y; la.half = half; la.L = n_list; la.n_builds = n_builds;
    la.active = active; la.pose = pose; la.list = scene ? view : people;
    la.n_list = local->mark_people && fov ? (scene ? view_n : n_people_dev) : nullptr;
    la.stencil = stencil_dev; la.maps = maps; la.map_org = map_org; la.map_index = d.map_index;
    la.n_costmaps = io->n_costmaps; la.size_x = io->size_x; la.size_y = io->size_y; la.resolution = io->resolution;
    la.window = windows; la.origin = window_org; la.marked = marked;
    la.window_log = logs_local ? window_log : nullptr; la.origin_log = logs_local ? window_org_log : nullptr;
    d.maps = windows; d.map_org = window_org; d.map_index = nullptr;
    d.n_costmaps = B; d.size_x = local->size_x; d.size_y = local->size_y;
    fa.costmap_origin = window_org; fa.costmap_index = nullptr;
    fa.n_costmaps = B; fa.size_x = local->size_x; fa.size_y = local->size_y;
  }

  const SceneView sv{B, R, K, n_view, active, pose, speed, people, K > 0 ? n_people_dev : nullptr, view, view_n};
  RobotMetrics rm{B, R, 0, pose, ticks, robot_min, robot_intimate};

  const int prep_rows = stride > pp.K ? stride : pp.K;
  const unsigned g_prep = (unsigned)((Bz * prep_rows + 255) / 256), g_step = (unsigned)((Bz + 3) / 4);
  const unsigned g_view = (unsigned)((Bz * n_view + 255) / 256), g_robots = (unsigned)((Bz + 255) / 256);
  for (int k = 0; k < T; ++k) {
    rc = smpc_trajectorize_batch_device(h, &ta, st);
    if (rc != SMPC_OK) return rc;
    pp.t = (double)k * io->control_period;
    smpc_episode_prep_kernel<<<g_prep, 256, 0, st>>>(pp);
    SMPC_FLEET_CUDA(cudaGetLastError());
    smpc_handle_count_launch(h);
    if (scene && fov) {
      smpc_scene_view_kernel<<<g_view, 256, 0, st>>>(sv);
      SMPC_FLEET_CUDA(cudaGetLastError());
      smpc_handle_count_launch(h);
    }
    if (tracked) {  // publish into slot k mod D; the FOV filter reads slot (k - latency) mod D
      const size_t sp = (size_t)k % Dz, sd = (size_t)(k + 1) % Dz;
      tka.p.k = k;
      tka.pub = ring + sp * Bz * Lz * 5; tka.pub_n = ring_n + sp * Bz; tka.pub_id = ring_id + sp * Bz * Lz;
      tka.del = ring + sd * Bz * Lz * 5; tka.del_n = ring_n + sd * Bz; tka.del_id = ring_id + sd * Bz * Lz;
      fa.people_in = tka.del; fa.n_people_in = tka.del_n;
      rc = smpc_tracked_perception_enqueue(h, tka, st);
      if (rc != SMPC_OK) return rc;
    } else if (perceive) {
      pa.k = k;
      rc = smpc_perception_enqueue(h, pa, st);
      if (rc != SMPC_OK) return rc;
    }
    if (local && k % n_period == 0) {
      la.build = k / n_period;
      rc = smpc_local_costmap_enqueue(h, la, st);
      if (rc != SMPC_OK) return rc;
    }
    if (fov) {
      rc = smpc_fov_filter_batch_device(h, &fa, st);
      if (rc != SMPC_OK) return rc;
    }
    rc = smpc_fleet_tick_enqueue(h, d, st);
    if (rc != SMPC_OK) return rc;
    if (reactive) {
      ca.k = k;
      rc = orca ? smpc_orca_step_enqueue(h, ca, *orca, st) : smpc_crowd_step_enqueue(h, ca, st);
      if (rc != SMPC_OK) return rc;
    }
    es.k = k;
    smpc_episode_step_kernel<<<g_step, 128, 0, st>>>(es);
    SMPC_FLEET_CUDA(cudaGetLastError());
    smpc_handle_count_launch(h);
    if (scene) {  // needs every robot's pose at k + 1
      rm.k = k;
      smpc_robot_metrics_kernel<<<g_robots, 256, 0, st>>>(rm);
      SMPC_FLEET_CUDA(cudaGetLastError());
      smpc_handle_count_launch(h);
    }
    if ((k + 1) % kPollTicks == 0 && k + 1 < T) {
      SMPC_FLEET_CUDA(cudaMemcpyAsync(host_active, n_active, sizeof(int), cudaMemcpyDeviceToHost, st));
      SMPC_FLEET_CUDA(cudaStreamSynchronize(st));
      if (*host_active == 0) break;
    }
  }

  // ---- results down
  struct Down { void* host; const void* dev; size_t bytes; };
  const Down downs[] = {
      {io->reached, reached, Bz}, {io->ticks, ticks, Bz * 4}, {io->path_length, path_length, Bz * 8},
      {io->min_person_dist, min_dist, Bz * 8}, {io->intimate_ticks, intimate, Bz * 4},
      {io->personal_ticks, personal, Bz * 4}, {io->collision_ticks, collision, Bz * 4},
      {io->not_optimized_ticks, not_opt, Bz * 4}, {io->cmd_variation, cmd_var, Bz * 8},
      {logs_pose ? io->pose_log : nullptr, pose_log, Bz * (T + 1) * 24},
      {logs_cmd ? io->cmd_log : nullptr, cmd_log, Bz * T * 16},
      {logs_opt ? io->optimized_log : nullptr, opt_log, Bz * T},
      {reactive ? crowd->people_disturbance : nullptr, disturbance, Bz * 8},
      {logs_people ? crowd->people_log : nullptr, people_log, Sz * (T + 1) * Kz * 40},
      {scene ? scene->robot_min_dist : nullptr, robot_min, Bz * 8},
      {scene ? scene->robot_intimate_ticks : nullptr, robot_intimate, Bz * 4},
      {perceive ? pc->unseen_personal_ticks : nullptr, unseen, Bz * 4},
      {logs_seen ? pc->seen_log : nullptr, seen_log, Bz * T * Lz * 40},
      {logs_seen ? pc->n_seen_log : nullptr, n_seen_log, Bz * T * 4},
      {tracked ? tk->untracked_personal_ticks : nullptr, untracked, Bz * 4},
      {tracked ? tk->track_rows : nullptr, track_rows, Bz * 4},
      {tracked ? tk->track_pos_err : nullptr, pos_err, Bz * 8},
      {tracked ? tk->track_vel_err : nullptr, vel_err, Bz * 8},
      {tracked && logs_seen ? tk->track_id_log : nullptr, id_log, Bz * T * Lz * 4},
      {local ? local->marked_rows : nullptr, marked, Bz * 4},
      {logs_local ? local->costmap_log : nullptr, window_log, Bz * n_builds * cells},
      {logs_local ? local->origin_log : nullptr, window_org_log, Bz * n_builds * 16},
  };
  for (const Down& c : downs)
    if (c.host) SMPC_FLEET_CUDA(cudaMemcpyAsync(c.host, c.dev, c.bytes, cudaMemcpyDeviceToHost, st));
  SMPC_FLEET_CUDA(cudaStreamSynchronize(st));

  // log rows after an episode is done were never written on the device: final pose, zero cmd / optimized
  for (int b = 0; b < B; ++b) {
    const int tb = io->ticks[b];
    if (logs_pose)
      for (int k = tb + 1; k <= T; ++k)
        std::memcpy(io->pose_log + ((size_t)b * (T + 1) + k) * 3, io->pose_log + ((size_t)b * (T + 1) + tb) * 3, 24);
    if (logs_cmd) std::memset(io->cmd_log + ((size_t)b * T + tb) * 2, 0, (size_t)(T - tb) * 16);
    if (logs_opt) std::memset(io->optimized_log + (size_t)b * T + tb, 0, (size_t)(T - tb));
    if (logs_seen) {
      std::memset(pc->seen_log + ((size_t)b * T + tb) * Lz * 5, 0, (size_t)(T - tb) * Lz * 40);
      std::memset(pc->n_seen_log + (size_t)b * T + tb, 0, (size_t)(T - tb) * 4);
    }
    if (tracked && logs_seen) std::fill_n(tk->track_id_log + ((size_t)b * T + tb) * Lz, (size_t)(T - tb) * Lz, -1);
    if (logs_local) {  // builds at ticks j * n_period >= tb never ran
      const int jb = (tb + n_period - 1) / n_period;
      std::memset(local->costmap_log + ((size_t)b * n_builds + jb) * cells, 0, (size_t)(n_builds - jb) * cells);
      std::fill_n(local->origin_log + ((size_t)b * n_builds + jb) * 2, (size_t)(n_builds - jb) * 2, (double)NAN);
    }
  }
  if (pc && !perceive) {  // no list: nothing reported, nobody missed
    std::memset(pc->unseen_personal_ticks, 0, Bz * 4);
    if (pc->n_seen_log) std::memset(pc->n_seen_log, 0, Bz * T * 4);
  }
  if (tk && !perceive) {  // no list: nothing tracked, nobody missed
    std::memset(tk->untracked_personal_ticks, 0, Bz * 4);
    std::memset(tk->track_rows, 0, Bz * 4);
    std::memset(tk->track_pos_err, 0, Bz * 8);
    std::memset(tk->track_vel_err, 0, Bz * 8);
  }
  for (int c = 0; c < S && logs_people; ++c) {  // the people of a finished scene stand where they were at its last tick
    int tc = 0;
    for (int r = 0; r < R; ++r) tc = std::max(tc, (int)io->ticks[c * R + r]);
    for (int k = tc + 1; k <= T; ++k)
      std::memcpy(crowd->people_log + ((size_t)c * (T + 1) + k) * Kz * 5,
                  crowd->people_log + ((size_t)c * (T + 1) + tc) * Kz * 5, Kz * 40);
  }
  return SMPC_OK;
}

}  // namespace

extern "C" int smpc_run_episodes(smpc_handle* h, smpc_episode_io* io) {
  return run_episodes(h, io, nullptr, nullptr, "run_episodes");
}

extern "C" int smpc_run_crowd_episodes(smpc_handle* h, smpc_episode_io* io, const smpc_crowd_io* crowd) {
  if (!crowd) return smpc_host_fail(SMPC_ERR_ARGUMENT, "run_crowd_episodes: NULL crowd");
  return run_episodes(h, io, crowd, nullptr, "run_crowd_episodes");
}

extern "C" int smpc_run_shared_episodes(smpc_handle* h, smpc_episode_io* io, const smpc_crowd_io* crowd,
                                        const smpc_scene_io* scene) {
  if (!crowd) return smpc_host_fail(SMPC_ERR_ARGUMENT, "run_shared_episodes: NULL crowd");
  if (!scene) return smpc_host_fail(SMPC_ERR_ARGUMENT, "run_shared_episodes: NULL scene");
  return run_episodes(h, io, crowd, scene, "run_shared_episodes");
}

extern "C" int smpc_run_weighted_episodes(smpc_handle* h, smpc_episode_io* io, const smpc_crowd_io* crowd,
                                          const smpc_scene_io* scene, const smpc_weight_sets* w) {
  const int rc = smpc_check_weight_sets(w, 0, "run_weighted_episodes");  // the indices: once B is known
  if (rc != SMPC_OK) return rc;
  if (scene && !crowd) return smpc_host_fail(SMPC_ERR_ARGUMENT, "run_weighted_episodes: a shared scene needs a crowd");
  return run_episodes(h, io, crowd, scene, "run_weighted_episodes", w);
}

namespace {

// SMPC_ERR_ARGUMENT unless the ORCA parameters are in range (`name` prefixes the message)
int check_orca_params(const smpc_orca_params* orca, const char* name) {
  auto fail_arg = [name](const char* msg) {
    return smpc_host_fail(SMPC_ERR_ARGUMENT, std::string(name) + ": " + msg);
  };
  auto positive = [](double x) { return std::isfinite(x) && x > 0.0; };
  if (!positive(orca->neighbor_dist) || !positive(orca->time_horizon) || !positive(orca->time_horizon_obst) ||
      !positive(orca->person_radius) || !positive(orca->robot_radius))
    return fail_arg("a distance, horizon or radius not finite and > 0");
  if (orca->max_neighbors < 1 || orca->max_neighbors > 16) return fail_arg("max_neighbors outside 1..16");
  if (!(orca->robot_responsibility >= 0.0 && orca->robot_responsibility <= 1.0))
    return fail_arg("robot_responsibility outside [0, 1]");
  return SMPC_OK;
}

// SMPC_ERR_ARGUMENT unless the perception parameters are in range and the outputs given (the stream indices: once B is
// known)
int check_perception(const smpc_perception* pc, const char* name) {
  auto fail_arg = [name](const char* msg) {
    return smpc_host_fail(SMPC_ERR_ARGUMENT, std::string(name) + ": " + msg);
  };
  if (!(pc->max_range > 0.0)) return fail_arg("max_range not > 0");
  if (!(std::isfinite(pc->occluder_radius) && pc->occluder_radius >= 0.0))
    return fail_arg("occluder_radius not finite and >= 0");
  if (pc->occluding_cost < 0 || pc->occluding_cost > 255) return fail_arg("occluding_cost outside 0..255");
  if (!(pc->detect_prob >= 0.0 && pc->detect_prob <= 1.0)) return fail_arg("detect_prob outside [0, 1]");
  if (!(std::isfinite(pc->pos_noise) && pc->pos_noise >= 0.0) || !(std::isfinite(pc->vel_noise) && pc->vel_noise >= 0.0))
    return fail_arg("pos_noise or vel_noise not finite and >= 0");
  if (!pc->unseen_personal_ticks) return fail_arg("missing output");
  if ((pc->seen_log == nullptr) != (pc->n_seen_log == nullptr)) return fail_arg("seen_log and n_seen_log not given together");
  return SMPC_OK;
}

// SMPC_ERR_ARGUMENT unless the tracker parameters are in range, the perception gives positions only and the outputs
// are given
int check_tracker(const smpc_tracker* tk, const smpc_perception* pc, const char* name) {
  auto fail_arg = [name](const char* msg) {
    return smpc_host_fail(SMPC_ERR_ARGUMENT, std::string(name) + ": " + msg);
  };
  if (!(std::isfinite(tk->accel_noise) && tk->accel_noise >= 0.0)) return fail_arg("accel_noise not finite and >= 0");
  if (!(std::isfinite(tk->meas_noise) && tk->meas_noise > 0.0) ||
      !(std::isfinite(tk->init_vel_std) && tk->init_vel_std > 0.0))
    return fail_arg("meas_noise or init_vel_std not finite and > 0");
  if (tk->confirm_hits < 1 || tk->confirm_hits > 16) return fail_arg("confirm_hits outside 1..16");
  if (tk->max_coast_ticks < 0 || tk->max_coast_ticks > 64) return fail_arg("max_coast_ticks outside 0..64");
  if (tk->latency_ticks < 0 || tk->latency_ticks > 16) return fail_arg("latency_ticks outside 0..16");
  if (pc->vel_noise != 0.0) return fail_arg("perception vel_noise not 0 (the tracker estimates velocities itself)");
  if (!tk->untracked_personal_ticks || !tk->track_rows || !tk->track_pos_err || !tk->track_vel_err)
    return fail_arg("missing output");
  if ((tk->track_id_log == nullptr) != (pc->seen_log == nullptr))
    return fail_arg("track_id_log and seen_log not given together");
  return SMPC_OK;
}

}  // namespace

extern "C" int smpc_run_orca_episodes(smpc_handle* h, smpc_episode_io* io, const smpc_crowd_io* crowd,
                                      const smpc_scene_io* scene, const smpc_weight_sets* w,
                                      const smpc_orca_params* orca) {
  auto fail_arg = [](const char* msg) {
    return smpc_host_fail(SMPC_ERR_ARGUMENT, std::string("run_orca_episodes: ") + msg);
  };
  if (!orca) return fail_arg("NULL orca");
  if (!crowd) return fail_arg("NULL crowd");
  const int orc = check_orca_params(orca, "run_orca_episodes");
  if (orc != SMPC_OK) return orc;
  if (w) {
    const int rc = smpc_check_weight_sets(w, 0, "run_orca_episodes");  // the indices: once B is known
    if (rc != SMPC_OK) return rc;
  }
  return run_episodes(h, io, crowd, scene, "run_orca_episodes", w, orca);
}

namespace {

// smpc_run_perceived_episodes (tk == NULL), smpc_run_tracked_episodes and smpc_run_local_costmap_episodes: the argument
// checks that need no B (perception may be NULL only with local given; the local costmap's fields: once the
// resolution is checked)
int run_perceived(smpc_handle* h, smpc_episode_io* io, const smpc_crowd_io* crowd, const smpc_scene_io* scene,
                  const smpc_weight_sets* w, const smpc_orca_params* orca, const smpc_perception* perception,
                  const smpc_tracker* tk, const char* name, const smpc_local_costmap* local = nullptr) {
  auto fail_arg = [name](const char* msg) {
    return smpc_host_fail(SMPC_ERR_ARGUMENT, std::string(name) + ": " + msg);
  };
  if (!perception && !local) return fail_arg("NULL perception");
  int rc = SMPC_OK;
  if (perception) {
    rc = check_perception(perception, name);
    if (rc != SMPC_OK) return rc;
  }
  if (tk) {
    if (!perception) return fail_arg("a tracker needs perception");
    rc = check_tracker(tk, perception, name);
    if (rc != SMPC_OK) return rc;
  }
  if (local) {
    if (!local->marked_rows) return fail_arg("missing output");
    if ((local->costmap_log == nullptr) != (local->origin_log == nullptr))
      return fail_arg("costmap_log and origin_log not given together");
  }
  if (scene && !crowd) return fail_arg("a shared scene needs a crowd");
  if (orca && !crowd) return fail_arg("an ORCA crowd needs a crowd");
  if (orca) {
    rc = check_orca_params(orca, name);
    if (rc != SMPC_OK) return rc;
  }
  if (w) {
    rc = smpc_check_weight_sets(w, 0, name);  // the indices: once B is known
    if (rc != SMPC_OK) return rc;
  }
  return run_episodes(h, io, crowd, scene, name, w, orca, perception, tk, local);
}

}  // namespace

extern "C" int smpc_run_perceived_episodes(smpc_handle* h, smpc_episode_io* io, const smpc_crowd_io* crowd,
                                           const smpc_scene_io* scene, const smpc_weight_sets* w,
                                           const smpc_orca_params* orca, const smpc_perception* perception) {
  return run_perceived(h, io, crowd, scene, w, orca, perception, nullptr, "run_perceived_episodes");
}

extern "C" int smpc_run_tracked_episodes(smpc_handle* h, smpc_episode_io* io, const smpc_crowd_io* crowd,
                                         const smpc_scene_io* scene, const smpc_weight_sets* w,
                                         const smpc_orca_params* orca, const smpc_perception* perception,
                                         const smpc_tracker* tracker) {
  if (!tracker) return smpc_host_fail(SMPC_ERR_ARGUMENT, "run_tracked_episodes: NULL tracker");
  return run_perceived(h, io, crowd, scene, w, orca, perception, tracker, "run_tracked_episodes");
}

extern "C" int smpc_run_local_costmap_episodes(smpc_handle* h, smpc_episode_io* io, const smpc_crowd_io* crowd,
                                               const smpc_scene_io* scene, const smpc_weight_sets* w,
                                               const smpc_orca_params* orca, const smpc_perception* perception,
                                               const smpc_tracker* tracker, const smpc_local_costmap* local) {
  if (!local) return smpc_host_fail(SMPC_ERR_ARGUMENT, "run_local_costmap_episodes: NULL local costmap");
  return run_perceived(h, io, crowd, scene, w, orca, perception, tracker, "run_local_costmap_episodes", local);
}
