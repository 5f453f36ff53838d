// smpc_host_state.h — internal accessors shared by the host translation units of libsmpc.so.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/smpc.h"

// per-handle stand-in for the reference's process-wide TrajectoryMemory singleton (trajectory_memory.hpp)
struct smpc_memory {
  std::vector<double> prev_poses;  // [n][3]
  std::vector<double> prev_cmds;   // [n][2]
};

// growing device allocation
struct smpc_devbuf {
  void* ptr = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    cap = 0;
    const size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMalloc(&ptr, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    cap = 0;
  }
};

// growing page-locked host allocation
struct smpc_pinbuf {
  void* ptr = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (ptr) cudaFreeHost(ptr);
    ptr = nullptr;
    cap = 0;
    const size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaHostAlloc(&ptr, want, cudaHostAllocDefault);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (ptr) cudaFreeHost(ptr);
    ptr = nullptr;
    cap = 0;
  }
};

// device-resident state of the fleet tick (smpc_optimize_batch): per-robot TrajectoryMemory, cached maps, scratch
struct smpc_fleet_state {
  std::mutex mu;
  smpc_devbuf scratch, maps, memory;
  smpc_pinbuf pin_in, pin_out, pin_maps;  // staging of small ticks: one copy per direction (see smpc_optimize_batch_on)
  int mem_robots = 0, mem_stride = 0;
  long long maps_version = -1;
  size_t maps_bytes = 0;
  std::vector<int32_t> host_n_each, host_s_each;
  void forget() { mem_robots = mem_stride = 0; }
  void release() {
    scratch.release();
    maps.release();
    memory.release();
    pin_in.release();
    pin_out.release();
    pin_maps.release();
    forget();
    maps_version = -1;
  }
};

// consecutive 256-byte aligned sub-buffers of one allocation (base NULL: only count the bytes)
struct smpc_carve {
  char* base;
  size_t off = 0;
  explicit smpc_carve(void* b) : base(static_cast<char*>(b)) {}
  template <class T>
  T* take(size_t count) {
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += (count * sizeof(T) + 255) & ~static_cast<size_t>(255);
    return p;
  }
};

// Device buffers of one fleet tick (all device pointers; rows of poses / cmds / robot / path have `stride` entries).
struct smpc_fleet_dev {
  int B, stride, A, nb;
  float time_step, max_time;
  // maps
  int n_costmaps, size_x, size_y;
  double resolution;
  const uint8_t* maps;
  const double* map_org;
  const int32_t* map_index;  // may be NULL
  int n_od_grids;
  uint32_t od_width, od_height;
  float od_resolution;
  const uint32_t* od;
  const double* od_org;
  const int32_t* od_index;  // may be NULL
  // per robot: poses in n_in, after the max_time cut n_each (0 = inactive) and s_each = n_each - 1 (1 when inactive)
  const int32_t* n_in;
  const int32_t* n_each;
  const int32_t* s_each;
  const double* people;  // [B][A][5]
  const int32_t* n_people;
  const double* speed;
  double* poses;  // in: seed, out: result
  double* cmds;
  // warm-start memory (smpc_fleet_memory)
  double* prev_poses;
  double* prev_cmds;
  int32_t* n_prev_poses;
  int32_t* n_prev_cmds;
  // stage buffers and outputs (smpc_fleet_carve_stages)
  double *init, *robot, *pose0, *u0, *path_xy, *goal_yaw, *agents, *cmds_new, *path_new, *cost0, *cost1;
  uint8_t *has_people, *usable, *optimized;
  int32_t *term, *iters, *n_out, *status;
  // per-robot critic weights (NULL = the handle's): robot b's critics use row weight_set[b] of weights [P][9]
  const double* weights;
  const int32_t* weight_set;
};

// Carves the stage buffers and outputs of smpc_fleet_dev (init .. path_new, then usable .. status) from c.
void smpc_fleet_carve_stages(smpc_carve& c, smpc_fleet_dev* d);
// Points d's memory fields at fs's per-robot warm-start memory for d->B robots of d->stride poses; (re-)creates it
// zeroed (= no memory yet) when the shape changed or after fs->forget().
cudaError_t smpc_fleet_memory(smpc_fleet_state* fs, smpc_fleet_dev* d, cudaStream_t st);
// Enqueues one fleet tick on st: memory seeding, people_to_status, format_to_optimize, project_people, the solve and
// the finish (outputs, memory update). No host synchronisation.
int smpc_fleet_tick_enqueue(smpc_handle* h, const smpc_fleet_dev& d, cudaStream_t st);

// One controller tick of the reactive crowd of smpc_run_crowd_episodes / smpc_run_shared_episodes (smpc_crowd.cu), all
// device pointers. B scenes of R robots each: robot r of scene b is robot b * R + r (R = 1: one robot per scene).
struct smpc_crowd_step_args {
  int B, R, K, T, k, stride, substeps;
  double dt_c;
  const uint8_t* active;       // [B*R] robots still running; a scene none of whose robots runs keeps its people
  const int32_t* n_people;     // [B] people of each scene (<= K)
  const double* pose;          // [B*R][3] robot pose of tick k
  const double* cmds;          // [B*R][stride][2] fleet tick output: row 0 is the command of tick k
  const double* goals;         // [B][K][2]
  const double* vdes;          // [B][K]
  uint8_t* has_goal;           // [B][K] lightsfm goal flags
  double* people;              // [B][K][5] in: tick k, out: tick k + 1
  double* disturbance;         // [B*R] accumulated while the robot runs
  double* people_log;          // [B][T+1][K][5] or NULL
  int n_od_grids;
  uint32_t od_width, od_height;
  float od_resolution;
  const uint32_t* od;
  const double* od_org;
  const int32_t* od_index;     // [B*R], equal within a scene, or NULL (grid (b * R) % n_od_grids)
};
// Enqueues smpc_crowd_step_kernel on st (one launch).
int smpc_crowd_step_enqueue(smpc_handle* h, const smpc_crowd_step_args& a, cudaStream_t st);
// Enqueues smpc_orca_step_kernel (smpc_orca.cu) on st (one launch): the same tick of the same crowd state, with the
// people moved by ORCA under the checked parameters o instead of the social force model.
int smpc_orca_step_enqueue(smpc_handle* h, const smpc_crowd_step_args& a, const smpc_orca_params& o, cudaStream_t st);

// One controller tick of the perception stage of smpc_run_perceived_episodes (smpc_perception.cu), all device pointers:
// robot b's list (L rows, n_list[b] of them valid) cut to the rows its sensor reports, compacted in input order.
struct smpc_perception_args {
  int B, R, K, L, T, k;           // R robots per scene (1: the list holds people only)
  double max_range, occluder_r2, detect_prob, pos_noise, vel_noise;
  int occluding_cost;
  unsigned long long seed;
  const uint8_t* active;          // [B] robots running tick k; the others report nothing (n_seen = 0)
  const double* pose;             // [B][3] robot pose of tick k
  const double* list;             // [B][L][5] the FOV filter's input without perception
  const int32_t* n_list;          // [B]
  const int32_t* stream_index;    // [B] or NULL (= b)
  const uint8_t* maps;
  const double* map_org;
  const int32_t* map_index;       // may be NULL (map b % n_costmaps)
  int n_costmaps, size_x, size_y;
  double resolution;
  double* seen;                   // [B][L][5] out: the reported rows
  int32_t* n_seen;                // [B] out
  int32_t* unseen;                // [B] += 1 when a person within 1.2 m went unreported
  double* seen_log;               // [B][T][L][5] or NULL: row k of the robots running tick k
  int32_t* n_seen_log;            // [B][T] or NULL
};
// Enqueues smpc_perception_kernel on st (one launch).
int smpc_perception_enqueue(smpc_handle* h, const smpc_perception_args& a, cudaStream_t st);

// One controller tick of the tracked perception of smpc_run_tracked_episodes (smpc_tracker.cu), all device pointers:
// the detections of the perception stage (p; its seen / n_seen are unused) update one constant-velocity Kalman track
// per agent id, the confirmed tracks are published into the ring slot of tick k, and the FOV filter reads the slot of
// tick k - latency, which p.seen_log / p.n_seen_log and id_log record.
struct smpc_tracker_args {
  smpc_perception_args p;
  int M;                          // track slots per robot: K + R in shared scenes, else K
  int confirm_hits, max_coast;
  double dt, accel_noise, meas_noise, init_vel_std;
  double *px, *py, *vx, *vy;      // [B][M] track state, zero at the start of a call
  double *p_pp, *p_pv, *p_vv;     // [B][M] the per-axis covariance both axes share
  int32_t *hits, *misses;         // [B][M]; hits == 0: no track
  double* pub;                    // [B][L][5] the ring slot of tick k: the published rows
  int32_t *pub_n, *pub_id;        // [B], [B][L]
  const double* del;              // [B][L][5] the ring slot of tick k - latency (= pub when latency is 0)
  const int32_t* del_id;          // [B][L]
  int32_t* del_n;                 // [B] (zeroed for a finished robot: the FOV filter then reads nobody)
  int32_t *untracked, *track_rows;  // [B] accumulated over the ticks a robot runs
  double *pos_err, *vel_err;      // [B]
  int32_t* id_log;                // [B][T][L] or NULL: the ids of the rows of p.seen_log
};
// Enqueues smpc_tracked_perception_kernel on st (one launch).
int smpc_tracked_perception_enqueue(smpc_handle* h, const smpc_tracker_args& a, cudaStream_t st);

// One build of the rolling local costmaps of smpc_run_local_costmap_episodes (smpc_local_costmap.cu), all device
// pointers: robot b's window of sx x sy cells around its pose of tick k, the static layer cropped from its static costmap
// and, with n_list given, the stencil splatted on the cell of every row of its true list that lies inside the window.
struct smpc_local_costmap_args {
  int B, sx, sy, half;            // window size, stencil half-width (<= 32)
  int L, build, n_builds;         // list rows; this build's index k / update_period_ticks, of n_builds
  const uint8_t* active;          // [B] robots running tick k; the others build nothing
  const double* pose;             // [B][3] robot pose of tick k
  const double* list;             // [B][L][5] true positions of the people (shared scenes: the scene view)
  const int32_t* n_list;          // [B], or NULL: no people layer
  const uint8_t* stencil;         // [2 half + 1][2 half + 1]
  const uint8_t* maps;            // the static costmaps
  const double* map_org;
  const int32_t* map_index;       // may be NULL (map b % n_costmaps)
  int n_costmaps, size_x, size_y;
  double resolution;
  uint8_t* window;                // [B][sy][sx] out
  double* origin;                 // [B][2] out
  int32_t* marked;                // [B] += rows marked
  uint8_t* window_log;            // [B][n_builds][sy][sx] or NULL
  double* origin_log;             // [B][n_builds][2] or NULL
};
// Enqueues smpc_local_costmap_kernel on st (one launch).
int smpc_local_costmap_enqueue(smpc_handle* h, const smpc_local_costmap_args& a, cudaStream_t st);
// SMPC_ERR_ARGUMENT unless every field of the smpc_local_costmap l that the build reads is in range and the stencil at
// resolution res has a half-width <= 32; then the stencil, row-major [2 half + 1]^2, and its half-width
int smpc_local_costmap_build_stencil(const smpc_local_costmap* l, double res, std::vector<uint8_t>* stencil, int* half,
                                     const char* name);

const smpc_params* smpc_handle_params(smpc_handle* h);
smpc_fleet_state* smpc_handle_fleet(smpc_handle* h);
smpc_fleet_state* smpc_handle_single(smpc_handle* h);
smpc_fleet_state* smpc_handle_episodes(smpc_handle* h);
int smpc_handle_device(smpc_handle* h);
smpc_memory* smpc_handle_memory(smpc_handle* h);
int smpc_host_fail(int code, const std::string& msg);
cudaStream_t smpc_handle_stream(smpc_handle* h);
void smpc_handle_count_launch(smpc_handle* h);
// the fleet tick on an explicit state (smpc_optimize_batch uses the handle's fleet state, smpc_optimize its own);
// w != NULL: per-robot critic weights (smpc_optimize_batch_weighted)
int smpc_optimize_batch_on(smpc_handle* h, smpc_fleet_state* fs, smpc_fleet_io* io, const smpc_weight_sets* w = nullptr);
// SMPC_ERR_ARGUMENT unless w is a valid weight table for n robots: n_sets >= 1, arrays given, every weight finite, every
// index in 0..n_sets-1 (`name` prefixes the message)
int smpc_check_weight_sets(const smpc_weight_sets* w, int n, const char* name);
// smpc_solve_batch_device with per-problem critic weights (device pointers weights [P][9], weight_set [B]): the solve
// of the fleet tick (people columns, unicycle blocks only)
int smpc_solve_batch_weighted(smpc_handle* h, const smpc_batch* in, smpc_result* out, const double* weights,
                              const int32_t* weight_set, cudaStream_t stream);

#define SMPC_FLEET_CUDA(call)                                                                              \
  do {                                                                                                     \
    cudaError_t e__ = (call);                                                                              \
    if (e__ != cudaSuccess) return smpc_host_fail(SMPC_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); \
  } while (0)
