// smpc_host.cu — host side of libsmpc.so: the C-ABI declared in include/smpc.h.
// Mirrors OptimizerParams::get / Optimizer::initialize / the ceres::Solve call of the reference
// (src/optimizer.cpp:16-132, :381) for batches of problems. No CPU compute path exists here: every
// solve / eval entry launches the sm_100a kernels of smpc_kernels.cu or returns an error.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <mutex>
#include <sstream>
#include <string>
#include <vector>

#include "../../include/smpc.h"
#include "smpc_device.cuh"
#include "smpc_host_state.h"
#include "smpc_internal.h"

namespace {

thread_local std::string g_last_error;

int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}

int cuda_fail(cudaError_t e, const char* what) {
  return fail(SMPC_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

#define SMPC_CUDA(call)                                   \
  do {                                                    \
    cudaError_t e__ = (call);                             \
    if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
  } while (0)

constexpr int kMaxChunks = 8;  // chunks of the host-buffer pipeline (one queue counter each)
constexpr int kMapChunks = 8;  // pieces the per-problem costmaps are streamed in under a running solve

struct DeviceBuffer {
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

struct PinnedBuffer {  // page-locked host staging owned by a handle
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

// Small host batches (single solves, a robot's few problems): every input array is first gathered into ONE page-locked
// staging block laid out like the device staging, so the call makes one host-to-device and one device-to-host copy
// instead of ~10 + ~9 small ones (each a driver round trip of several microseconds from pageable memory).
constexpr size_t kPackedBytes = 256u << 10;

const char* const kSolverTypes[] = {"DENSE_SCHUR", "SPARSE_SCHUR", "DENSE_NORMAL_CHOLESKY", "DENSE_QR",
                                    "SPARSE_NORMAL_CHOLESKY"};  // reference optimizer.hpp:71-77

bool valid_solver_type(const char* s) {
  for (const char* t : kSolverTypes)
    if (std::strcmp(s, t) == 0) return true;
  return false;
}

}  // namespace

struct smpc_handle {
  smpc_params params;
  int device = 0;
  int n_sm = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t stream2 = nullptr;  // second lane of the chunked host-buffer pipeline (smpc_solve_batch)
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_shared = nullptr;
  bool timed = false;
  int* queue = nullptr;
  long long launches = 0;
  int forced_warps = 0;  // 0 = pick warps-per-CTA from the batch size; SMPC_WARPS env overrides (4 / 16 with people, 4 / 12 without)
  int park_quantum = 32; // evaluations per time slice of the solve queue (0 = off); SMPC_PARK_QUANTUM env overrides
  DeviceBuffer park_buf; // parked group states + ring + counters of the time-sliced queue
  PinnedBuffer pin_in, pin_out;  // staging of the packed small-batch path (kPackedBytes)
  int stream_maps = 1;   // 1 = stream per-problem costmaps under the solve (pinned host buffers only); SMPC_STREAM_MAPS=0 disables
  unsigned* arrival = nullptr;       // device: {problems whose costmap has arrived, kernel gave up waiting}
  unsigned* arrival_host = nullptr;  // pinned: the values the copy stream writes to arrival[0], one per map chunk
  int cta_sync = -1;     // CTA barrier per evaluation: -1 = default (on), SMPC_CTA_SYNC env overrides (0 / 1)
  int forced_chunks = 0; // 0 = pick the chunk count of the host-buffer pipeline from the batch; SMPC_CHUNKS env overrides (1..8)
  int forced_group = 0;  // 0 = pick lanes-per-problem from the batch size; SMPC_GROUP env / smpc_set_group override
  std::mutex mu;
  // staging for the host-buffer entry points
  DeviceBuffer in_buf, out_buf;
  DeviceBuffer pack_buf;  // agent records (x, y, vx, vy) + validity bytes of the current batch
  smpc_memory memory;  // (unused since round 2: the level-2 memory lives on the device, smpc_fleet_state)
  smpc_fleet_state fleet;        // fleet tick (smpc_optimize_batch)
  smpc_fleet_state single;       // the one-robot fleet behind smpc_optimize
  smpc_fleet_state episodes;     // closed-loop episodes (smpc_run_episodes)
};

const smpc_params* smpc_handle_params(smpc_handle* h) { return &h->params; }
smpc_memory* smpc_handle_memory(smpc_handle* h) { return &h->memory; }
smpc_fleet_state* smpc_handle_fleet(smpc_handle* h) { return &h->fleet; }
smpc_fleet_state* smpc_handle_single(smpc_handle* h) { return &h->single; }
smpc_fleet_state* smpc_handle_episodes(smpc_handle* h) { return &h->episodes; }
int smpc_handle_device(smpc_handle* h) { return h->device; }
int smpc_host_fail(int code, const std::string& msg) { return fail(code, msg); }
cudaStream_t smpc_handle_stream(smpc_handle* h) { return h->stream; }
void smpc_handle_count_launch(smpc_handle* h) { h->launches += 1; }

namespace {

int derive_dims(const smpc_params* p, int S, int* ch, int* bl, int* nb, int* n_bounded) {
  if (S < 1) return fail(SMPC_ERR_ARGUMENT, "n_steps must be >= 1 (the reference needs a path of >= 2 poses)");
  if (p->control_horizon < 1 || p->parameter_block_length < 1)
    return fail(SMPC_ERR_PARAM, "control_horizon and parameter_block_length must be >= 1");
  const int c = std::min(p->control_horizon, S);         // src/optimizer.cpp:248
  const int b = std::min(p->parameter_block_length, c);  // src/optimizer.cpp:249
  if (ch) *ch = c;
  if (bl) *bl = b;
  if (nb) *nb = (c + b - 1) / b;
  if (n_bounded) *n_bounded = c / b;
  return SMPC_OK;
}

int make_dev_params(const smpc_params& p, int S, smpc::DevParams* d) {
  int rc = derive_dims(&p, S, &d->ch, &d->bl, &d->nb, &d->n_bounded);
  if (rc != SMPC_OK) return rc;
  if (d->nb > smpc::max_supported_blocks())
    return fail(SMPC_ERR_UNSUPPORTED, "more than " + std::to_string(smpc::max_supported_blocks()) +
                                          " parameter blocks are not built into this libsmpc.so");
  if (S > smpc::kMaxSteps) return fail(SMPC_ERR_UNSUPPORTED, "n_steps > 64 is not supported");
  d->w_distance = p.distance_w;
  d->w_social = p.socialwork_w;
  d->w_velocity = p.velocity_w;
  d->w_angle = p.angle_w;
  d->w_agent_angle = p.agent_angle_w;
  d->w_prox = p.proxemics_w;
  d->w_vf = p.velocity_feasibility_w;
  d->w_obstacle = p.obstacle_w;
  d->w_goal = p.goal_align_w;
  d->param_tol = p.param_tol;
  d->fn_tol = p.fn_tol;
  d->gradient_tol = p.gradient_tol;
  d->max_iterations = p.max_iterations;
  d->ceres_compat = p.ceres_compat ? p.ceres_compat : 200;
  d->max_evaluations = p.max_evaluations > 0 ? p.max_evaluations : 0;
  d->dof = p.omni_solve ? 3 : 2;
  if (d->dof == 3 && d->nb > 6)
    return fail(SMPC_ERR_UNSUPPORTED, "omni_solve is built for up to 6 parameter blocks (18 parameters)");
  d->control_horizon = p.control_horizon;
  d->block_length = p.parameter_block_length;
  return SMPC_OK;
}

int check_batch(const smpc_batch* in) {
  if (!in) return fail(SMPC_ERR_ARGUMENT, "batch is NULL");
  if (in->n_problems < 0) return fail(SMPC_ERR_ARGUMENT, "n_problems < 0");
  if (in->n_agents < 0) return fail(SMPC_ERR_ARGUMENT, "n_agents < 0");
  if (in->n_problems == 0) return SMPC_OK;
  if (!in->pose0 || !in->u0 || !in->path_xy || !in->goal_yaw) return fail(SMPC_ERR_ARGUMENT, "pose0/u0/path_xy/goal_yaw missing");
  if (!in->costmaps || !in->costmap_origin || in->n_costmaps < 1 || in->size_x < 1 || in->size_y < 1)
    return fail(SMPC_ERR_ARGUMENT, "costmap missing (the reference always dereferences costmap->getCharMap())");
  if (!(in->resolution > 0.0)) return fail(SMPC_ERR_ARGUMENT, "costmap resolution must be > 0");
  if (!(in->dt > 0.0)) return fail(SMPC_ERR_ARGUMENT, "dt must be > 0");
  if (in->scenario_index && in->n_scenarios < 1) return fail(SMPC_ERR_ARGUMENT, "scenario_index given but n_scenarios < 1");
  return SMPC_OK;
}

void to_dev_batch(const smpc_batch& in, smpc::DevBatch* d) {
  d->B = in.n_problems;
  d->S = in.n_steps;
  d->A = (in.agents != nullptr) ? in.n_agents : 0;
  d->M = in.n_costmaps;
  d->size_x = in.size_x;
  d->size_y = in.size_y;
  d->resolution = in.resolution;
  d->dt = in.dt;
  d->pose0 = in.pose0;
  d->u0 = in.u0;
  d->path_xy = in.path_xy;
  d->goal_yaw = in.goal_yaw;
  d->agents = in.agents;
  d->has_people = in.has_people;
  d->costmaps = in.costmaps;
  d->costmap_origin = in.costmap_origin;
  d->costmap_index = in.costmap_index;
  d->n_steps_each = in.n_steps_each;
  d->arrival = nullptr;
  d->park_state = nullptr;
  d->park_ring = nullptr;
  d->park_counters = nullptr;
  d->park_quantum = 0;
  d->cta_sync = 1;
  d->scenario = in.scenario_index;
  d->n_rows = in.scenario_index ? in.n_scenarios : in.n_problems;
}

// Build the packed agent records of a batch in the handle's scratch buffer (one small kernel per batch).
int pack_agents(smpc_handle* h, smpc::DevBatch* bt, cudaStream_t stream);

void to_dev_result(const smpc_result& out, smpc::DevResult* d) {
  d->u = out.u;
  d->cmds = out.cmds;
  d->path = out.path;
  d->cost_initial = out.cost_initial;
  d->cost_final = out.cost_final;
  d->iterations = out.iterations;
  d->termination = out.termination;
  d->usable = out.usable;
  d->n_evals = out.n_evals;
  d->trace = (out.trace_rows > 0) ? out.trace : nullptr;
  d->trace_rows = out.trace_rows;
}

size_t align256(size_t v) { return (v + 255) & ~static_cast<size_t>(255); }

// `total_problems` sizes the scratch buffer (>= bt->B); `first` = index of this batch's first problem inside it, so
// that the chunks of one host-buffer call pack into disjoint slices.
int pack_agents_at(smpc_handle* h, smpc::DevBatch* bt, size_t total_problems, size_t first, cudaStream_t stream) {
  bt->agents_packed = nullptr;
  bt->agents_valid = nullptr;
  if (bt->A <= 0 || bt->agents == nullptr) return SMPC_OK;
  const size_t S1 = static_cast<size_t>(bt->S) + 1;
  if (bt->scenario) {  // per-scene arrays: all n_rows scenes are packed once (scenario batches are never chunked)
    total_problems = static_cast<size_t>(bt->n_rows);
    first = 0;
  }
  const size_t all_rows = total_problems * bt->A;
  const size_t rows = (bt->scenario ? static_cast<size_t>(bt->n_rows) : static_cast<size_t>(bt->B)) * bt->A;
  const size_t rec_bytes = align256(all_rows * S1 * 4 * sizeof(double));
  SMPC_CUDA(h->pack_buf.reserve(rec_bytes + all_rows * S1));
  double* packed = static_cast<double*>(h->pack_buf.ptr) + first * bt->A * S1 * 4;
  uint8_t* valid = static_cast<uint8_t*>(h->pack_buf.ptr) + rec_bytes + first * bt->A * S1;
  SMPC_CUDA(smpc::launch_pack_agents(static_cast<long long>(rows), static_cast<int>(S1), bt->agents, packed, valid, stream));
  h->launches += 1;
  bt->agents_packed = packed;
  bt->agents_valid = valid;
  return SMPC_OK;
}

int pack_agents(smpc_handle* h, smpc::DevBatch* bt, cudaStream_t stream) {
  return pack_agents_at(h, bt, static_cast<size_t>(bt->B), 0, stream);
}

struct Carver {  // carve aligned sub-buffers out of one device allocation
  char* base;
  size_t off = 0;
  explicit Carver(void* b) : base(static_cast<char*>(b)) {}
  void* take(size_t bytes) {
    void* p = base ? base + off : nullptr;
    off += align256(bytes);
    return p;
  }
};

// ---- YAML subtree reader (indentation based; enough for Nav2 parameter files) ---------------------------
std::string trim(const std::string& s) {
  size_t a = s.find_first_not_of(" \t\r\n");
  if (a == std::string::npos) return "";
  size_t b = s.find_last_not_of(" \t\r\n");
  return s.substr(a, b - a + 1);
}

std::string strip_comment(const std::string& s) {
  bool in_s = false, in_d = false;
  for (size_t i = 0; i < s.size(); ++i) {
    if (s[i] == '\'' && !in_d) in_s = !in_s;
    if (s[i] == '"' && !in_s) in_d = !in_d;
    if (s[i] == '#' && !in_s && !in_d && (i == 0 || s[i - 1] == ' ' || s[i - 1] == '\t')) return s.substr(0, i);
  }
  return s;
}

// Flatten every `key: value` leaf below `<plugin>:` into "a.b.c" -> "value".
bool read_plugin_subtree(const std::string& path, const std::string& plugin, std::map<std::string, std::string>* kv,
                         std::string* err) {
  std::ifstream f(path);
  if (!f) {
    *err = "cannot open " + path;
    return false;
  }
  std::string line;
  bool inside = false;
  int plugin_indent = -1;
  std::vector<std::pair<int, std::string>> stack;
  while (std::getline(f, line)) {
    const std::string body = strip_comment(line);
    if (trim(body).empty()) continue;
    const int indent = static_cast<int>(body.find_first_not_of(' '));
    const std::string t = trim(body);
    const size_t colon = t.find(':');
    if (colon == std::string::npos) continue;
    const std::string key = trim(t.substr(0, colon));
    std::string val = trim(t.substr(colon + 1));
    if (!inside) {
      if (key == plugin && val.empty()) {
        inside = true;
        plugin_indent = indent;
        stack.clear();
      }
      continue;
    }
    if (indent <= plugin_indent) break;  // left the subtree
    while (!stack.empty() && stack.back().first >= indent) stack.pop_back();
    if (val.empty()) {
      stack.emplace_back(indent, key);
      continue;
    }
    if (val.size() >= 2 && ((val.front() == '"' && val.back() == '"') || (val.front() == '\'' && val.back() == '\'')))
      val = val.substr(1, val.size() - 2);
    std::string full;
    for (auto& s : stack) full += s.second + ".";
    (*kv)[full + key] = val;
  }
  if (!inside) {
    *err = "plugin subtree '" + plugin + ":' not found in " + path;
    return false;
  }
  return true;
}

bool parse_bool(const std::string& v) { return v == "true" || v == "True" || v == "TRUE" || v == "1"; }

}  // namespace

extern "C" {

int smpc_abi_version(void) { return SMPC_ABI_VERSION; }

const char* smpc_last_error(void) { return g_last_error.c_str(); }

void smpc_params_default(smpc_params* p) {
  if (!p) return;
  std::memset(p, 0, sizeof(*p));
  // src/optimizer.cpp:26-84
  std::snprintf(p->linear_solver_type, sizeof(p->linear_solver_type), "%s", "SPARSE_NORMAL_CHOLESKY");
  p->param_tol = 1e-15;
  p->fn_tol = 1e-7;
  p->gradient_tol = 1e-10;
  p->max_iterations = 100;
  p->debug = 0;
  p->control_horizon = 5;
  p->parameter_block_length = 5;
  p->discretization = 0;
  p->distance_w = 3.0;
  p->socialwork_w = 1.0;
  p->velocity_w = 0.5;
  p->angle_w = 0.0;
  p->agent_angle_w = 0.5;
  p->proxemics_w = 90.0;
  p->velocity_feasibility_w = 0.5;
  p->obstacle_w = 0.0;
  p->goal_align_w = 0.0;
  p->current_path_w = 1.0f;
  p->current_cmds_w = 1.0f;
  // src/path_trajectorizer.cpp:52-59
  p->max_time = 3.0f;
  p->time_step = 0.05f;
  p->omnidirectional = 0;
  p->traj_desired_linear_vel = 0.4;
  p->lookahead_dist = 0.4;
  p->max_angular_vel = 1.0;
  p->transform_tolerance = 0.1;
  std::snprintf(p->base_frame, sizeof(p->base_frame), "%s", "base_footprint");
  // src/social_mpc_controller.cpp:59-65
  p->desired_linear_vel = 0.5;
  p->fov_angle = M_PI / 4.0;
  p->ceres_compat = 200;
  p->max_evaluations = 0;
  p->omni_solve = 0;
}

int smpc_params_from_yaml(const char* yaml_path, const char* plugin_name, smpc_params* p) {
  if (!yaml_path || !plugin_name || !p) return fail(SMPC_ERR_ARGUMENT, "NULL argument");
  std::map<std::string, std::string> kv;
  std::string err;
  if (!read_plugin_subtree(yaml_path, plugin_name, &kv, &err)) return fail(SMPC_ERR_IO, err);
  smpc_params_default(p);
  auto num = [&](const char* key, double* out) {
    auto it = kv.find(key);
    if (it != kv.end()) *out = std::strtod(it->second.c_str(), nullptr);
  };
  auto inum = [&](const char* key, int* out) {
    auto it = kv.find(key);
    if (it != kv.end()) *out = static_cast<int>(std::strtol(it->second.c_str(), nullptr, 10));
  };
  auto fnum = [&](const char* key, float* out) {
    auto it = kv.find(key);
    if (it != kv.end()) *out = static_cast<float>(std::strtod(it->second.c_str(), nullptr));
  };
  if (kv.count("optimizer.linear_solver_type"))
    std::snprintf(p->linear_solver_type, sizeof(p->linear_solver_type), "%s", kv["optimizer.linear_solver_type"].c_str());
  if (!valid_solver_type(p->linear_solver_type)) {
    std::string valid;
    for (const char* t : kSolverTypes) valid += std::string(valid.empty() ? "" : ", ") + t;
    // mirrors the std::runtime_error at src/optimizer.cpp:42-44
    return fail(SMPC_ERR_PARAM, "Invalid parameter: linear_solver_type. Valid values are " + valid);
  }
  num("optimizer.param_tol", &p->param_tol);
  num("optimizer.fn_tol", &p->fn_tol);
  num("optimizer.gradient_tol", &p->gradient_tol);
  inum("optimizer.max_iterations", &p->max_iterations);
  if (kv.count("optimizer.debug_optimizer")) p->debug = parse_bool(kv["optimizer.debug_optimizer"]) ? 1 : 0;
  inum("optimizer.control_horizon", &p->control_horizon);
  inum("optimizer.parameter_block_length", &p->parameter_block_length);
  inum("optimizer.discretization", &p->discretization);
  fnum("optimizer.current_path_weight", &p->current_path_w);
  fnum("optimizer.current_cmds_weight", &p->current_cmds_w);
  num("optimizer.weights.distance_weight", &p->distance_w);
  num("optimizer.weights.social_weight", &p->socialwork_w);
  num("optimizer.weights.velocity_weight", &p->velocity_w);
  num("optimizer.weights.angle_weight", &p->angle_w);
  num("optimizer.weights.agent_angle_weight", &p->agent_angle_w);
  num("optimizer.weights.proxemics_weight", &p->proxemics_w);
  num("optimizer.weights.velocity_feasibility_weight", &p->velocity_feasibility_w);
  num("optimizer.weights.obstacle_weight", &p->obstacle_w);
  num("optimizer.weights.goal_align_weight", &p->goal_align_w);
  fnum("trajectorizer.max_time", &p->max_time);
  fnum("trajectorizer.time_step", &p->time_step);
  if (kv.count("trajectorizer.omnidirectional")) p->omnidirectional = parse_bool(kv["trajectorizer.omnidirectional"]) ? 1 : 0;
  num("trajectorizer.desired_linear_vel", &p->traj_desired_linear_vel);
  num("trajectorizer.lookahead_dist", &p->lookahead_dist);
  num("trajectorizer.max_angular_vel", &p->max_angular_vel);
  num("trajectorizer.transform_tolerance", &p->transform_tolerance);
  if (kv.count("trajectorizer.base_frame"))
    std::snprintf(p->base_frame, sizeof(p->base_frame), "%s", kv["trajectorizer.base_frame"].c_str());
  num("desired_linear_vel", &p->desired_linear_vel);
  num("fov_angle", &p->fov_angle);
  return SMPC_OK;
}

int smpc_problem_dims(const smpc_params* p, int n_steps, int* ch, int* bl, int* n_blocks, int* n_bounded) {
  if (!p) return fail(SMPC_ERR_ARGUMENT, "params is NULL");
  return derive_dims(p, n_steps, ch, bl, n_blocks, n_bounded);
}

int smpc_create(const smpc_params* p, int device, smpc_handle** out) {
  if (!p || !out) return fail(SMPC_ERR_ARGUMENT, "NULL argument");
  if (!valid_solver_type(p->linear_solver_type)) return fail(SMPC_ERR_PARAM, "Invalid parameter: linear_solver_type");
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev == 0)
    return fail(SMPC_ERR_CUDA, std::string("no CUDA device available (libsmpc has no CPU path): ") + cudaGetErrorString(e));
  if (device < 0 || device >= n_dev) return fail(SMPC_ERR_ARGUMENT, "device index out of range");
  SMPC_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  SMPC_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10)
    return fail(SMPC_ERR_UNSUPPORTED, "libsmpc.so is built for sm_100a (B200); found compute capability " +
                                          std::to_string(prop.major) + "." + std::to_string(prop.minor));
  smpc_handle* h = new smpc_handle();
  h->params = *p;
  h->device = device;
  h->n_sm = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&h->stream2, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&h->ev0) != cudaSuccess || cudaEventCreate(&h->ev1) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->ev_shared, cudaEventDisableTiming) != cudaSuccess ||
      cudaMalloc(&h->queue, kMaxChunks * sizeof(int)) != cudaSuccess ||
      cudaMalloc(&h->arrival, 2 * sizeof(unsigned)) != cudaSuccess ||
      cudaHostAlloc(&h->arrival_host, (kMapChunks + 2) * sizeof(unsigned), cudaHostAllocDefault) != cudaSuccess) {
    e = cudaGetLastError();
    smpc_destroy(h);
    return cuda_fail(e, "smpc_create resources");
  }
  if (const char* env = std::getenv("SMPC_GROUP")) h->forced_group = std::atoi(env);
  if (const char* env = std::getenv("SMPC_WARPS")) h->forced_warps = std::atoi(env);
  if (const char* env = std::getenv("SMPC_CHUNKS")) h->forced_chunks = std::atoi(env);
  if (const char* env = std::getenv("SMPC_STREAM_MAPS")) h->stream_maps = std::atoi(env);
  if (const char* env = std::getenv("SMPC_PARK_QUANTUM")) h->park_quantum = std::max(0, std::atoi(env));
  if (const char* env = std::getenv("SMPC_CTA_SYNC")) h->cta_sync = std::atoi(env) != 0;
  *out = h;
  return SMPC_OK;
}

int smpc_set_group(smpc_handle* h, int lanes_per_problem) {
  if (!h) return fail(SMPC_ERR_ARGUMENT, "handle is NULL");
  if (lanes_per_problem != 0 && lanes_per_problem != 4 && lanes_per_problem != 8 && lanes_per_problem != 16 &&
      lanes_per_problem != 32)
    return fail(SMPC_ERR_ARGUMENT, "lanes_per_problem must be 0 (auto), 4, 8, 16 or 32");
  h->forced_group = lanes_per_problem;
  return SMPC_OK;
}

void smpc_destroy(smpc_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->stream2) cudaStreamSynchronize(h->stream2);
  h->in_buf.release();
  h->out_buf.release();
  h->pack_buf.release();
  h->park_buf.release();
  h->pin_in.release();
  h->pin_out.release();
  h->fleet.release();
  h->single.release();
  h->episodes.release();
  if (h->queue) cudaFree(h->queue);
  if (h->arrival) cudaFree(h->arrival);
  if (h->arrival_host) cudaFreeHost(h->arrival_host);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->ev_shared) cudaEventDestroy(h->ev_shared);
  if (h->stream2) cudaStreamDestroy(h->stream2);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

// One solve launch of `in` (device pointers) on `stream`. `queue` = this launch's work-queue counter; the packed agent
// records go to slice [first, first + B) of a scratch buffer sized for `total_problems`.
static int launch_solve_on(smpc_handle* h, const smpc_batch* in, smpc_result* out, int* queue, size_t total_problems,
                           size_t first, bool timed, cudaStream_t stream, unsigned* arrival = nullptr) {
  smpc::DevParams prm;
  int rc = make_dev_params(h->params, in->n_steps, &prm);
  if (rc != SMPC_OK) return rc;
  smpc::DevBatch bt;
  to_dev_batch(*in, &bt);
  bt.arrival = arrival;
  bt.cta_sync = (h->cta_sync < 0) ? 1 : h->cta_sync;
  smpc::DevResult rs;
  to_dev_result(*out, &rs);
  rc = pack_agents_at(h, &bt, total_problems, first, stream);
  if (rc != SMPC_OK) return rc;
  SMPC_CUDA(cudaMemsetAsync(queue, 0, sizeof(int), stream));
  // parking area of the time-sliced queue (the launcher drops it again when the batch is not a few waves large). One
  // area per handle: only the single-launch calls use it (the chunks of the host pipeline run concurrently).
  const bool people = bt.A > 0 && bt.agents != nullptr && bt.has_people != nullptr;  // = batch_has_people of the launcher
  if (h->park_quantum > 0 && !people && total_problems == static_cast<size_t>(in->n_problems) &&
      in->n_problems <= (1 << 18)) {
    const size_t Bp = static_cast<size_t>(in->n_problems);
    const size_t state_bytes = align256(Bp * smpc::layout_total(prm.nb, in->n_steps, prm.dof) * sizeof(double));
    const size_t ring_bytes = align256(Bp * sizeof(int));
    SMPC_CUDA(h->park_buf.reserve(state_bytes + ring_bytes + 256));
    char* base = static_cast<char*>(h->park_buf.ptr);
    bt.park_state = reinterpret_cast<double*>(base);
    bt.park_ring = reinterpret_cast<int*>(base + state_bytes);
    bt.park_counters = reinterpret_cast<int*>(base + state_bytes + ring_bytes);
    bt.park_quantum = h->park_quantum;
    SMPC_CUDA(cudaMemsetAsync(bt.park_ring, 0xFF, ring_bytes, stream));
    SMPC_CUDA(cudaMemsetAsync(bt.park_counters, 0, 4 * sizeof(int), stream));
  }
  if (timed) SMPC_CUDA(cudaEventRecord(h->ev0, stream));
  SMPC_CUDA(smpc::launch_solve(prm, bt, rs, queue, h->n_sm, h->forced_group, h->forced_warps, stream));
  if (timed) SMPC_CUDA(cudaEventRecord(h->ev1, stream));
  h->timed = timed;
  h->launches += 1;
  return SMPC_OK;
}

static int solve_device_locked(smpc_handle* h, const smpc_batch* in, smpc_result* out, cudaStream_t stream) {
  int rc = check_batch(in);
  if (rc != SMPC_OK) return rc;
  if (!out) return fail(SMPC_ERR_ARGUMENT, "result is NULL");
  if (in->n_problems == 0) return SMPC_OK;
  SMPC_CUDA(cudaSetDevice(h->device));
  return launch_solve_on(h, in, out, h->queue, static_cast<size_t>(in->n_problems), 0, true, stream);
}

int smpc_solve_batch_device(smpc_handle* h, const smpc_batch* in, smpc_result* out, void* stream) {
  if (!h) return fail(SMPC_ERR_ARGUMENT, "handle is NULL");
  std::lock_guard<std::mutex> lk(h->mu);
  return solve_device_locked(h, in, out, stream ? static_cast<cudaStream_t>(stream) : h->stream);
}

// Chunk plan of the host-buffer pipeline (pure: no CUDA call, exported for the CPU test suite as
// smpc_debug_plan_chunks). Chunking pays where the copies are a large share of the call: batches with people (28 kB
// per problem at 20 agents; measured +22 % end to end at A = 20, +14 % at A = 50, +3 % at A = 3). People-free batches
// are one chunk: their copies are small next to the solve and smaller launches balance worse (measured -2..-13 %);
// they stream their inputs into the one launch instead. A chunk must not push the launch heuristics of
// smpc_kernels_nb.inc into another kernel variant than the whole batch would get: 16-warp CTAs need >= 2 warps per warp
// slot, i.e. >= 2 * 16 * n_sm problems per launch — also for the ragged last chunk. Shared costmaps addressed by
// b % M need chunk starts that are multiples of M.
static void plan_chunks(int n_sm, size_t B, bool people, size_t M, bool maps_per_problem, bool has_index, int forced_chunks,
                        size_t* n_chunks_out, size_t* chunk_out) {
  const size_t w16_min = 2 * 16 * static_cast<size_t>(n_sm);
  size_t n_chunks = 1;
  if (people) n_chunks = std::min<size_t>(kMaxChunks, B / (w16_min + 128));
  if (forced_chunks >= 1) n_chunks = std::min<size_t>(forced_chunks, kMaxChunks);
  n_chunks = std::max<size_t>(1, std::min(n_chunks, B));
  size_t chunk = B;
  for (; n_chunks > 1; --n_chunks) {
    chunk = ((B + n_chunks - 1) / n_chunks + 255) & ~static_cast<size_t>(255);
    const size_t used = (B + chunk - 1) / chunk;  // chunks actually needed at this (rounded-up) size
    const size_t last = B - (used - 1) * chunk;
    const bool modulo_ok = maps_per_problem || has_index || (chunk % M) == 0;  // b % M must not shift
    const bool size_ok = forced_chunks >= 1 || last >= w16_min;
    if (modulo_ok && size_ok) {
      n_chunks = used;
      break;
    }
  }
  if (n_chunks <= 1) {
    n_chunks = 1;
    chunk = B;
  }
  *n_chunks_out = n_chunks;
  *chunk_out = chunk;
}

int smpc_debug_plan_chunks(int n_sm, int n_problems, int has_people, int n_costmaps, int maps_per_problem, int has_index,
                           int forced_chunks, int* n_chunks, int* chunk) {
  if (n_sm < 1 || n_problems < 1 || n_costmaps < 1 || !n_chunks || !chunk) return fail(SMPC_ERR_ARGUMENT, "bad plan arguments");
  size_t n = 1, c = static_cast<size_t>(n_problems);
  plan_chunks(n_sm, static_cast<size_t>(n_problems), has_people != 0, static_cast<size_t>(n_costmaps), maps_per_problem != 0,
              has_index != 0, forced_chunks, &n, &c);
  *n_chunks = static_cast<int>(n);
  *chunk = static_cast<int>(c);
  return SMPC_OK;
}

// Host buffers in, host buffers out. The batch is cut into up to kMaxChunks chunks of consecutive problems that
// alternate between two streams: chunk k+1's host-to-device copies run while chunk k solves, and chunk k's results
// travel back while chunk k+1 solves (problems are independent, so a chunk is a complete batch of its own). Copies
// overlap only when the caller's buffers are page-locked; pageable buffers work, serialised by the driver.
int smpc_solve_batch(smpc_handle* h, const smpc_batch* in, smpc_result* out) {
  if (!h) return fail(SMPC_ERR_ARGUMENT, "handle is NULL");
  std::lock_guard<std::mutex> lk(h->mu);
  int rc = check_batch(in);
  if (rc != SMPC_OK) return rc;
  if (!out) return fail(SMPC_ERR_ARGUMENT, "result is NULL");
  if (in->n_problems == 0) return SMPC_OK;
  int nb = 0;
  rc = derive_dims(&h->params, in->n_steps, nullptr, nullptr, &nb, nullptr);
  if (rc != SMPC_OK) return rc;
  SMPC_CUDA(cudaSetDevice(h->device));
  const size_t B = in->n_problems, S1 = static_cast<size_t>(in->n_steps) + 1, A = in->agents ? in->n_agents : 0;
  const size_t dof = h->params.omni_solve ? 3 : 2;  // parameters per block: (v, w) or the omnidirectional (vx, vy, w)
  const size_t M = in->n_costmaps, P = dof * static_cast<size_t>(nb);
  const size_t map_cells = static_cast<size_t>(in->size_x) * in->size_y;

  // ---- chunking. Costmaps follow their problems when map b belongs to problem b (no index, M == B); otherwise the
  //      M maps are shared: they go up once, ahead of the first chunk, and every chunk start must keep b % M intact.
  // an explicit identity index (map b for problem b) is the same thing as no index with M == B
  bool identity_index = (in->costmap_index != nullptr) && (M == B) && (in->scenario_index == nullptr);
  for (size_t b = 0; identity_index && b < B; ++b) identity_index = in->costmap_index[b] == static_cast<int32_t>(b);
  const int32_t* host_index = identity_index ? nullptr : in->costmap_index;
  // scenario sharing: the per-scene arrays (R rows) go up once like shared costmaps and the batch is one launch — only
  // u0 and the scenario index are per problem, so there is nothing worth chunking or streaming
  const bool scenes = in->scenario_index != nullptr;
  const size_t R = scenes ? static_cast<size_t>(in->n_scenarios) : B;
  const bool maps_per_problem = !scenes && (host_index == nullptr) && (M == B);
  size_t n_chunks = 1, chunk = B;
  if (!scenes)
    plan_chunks(h->n_sm, B, A > 0 && in->has_people, M, maps_per_problem, host_index != nullptr, h->forced_chunks,
                &n_chunks, &chunk);

  // ---- device staging: every array whole, same layout as the host's, so a chunk is a pointer offset
  struct Item { const void* host; size_t per_problem; size_t shared_bytes; char* dev; };
  enum { kPose, kU0, kPath, kGoal, kAgents, kHas, kIndex, kMaps, kOrigin, kNEach, kScene, kItems };
  // per-scene arrays: per problem normally, ONE shared block of R rows with scenario sharing
  auto scene_item = [&](const void* host, size_t row_bytes) {
    return scenes ? Item{host, 0, row_bytes * R, nullptr} : Item{host, row_bytes, 0, nullptr};
  };
  Item items[kItems] = {
      scene_item(in->pose0, 3 * 8),
      {in->u0, P * 8, 0, nullptr},
      scene_item(in->path_xy, 2 * S1 * 8),
      scene_item(in->goal_yaw, 8),
      scene_item(A ? in->agents : nullptr, A * 6 * S1 * 8),
      scene_item(in->has_people, 1),
      scene_item(host_index, 4),
      {in->costmaps, maps_per_problem ? map_cells : 0, maps_per_problem ? 0 : M * map_cells, nullptr},
      {in->costmap_origin, maps_per_problem ? 16 : 0, maps_per_problem ? 0 : M * 16, nullptr},
      scene_item(in->n_steps_each, 4),
      {in->scenario_index, 4, 0, nullptr},
  };
  size_t total = 0;
  for (auto& it : items)
    if (it.host) total += align256(it.per_problem * B + it.shared_bytes);
  SMPC_CUDA(h->in_buf.reserve(total));
  Carver cin(h->in_buf.ptr);
  for (auto& it : items)
    if (it.host) it.dev = static_cast<char*>(cin.take(it.per_problem * B + it.shared_bytes));

  struct OItem { void* host; size_t per_problem; char* dev; };
  enum { kOU, kOCmds, kOPath, kOCi, kOCf, kOIt, kOTerm, kOUsable, kOEvals, kOTrace, kOItems };
  const size_t trace_rows = (out->trace && out->trace_rows > 0) ? static_cast<size_t>(out->trace_rows) : 0;
  OItem oitems[kOItems] = {
      {out->u, P * 8, nullptr},        {out->cmds, S1 * dof * 8, nullptr}, {out->path, S1 * 3 * 8, nullptr},
      {out->cost_initial, 8, nullptr}, {out->cost_final, 8, nullptr},    {out->iterations, 4, nullptr},
      {out->termination, 4, nullptr},  {out->usable, 1, nullptr},        {out->n_evals, 2 * 4, nullptr},
      {trace_rows ? out->trace : nullptr, trace_rows * 8 * 8, nullptr},
  };
  size_t ototal = 0;
  for (auto& it : oitems)
    if (it.host) ototal += align256(it.per_problem * B);
  SMPC_CUDA(h->out_buf.reserve(ototal));
  Carver cout_(h->out_buf.ptr);
  for (auto& it : oitems)
    if (it.host) it.dev = static_cast<char*>(cout_.take(it.per_problem * B));
  // Rows a problem does not write (beyond its own horizon / blocks with n_steps_each, unused trace rows) come back as
  // zero bytes (trace: NaN) instead of stale staging memory.
  if (in->n_steps_each) SMPC_CUDA(cudaMemsetAsync(h->out_buf.ptr, 0, ototal, h->stream));
  if (trace_rows) SMPC_CUDA(cudaMemsetAsync(oitems[kOTrace].dev, 0xFF, trace_rows * 64 * B, h->stream));
  if (in->n_steps_each || trace_rows) {
    SMPC_CUDA(cudaEventRecord(h->ev_shared, h->stream));
    SMPC_CUDA(cudaStreamWaitEvent(h->stream2, h->ev_shared, 0));
  }

  // ---- people-free batch with one costmap per problem: the maps are 90 % of the input bytes. They stream in on the
  //      second stream WHILE the solve runs: problems are handed out in index order and a group waits until the
  //      arrival counter has passed its problem (wait_for_costmap). Only with page-locked host maps (the copies must
  //      be truly asynchronous) and no other kernel of this call in flight (nothing may need an SM while groups wait).
  // Large batches stream their other per-problem arrays (seed path, pose, start controls: 0.5 kB per problem) the same
  // way once those are worth more than the extra copy calls (>= 8 MB).
  bool stream_maps = false;   // streaming mode on (the name is historical: maps were the first thing streamed)
  bool streamed[kItems] = {false, false, false, false, false, false, false, false, false, false, false};
  if (h->stream_maps && n_chunks == 1 && !scenes && !(A > 0 && in->has_people) && B >= 1024) {
    size_t small_bytes = 0;
    for (int k = 0; k < kItems; ++k)
      if (k != kMaps && items[k].host && items[k].per_problem) small_bytes += items[k].per_problem * B;
    const bool stream_small = small_bytes >= (8u << 20);
    bool all_pinned = true;
    for (int k = 0; k < kItems; ++k) {
      if (!(items[k].host && items[k].per_problem)) continue;
      if (!((k == kMaps && maps_per_problem) || (k != kMaps && stream_small))) continue;
      cudaPointerAttributes attr;
      if (cudaPointerGetAttributes(&attr, items[k].host) == cudaSuccess && attr.type == cudaMemoryTypeHost) {
        streamed[k] = true;
      } else {
        (void)cudaGetLastError();
        all_pinned = false;
      }
    }
    for (int k = 0; k < kItems; ++k) {
      if (!all_pinned) streamed[k] = false;
      stream_maps = stream_maps || streamed[k];
    }
  }

  // ---- shared arrays first (stream 1), the second stream waits for them
  cudaStream_t lanes[2] = {h->stream, h->stream2};
  // an error return below must not leave copies or kernels of this call in flight on either stream (the caller may
  // free or reuse its host arrays as soon as the call returns)
  struct Quiesce {
    cudaStream_t a, b;
    bool armed;
    ~Quiesce() {
      if (!armed) return;
      (void)cudaStreamSynchronize(a);
      (void)cudaStreamSynchronize(b);
      (void)cudaGetLastError();
    }
  } quiesce{lanes[0], lanes[1], true};
  // small batch: one staged block in, one staged block out (kPackedBytes)
  const bool packed = n_chunks == 1 && !stream_maps && total <= kPackedBytes && ototal <= kPackedBytes;
  if (packed) {
    SMPC_CUDA(h->pin_in.reserve(total));
    SMPC_CUDA(h->pin_out.reserve(ototal));
    char* stage = static_cast<char*>(h->pin_in.ptr);
    const char* dev0 = static_cast<const char*>(h->in_buf.ptr);
    for (auto& it : items)
      if (it.host) std::memcpy(stage + (it.dev - dev0), it.host, it.per_problem * B + it.shared_bytes);
    SMPC_CUDA(cudaMemcpyAsync(h->in_buf.ptr, stage, total, cudaMemcpyHostToDevice, lanes[0]));
  }
  bool any_shared = false;
  for (auto& it : items)
    if (!packed && it.host && it.shared_bytes) {
      SMPC_CUDA(cudaMemcpyAsync(it.dev, it.host, it.shared_bytes, cudaMemcpyHostToDevice, lanes[0]));
      any_shared = true;
    }
  if (any_shared && n_chunks > 1) {
    SMPC_CUDA(cudaEventRecord(h->ev_shared, lanes[0]));
    SMPC_CUDA(cudaStreamWaitEvent(lanes[1], h->ev_shared, 0));
  }

  for (size_t c = 0; c < n_chunks; ++c) {
    const size_t c0 = c * chunk, n = std::min(chunk, B - c0);
    cudaStream_t st = lanes[c & 1];
    for (int k = 0; k < kItems; ++k) {
      const Item& it = items[k];
      if (!packed && it.host && it.per_problem && !streamed[k])
        SMPC_CUDA(cudaMemcpyAsync(it.dev + it.per_problem * c0, static_cast<const char*>(it.host) + it.per_problem * c0,
                                  it.per_problem * n, cudaMemcpyHostToDevice, st));
    }
    if (stream_maps) {  // reset the arrival words before anything of this call can read or write them
      SMPC_CUDA(cudaMemsetAsync(h->arrival, 0, 2 * sizeof(unsigned), st));
      SMPC_CUDA(cudaEventRecord(h->ev_shared, st));
      SMPC_CUDA(cudaStreamWaitEvent(lanes[1], h->ev_shared, 0));
    }
    auto at = [&](int k) -> const void* { return items[k].dev ? items[k].dev + items[k].per_problem * c0 : nullptr; };
    smpc_batch din = *in;
    din.n_problems = static_cast<int>(n);
    din.pose0 = static_cast<const double*>(at(kPose));
    din.u0 = static_cast<const double*>(at(kU0));
    din.path_xy = static_cast<const double*>(at(kPath));
    din.goal_yaw = static_cast<const double*>(at(kGoal));
    din.agents = static_cast<const double*>(at(kAgents));
    din.has_people = static_cast<const uint8_t*>(at(kHas));
    din.costmap_index = static_cast<const int32_t*>(at(kIndex));
    din.costmaps = static_cast<const uint8_t*>(at(kMaps));
    din.costmap_origin = static_cast<const double*>(at(kOrigin));
    din.n_steps_each = static_cast<const int32_t*>(at(kNEach));
    din.scenario_index = static_cast<const int32_t*>(at(kScene));
    if (maps_per_problem) din.n_costmaps = static_cast<int>(n);
    auto oat = [&](int k) -> void* { return oitems[k].dev ? oitems[k].dev + oitems[k].per_problem * c0 : nullptr; };
    smpc_result dout;
    dout.u = static_cast<double*>(oat(kOU));
    dout.cmds = static_cast<double*>(oat(kOCmds));
    dout.path = static_cast<double*>(oat(kOPath));
    dout.cost_initial = static_cast<double*>(oat(kOCi));
    dout.cost_final = static_cast<double*>(oat(kOCf));
    dout.iterations = static_cast<int32_t*>(oat(kOIt));
    dout.termination = static_cast<int32_t*>(oat(kOTerm));
    dout.usable = static_cast<uint8_t*>(oat(kOUsable));
    dout.n_evals = static_cast<int32_t*>(oat(kOEvals));
    dout.trace = static_cast<double*>(oat(kOTrace));
    dout.trace_rows = static_cast<int>(trace_rows);
    if (stream_maps) {
      // Feed the solve its streamed inputs, piece by piece, each followed by its arrival count. Everything is enqueued BEFORE
      // the kernel launch: the copies then make progress whether or not the launch call returns early (profilers,
      // compute-sanitizer and CUDA_LAUNCH_BLOCKING=1 make launches synchronous — pieces enqueued after the launch
      // would never arrive and the solve would wait for its timeout).
      // pieces end on multiples of 128 problems: no cache line of any per-problem array (down to 1 byte per problem)
      // holds data of two pieces, so a line read through the read-only path can never be half-arrived
      const size_t piece = ((B + kMapChunks - 1) / kMapChunks + 127) & ~static_cast<size_t>(127);
      int k = 0;
      for (size_t p0 = 0; p0 < B; p0 += piece, ++k) {
        const size_t pn = std::min(piece, B - p0);
        for (int i = 0; i < kItems; ++i) {
          if (!streamed[i]) continue;
          const Item& it = items[i];
          SMPC_CUDA(cudaMemcpyAsync(it.dev + it.per_problem * p0, static_cast<const char*>(it.host) + it.per_problem * p0,
                                    it.per_problem * pn, cudaMemcpyHostToDevice, lanes[1]));
        }
        h->arrival_host[k] = static_cast<unsigned>(p0 + pn);
        SMPC_CUDA(cudaMemcpyAsync(h->arrival, h->arrival_host + k, sizeof(unsigned), cudaMemcpyHostToDevice, lanes[1]));
      }
    }
    rc = launch_solve_on(h, &din, &dout, h->queue + c, B, c0, /*timed=*/n_chunks == 1, st,
                         stream_maps ? h->arrival : nullptr);
    if (rc != SMPC_OK) return rc;
    if (packed) {
      SMPC_CUDA(cudaMemcpyAsync(h->pin_out.ptr, h->out_buf.ptr, ototal, cudaMemcpyDeviceToHost, st));
      continue;
    }
    for (auto& it : oitems)
      if (it.host)
        SMPC_CUDA(cudaMemcpyAsync(static_cast<char*>(it.host) + it.per_problem * c0, it.dev + it.per_problem * c0,
                                  it.per_problem * n, cudaMemcpyDeviceToHost, st));
  }
  if (stream_maps)
    SMPC_CUDA(cudaMemcpyAsync(h->arrival_host + kMapChunks, h->arrival, 2 * sizeof(unsigned), cudaMemcpyDeviceToHost,
                              lanes[0]));
  SMPC_CUDA(cudaStreamSynchronize(lanes[0]));
  if (n_chunks > 1 || stream_maps) SMPC_CUDA(cudaStreamSynchronize(lanes[1]));
  quiesce.armed = false;  // both streams are idle
  if (packed) {
    const char* stage = static_cast<const char*>(h->pin_out.ptr);
    const char* dev0 = static_cast<const char*>(h->out_buf.ptr);
    for (auto& it : oitems)
      if (it.host) std::memcpy(it.host, stage + (it.dev - dev0), it.per_problem * B);
  }
  if (stream_maps && h->arrival_host[kMapChunks + 1] != 0)
    return fail(SMPC_ERR_CUDA, "costmap stream stalled: the solve kernel waited 2 s for host-to-device copies");
  return SMPC_OK;
}

int smpc_eval_batch_device(smpc_handle* h, const smpc_batch* in, const double* x, smpc_eval_out* out, void* stream) {
  if (!h) return fail(SMPC_ERR_ARGUMENT, "handle is NULL");
  std::lock_guard<std::mutex> lk(h->mu);
  int rc = check_batch(in);
  if (rc != SMPC_OK) return rc;
  if (!x || !out) return fail(SMPC_ERR_ARGUMENT, "x / out is NULL");
  if (in->n_problems == 0) return SMPC_OK;
  smpc::DevParams prm;
  rc = make_dev_params(h->params, in->n_steps, &prm);
  if (rc != SMPC_OK) return rc;
  smpc::DevBatch bt;
  to_dev_batch(*in, &bt);
  smpc::DevEvalOut eo{out->cost, out->cost_plain, out->grad, out->hess, out->ok};
  SMPC_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : h->stream;
  rc = pack_agents(h, &bt, st);
  if (rc != SMPC_OK) return rc;
  SMPC_CUDA(smpc::launch_eval(prm, bt, x, eo, h->n_sm, h->forced_group, st));
  h->launches += 1;
  return SMPC_OK;
}

int smpc_eval_batch(smpc_handle* h, const smpc_batch* in, const double* x, smpc_eval_out* out) {
  if (!h) return fail(SMPC_ERR_ARGUMENT, "handle is NULL");
  int rc = check_batch(in);
  if (rc != SMPC_OK) return rc;
  if (!x || !out) return fail(SMPC_ERR_ARGUMENT, "x / out is NULL");
  if (in->n_problems == 0) return SMPC_OK;
  int nb = 0;
  rc = derive_dims(&h->params, in->n_steps, nullptr, nullptr, &nb, nullptr);
  if (rc != SMPC_OK) return rc;
  smpc_batch din = *in;
  smpc_eval_out dout = *out;
  const double* dx = nullptr;
  {
    std::lock_guard<std::mutex> lk(h->mu);
    SMPC_CUDA(cudaSetDevice(h->device));
    const size_t B = in->n_problems, S1 = static_cast<size_t>(in->n_steps) + 1, A = in->agents ? in->n_agents : 0;
    const size_t M = in->n_costmaps, P = (h->params.omni_solve ? 3 : 2) * static_cast<size_t>(nb), NH = P * (P + 1) / 2;
    const size_t R = in->scenario_index ? static_cast<size_t>(in->n_scenarios) : B;  // rows of the per-scene arrays
    struct Item { const void* host; size_t bytes; void** dev; };
    std::vector<Item> items = {
        {in->pose0, R * 3 * 8, (void**)&din.pose0},
        {in->u0, B * P * 8, (void**)&din.u0},
        {in->path_xy, R * 2 * S1 * 8, (void**)&din.path_xy},
        {in->goal_yaw, R * 8, (void**)&din.goal_yaw},
        {A ? in->agents : nullptr, R * A * 6 * S1 * 8, (void**)&din.agents},
        {in->has_people, R, (void**)&din.has_people},
        {in->costmaps, M * in->size_x * in->size_y, (void**)&din.costmaps},
        {in->costmap_origin, M * 2 * 8, (void**)&din.costmap_origin},
        {in->costmap_index, R * 4, (void**)&din.costmap_index},
        {in->n_steps_each, R * 4, (void**)&din.n_steps_each},
        {in->scenario_index, B * 4, (void**)&din.scenario_index},
        {x, B * P * 8, (void**)&dx},
    };
    size_t total = 0;
    for (auto& it : items) total += it.host ? align256(it.bytes) : 0;
    SMPC_CUDA(h->in_buf.reserve(total));
    Carver cin(h->in_buf.ptr);
    for (auto& it : items) {
      if (!it.host) {
        *it.dev = nullptr;
        continue;
      }
      void* d = cin.take(it.bytes);
      SMPC_CUDA(cudaMemcpyAsync(d, it.host, it.bytes, cudaMemcpyHostToDevice, h->stream));
      *it.dev = d;
    }
    const size_t ob[5] = {B * 8, B * P * 8, B * NH * 8, B, B * 8};
    void* hostp[5] = {out->cost, out->grad, out->hess, out->ok, out->cost_plain};
    void** devp[5] = {(void**)&dout.cost, (void**)&dout.grad, (void**)&dout.hess, (void**)&dout.ok,
                      (void**)&dout.cost_plain};
    size_t ototal = 0;
    for (int i = 0; i < 5; ++i) ototal += hostp[i] ? align256(ob[i]) : 0;
    SMPC_CUDA(h->out_buf.reserve(ototal));
    Carver co(h->out_buf.ptr);
    for (int i = 0; i < 5; ++i) *devp[i] = hostp[i] ? co.take(ob[i]) : nullptr;
  }
  rc = smpc_eval_batch_device(h, &din, dx, &dout, nullptr);
  if (rc != SMPC_OK) return rc;
  {
    std::lock_guard<std::mutex> lk(h->mu);
    const size_t B = in->n_problems, P = (h->params.omni_solve ? 3 : 2) * static_cast<size_t>(nb), NH = P * (P + 1) / 2;
    if (out->cost) SMPC_CUDA(cudaMemcpyAsync(out->cost, dout.cost, B * 8, cudaMemcpyDeviceToHost, h->stream));
    if (out->grad) SMPC_CUDA(cudaMemcpyAsync(out->grad, dout.grad, B * P * 8, cudaMemcpyDeviceToHost, h->stream));
    if (out->hess) SMPC_CUDA(cudaMemcpyAsync(out->hess, dout.hess, B * NH * 8, cudaMemcpyDeviceToHost, h->stream));
    if (out->ok) SMPC_CUDA(cudaMemcpyAsync(out->ok, dout.ok, B, cudaMemcpyDeviceToHost, h->stream));
    if (out->cost_plain)
      SMPC_CUDA(cudaMemcpyAsync(out->cost_plain, dout.cost_plain, B * 8, cudaMemcpyDeviceToHost, h->stream));
    SMPC_CUDA(cudaStreamSynchronize(h->stream));
  }
  return SMPC_OK;
}

int smpc_multistart_argmin_device(smpc_handle* h, int n_robots, int n_starts, int n_blocks, const double* cost_final,
                                  const uint8_t* usable, const double* u, int32_t* best_index, double* best_cost,
                                  double* best_u, void* stream) {
  if (!h) return fail(SMPC_ERR_ARGUMENT, "handle is NULL");
  if (n_robots < 0 || n_starts < 1 || n_blocks < 1 || !cost_final || !best_index || !best_cost)
    return fail(SMPC_ERR_ARGUMENT, "bad multistart arguments");
  if (best_u && !u) return fail(SMPC_ERR_ARGUMENT, "best_u requested without u");
  if (n_robots == 0) return SMPC_OK;
  std::lock_guard<std::mutex> lk(h->mu);
  SMPC_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : h->stream;
  SMPC_CUDA(smpc::launch_argmin(n_robots, n_starts, n_blocks * (h->params.omni_solve ? 3 : 2), cost_final, usable, u, best_index,
                                best_cost, best_u, st));
  h->launches += 1;
  return SMPC_OK;
}

double smpc_last_kernel_ms(smpc_handle* h) {
  if (!h || !h->timed) return -1.0;
  std::lock_guard<std::mutex> lk(h->mu);
  if (cudaEventSynchronize(h->ev1) != cudaSuccess) return -1.0;
  float ms = -1.0f;
  if (cudaEventElapsedTime(&ms, h->ev0, h->ev1) != cudaSuccess) return -1.0;
  return static_cast<double>(ms);
}

long long smpc_launch_count(smpc_handle* h) { return h ? h->launches : 0; }

int smpc_debug_polymin(smpc_handle* h, int n, const double* rows, double* out) {
  if (!h || !rows || !out || n < 0) return fail(SMPC_ERR_ARGUMENT, "bad polymin arguments");
  if (n == 0) return SMPC_OK;
  std::lock_guard<std::mutex> lk(h->mu);
  SMPC_CUDA(cudaSetDevice(h->device));
  SMPC_CUDA(h->in_buf.reserve(sizeof(double) * 10 * n));
  SMPC_CUDA(h->out_buf.reserve(sizeof(double) * n));
  SMPC_CUDA(cudaMemcpyAsync(h->in_buf.ptr, rows, sizeof(double) * 10 * n, cudaMemcpyHostToDevice, h->stream));
  SMPC_CUDA(smpc::launch_polymin(n, static_cast<const double*>(h->in_buf.ptr), static_cast<double*>(h->out_buf.ptr), h->stream));
  SMPC_CUDA(cudaMemcpyAsync(out, h->out_buf.ptr, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
  SMPC_CUDA(cudaStreamSynchronize(h->stream));
  h->launches += 1;
  return SMPC_OK;
}

int smpc_debug_math(smpc_handle* h, int kind, int n, const double* rows, double* out) {
  if (!h || !rows || !out || n < 0 || kind < 0 || kind > 2) return fail(SMPC_ERR_ARGUMENT, "bad debug_math arguments");
  if (n == 0) return SMPC_OK;
  std::lock_guard<std::mutex> lk(h->mu);
  SMPC_CUDA(cudaSetDevice(h->device));
  SMPC_CUDA(h->in_buf.reserve(sizeof(double) * 2 * n));
  SMPC_CUDA(h->out_buf.reserve(sizeof(double) * n));
  SMPC_CUDA(cudaMemcpyAsync(h->in_buf.ptr, rows, sizeof(double) * 2 * n, cudaMemcpyHostToDevice, h->stream));
  SMPC_CUDA(smpc::launch_math(kind, n, static_cast<const double*>(h->in_buf.ptr), static_cast<double*>(h->out_buf.ptr), h->stream));
  SMPC_CUDA(cudaMemcpyAsync(out, h->out_buf.ptr, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
  SMPC_CUDA(cudaStreamSynchronize(h->stream));
  h->launches += 1;
  return SMPC_OK;
}

int smpc_measure_fp64_peak(smpc_handle* h, double* tflops) {
  if (!h || !tflops) return fail(SMPC_ERR_ARGUMENT, "NULL argument");
  std::lock_guard<std::mutex> lk(h->mu);
  SMPC_CUDA(cudaSetDevice(h->device));
  double* sink = nullptr;
  SMPC_CUDA(cudaMalloc(&sink, sizeof(double)));
  const int iters = 4096;
  double best = 0.0;
  cudaEvent_t a, b;
  cudaEventCreate(&a);
  cudaEventCreate(&b);
  for (int rep = 0; rep < 6; ++rep) {
    cudaEventRecord(a, h->stream);
    cudaError_t e = smpc::launch_dfma_peak(sink, h->n_sm, iters, h->stream);
    cudaEventRecord(b, h->stream);
    if (e != cudaSuccess || cudaEventSynchronize(b) != cudaSuccess) {
      cudaFree(sink);
      return cuda_fail(e, "dfma peak kernel");
    }
    float ms = 0.f;
    cudaEventElapsedTime(&ms, a, b);
    const double flops = 2.0 * 8.0 * 16.0 * iters * 256.0 * 8.0 * h->n_sm;
    if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  cudaFree(sink);
  *tflops = best;
  return SMPC_OK;
}

}  // extern "C"
