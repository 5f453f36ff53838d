// smpc_project.cu — batched GPU version of Optimizer::project_people (reference src/optimizer.cpp:554-671) with the
// lightsfm social force model it calls (include/nav2_social_mpc_controller/sfm.hpp:188-323, 462-560) and
// computeObstacle (:673-728). One warp per problem: lanes own people, the horizon is walked sequentially, the agent
// states of the current step live in shared memory. Same arithmetic as the host version in smpc_optimize.cu.
#include <cuda_runtime.h>

#include <cmath>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/smpc.h"
#include "smpc_host_state.h"
#include "smpc_math.cuh"
#include "smpc_sfm.cuh"

namespace {

constexpr int kMaxAgents = 64;  // people + robot
constexpr int kWarps = 4;

struct AgentSmem {  // structure of arrays, one slot per agent of the current step
  double px[kMaxAgents], py[kMaxAgents], vx[kMaxAgents], vy[kMaxAgents];
  double nx[kMaxAgents], ny[kMaxAgents], nvx[kMaxAgents], nvy[kMaxAgents];  // next-step staging
};

using smpc::nearest_obstacle;
using smpc::sfm_pair;
using smpc::wrap_pi;

__global__ void __launch_bounds__(kWarps * 32) smpc_project_kernel(smpc_project_args a) {
  __shared__ AgentSmem sm[kWarps];
  AgentSmem& s = sm[threadIdx.x >> 5];
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int n_warps = (gridDim.x * blockDim.x) >> 5;
  const int A = a.n_agents, stride = a.n_steps + 1;
  const double dt = (double)a.time_step;
  const double kDesired = 2.0, kObstacle = 20.0, kSigma = 0.2, kRelax = 0.5;  // pair-force constants: smpc_sfm.cuh

  for (int b = warp; b < a.n_problems; b += n_warps) {
    // this problem's own horizon (rows keep the stride of the batch's longest one)
    const int S = a.n_steps_each ? min(max(a.n_steps_each[b], 1), a.n_steps) : a.n_steps;
    const double* robot = a.robot + (size_t)b * stride * 6;
    const double* init = a.people_init + (size_t)b * A * 6;
    double* out = a.agents + (size_t)b * A * 6 * stride;
    const int gi = a.od_index ? a.od_index[b] : (b % a.n_grids);
    const uint32_t* idx = a.od_indexes + (size_t)gi * a.od_width * a.od_height;
    const double ox = a.od_origin[2 * gi], oy = a.od_origin[2 * gi + 1];
    const bool grid_ok = !(a.od_width == 100 && a.od_height == 100);  // "grid is NOT valid" (:598-603)
    int err = 0;

    // step 0 = the raw (uncompacted) initial people; invalid everything else for now
    for (int e = lane; e < A * 6; e += 32) {
      const int k = e / 6, c = e % 6;
      out[((size_t)k * 6 + c) * stride] = init[e];
    }
    // compaction of the valid people: slot of agent k = number of valid agents before it
    // per-lane agent state (lane owns compacted slots lane, lane + 32)
    double yaw[2], lv[2], av[2], gx[2], gy[2], obx[2], oby[2], vdes[2];
    bool has_goal[2], mine[2];
    int n = 0;
    {
      int slot_of[2] = {-1, -1};
      // sequential prefix over agents in chunks of 32
      for (int base = 0; base < A; base += 32) {
        const int k = base + lane;
        const bool valid = (k < A) && grid_ok && !(init[k * 6 + 3] == -1.0);
        const unsigned m = __ballot_sync(0xffffffffu, valid);
        const int my_slot = n + __popc(m & ((1u << lane) - 1u));
        if (valid) {
          // hand the agent to the lane that owns its compacted slot through shared memory
          s.px[my_slot] = init[k * 6 + 0];
          s.py[my_slot] = init[k * 6 + 1];
          s.nx[my_slot] = init[k * 6 + 2];   // yaw
          s.ny[my_slot] = init[k * 6 + 4];   // lv
          s.nvx[my_slot] = init[k * 6 + 5];  // av
        }
        n += __popc(m);
      }
      __syncwarp();
      for (int q = 0; q < 2; ++q) {
        const int slot = lane + 32 * q;
        mine[q] = slot < n;
        slot_of[q] = slot;
        yaw[q] = lv[q] = av[q] = gx[q] = gy[q] = obx[q] = oby[q] = 0.0;
        vdes[q] = 0.5;
        has_goal[q] = false;
        if (mine[q]) {
          yaw[q] = s.nx[slot];
          lv[q] = s.ny[slot];
          av[q] = s.nvx[slot];
        }
      }
      __syncwarp();
      for (int q = 0; q < 2; ++q) {
        if (!mine[q]) continue;
        const int slot = slot_of[q];
        double sy, cy;
        sincos(yaw[q], &sy, &cy);
        s.vx[slot] = lv[q] * cy;
        s.vy[slot] = lv[q] * sy;
        gx[q] = s.px[slot] + (double)a.max_time * s.vx[slot];
        gy[q] = s.py[slot] + (double)a.max_time * s.vy[slot];
        has_goal[q] = true;
        if (!nearest_obstacle(a.od_width, a.od_height, a.od_resolution, idx, ox, oy, s.px[slot], s.py[slot], &obx[q], &oby[q]))
          err = 1;
      }
      __syncwarp();
    }
    if (__any_sync(0xffffffffu, err != 0)) {
      // the reference throws here; mark every projected agent invalid and report
      for (int e = lane; e < A * S; e += 32) {
        const int k = e / S, i = e % S + 1;
        for (int c = 0; c < 6; ++c) out[((size_t)k * 6 + c) * stride + i] = (c == 3) ? -1.0 : 0.0;
      }
      if (lane == 0 && a.status) a.status[b] = 1;
      continue;
    }

    const double goal_rx = robot[(size_t)S * 6 + 0], goal_ry = robot[(size_t)S * 6 + 1];
    for (int i = 0; i < S; ++i) {
      // robot appended as agent n (its own force / update are discarded by the reference)
      if (lane == 0) {
        const double ryaw = robot[(size_t)i * 6 + 2], rlv = robot[(size_t)i * 6 + 4];
        double sy, cy;
        sincos(ryaw, &sy, &cy);
        s.px[n] = robot[(size_t)i * 6 + 0];
        s.py[n] = robot[(size_t)i * 6 + 1];
        s.vx[n] = rlv * cy;
        s.vy[n] = rlv * sy;
      }
      __syncwarp();
      for (int q = 0; q < 2; ++q) {
        const int slot = lane + 32 * q;
        if (!mine[q]) continue;
        const double px = s.px[slot], py = s.py[slot], vx = s.vx[slot], vy = s.vy[slot];
        // desired force (sfm.hpp:188-204)
        double fx, fy;
        {
          const double dx = gx[q] - px, dy = gy[q] - py;
          const double dn = sqrt(dx * dx + dy * dy);
          if (has_goal[q] && dn > 0.25) {
            const double z = dx * dx + dy * dy;
            double ex = dx, ey = dy;
            if (z > 0.0) {
              const double sq = sqrt(z);
              ex = dx / sq;
              ey = dy / sq;
            }
            fx = kDesired * (ex * vdes[q] - vx) / kRelax;
            fy = kDesired * (ey * vdes[q] - vy) / kRelax;
          } else {
            fx = -vx / kRelax;
            fy = -vy / kRelax;
          }
        }
        // obstacle force (sfm.hpp:206-221): obstacles1 holds ONE entry
        {
          const double mx = px - obx[q], my = py - oby[q];
          const double mn = sqrt(mx * mx + my * my);
          const double distance = mn - 0.5;
          const double z = mx * mx + my * my;
          double ex = mx, ey = my;
          if (z > 0.0) {
            const double sq = sqrt(z);
            ex = mx / sq;
            ey = my / sq;
          }
          const double k = kObstacle * exp(-distance / kSigma);
          fx += (k * ex) / 1.0;
          fy += (k * ey) / 1.0;
        }
        // social force from every other agent incl. the robot (sfm.hpp:239-281)
        double sfx = 0.0, sfy = 0.0;
        for (int k = 0; k <= n; ++k) {
          if (k == slot) continue;
          const double2 f = sfm_pair(s.px[k] - px, s.py[k] - py, vx - s.vx[k], vy - s.vy[k], sfx, sfy);
          sfx = f.x;
          sfy = f.y;
        }
        fx += sfx;
        fy += sfy;
        // updatePosition (sfm.hpp:512-545)
        double nvx = vx + fx * dt, nvy = vy + fy * dt;
        const double vn = sqrt(nvx * nvx + nvy * nvy);
        if (vn > vdes[q]) {
          const double z = nvx * nvx + nvy * nvy;
          if (z > 0.0) {
            const double sq = sqrt(z);
            nvx = nvx / sq;
            nvy = nvy / sq;
          }
          nvx *= vdes[q];
          nvy *= vdes[q];
        }
        const double y0 = yaw[q];
        yaw[q] = wrap_pi(atan2(nvy, nvx));
        av[q] = wrap_pi(yaw[q] - y0) / dt;
        const double npx = px + nvx * dt, npy = py + nvy * dt;
        lv[q] = sqrt(nvx * nvx + nvy * nvy);
        if (has_goal[q]) {
          const double dx = gx[q] - npx, dy = gy[q] - npy;
          if (sqrt(dx * dx + dy * dy) <= 0.25) has_goal[q] = false;
        }
        s.nx[slot] = npx;
        s.ny[slot] = npy;
        s.nvx[slot] = nvx;
        s.nvy[slot] = nvy;
      }
      __syncwarp();
      for (int q = 0; q < 2; ++q) {
        const int slot = lane + 32 * q;
        if (!mine[q]) continue;
        s.px[slot] = s.nx[slot];
        s.py[slot] = s.ny[slot];
        s.vx[slot] = s.nvx[slot];
        s.vy[slot] = s.nvy[slot];
        if (!nearest_obstacle(a.od_width, a.od_height, a.od_resolution, idx, ox, oy, s.px[slot], s.py[slot], &obx[q], &oby[q]))
          err = 1;
        double* o = out + (size_t)slot * 6 * stride + (i + 1);
        o[0] = s.px[slot];
        o[stride] = s.py[slot];
        o[2 * stride] = yaw[q];
        o[3 * stride] = (double)((float)(i + 1) * a.time_step);
        o[4 * stride] = lv[q];
        o[5 * stride] = av[q];
      }
      // padded (invalid) columns of this step
      for (int k = n + lane; k < A; k += 32) {
        double* o = out + (size_t)k * 6 * stride + (i + 1);
        o[0] = 0.0; o[stride] = 0.0; o[2 * stride] = 0.0; o[3 * stride] = -1.0; o[4 * stride] = 0.0; o[5 * stride] = 0.0;
      }
      __syncwarp();
    }
    const bool any_err = __any_sync(0xffffffffu, err != 0);
    if (lane == 0 && a.status) a.status[b] = any_err ? 1 : 0;
  }
}

// format_to_optimize (reference src/optimizer.cpp:484-551) + unpacking (:197-237), one thread per (problem, pose).
// P = a.n_poses is the row stride; robot b keeps Pb = n_poses_each[b] poses (the caller has applied the max_time cut).
__global__ void smpc_format_kernel(smpc_format_args a) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int P = a.n_poses;
  if (t >= (long long)a.n_problems * P) return;
  const int b = (int)(t / P), i = (int)(t % P);
  const int Pb = a.n_poses_each ? a.n_poses_each[b] : P;
  if (Pb < 2) {
    // inactive robot ("Path has less than 2 points", :158-162): give the solve a finite one-step dummy, no people
    if (i == 0) {
      for (int c = 0; c < 3; ++c) a.pose0[3 * b + c] = 0.0;
      for (int c = 0; c < 2 * a.n_blocks; ++c) a.u0[(size_t)b * a.n_blocks * 2 + c] = 0.0;
      a.goal_yaw[b] = 0.0;
      for (int k = 0; k < 2; ++k) {
        a.path_xy[(size_t)b * 2 * P + k] = 0.0;
        a.path_xy[(size_t)b * 2 * P + P + k] = 0.0;
        for (int c = 0; c < 6; ++c) a.robot[((size_t)b * P + k) * 6 + c] = 0.0;
      }
      if (a.has_people) a.has_people[b] = 0;
    }
    return;
  }
  if (i >= Pb) return;
  const double* cp = a.poses + ((size_t)b * P + i) * 3;
  const int n_prev_poses_b = a.n_prev_poses_each ? a.n_prev_poses_each[b] : a.n_prev_poses;
  const bool have_prev = a.prev_poses != nullptr && n_prev_poses_b > 0;
  // first tick: previous = current (TrajectoryMemory seeding, :177-181) -> blending happens against itself
  const int n_prev_poses = have_prev ? n_prev_poses_b : Pb;
  const double wp = a.current_path_w, wc = a.current_cmds_w;
  double x = cp[0], y = cp[1], yaw = cp[2];
  if (i < n_prev_poses) {
    const double* pp = have_prev ? a.prev_poses + ((size_t)b * a.n_prev_poses + i) * 3 : cp;
    x = wp * cp[0] + (1.0 - wp) * pp[0];
    y = wp * cp[1] + (1.0 - wp) * pp[1];
    const double sm = wp * cp[2] + (1.0 - wp) * pp[2];
    double sh, ch;
    sincos(sm * 0.5, &sh, &ch);
    yaw = atan2(2.0 * (ch * sh), ch * ch - sh * sh);  // setRPY -> getYaw (:517-525)
  }
  double lv, av;
  if (i == 0) {
    lv = a.speed[2 * b];
    av = a.speed[2 * b + 1];
  } else {
    const int cstride = a.cmds_stride > 0 ? a.cmds_stride : P - 1;
    const double* cc = a.cmds + ((size_t)b * cstride + (i - 1)) * 2;
    const int n_prev_cmds_b = a.n_prev_cmds_each ? a.n_prev_cmds_each[b] : a.n_prev_cmds;
    const bool have_pc = a.prev_cmds != nullptr && (i - 1) < n_prev_cmds_b;  // SURVEY Q11 guard
    const double* pc = have_pc ? a.prev_cmds + ((size_t)b * a.n_prev_cmds + (i - 1)) * 2 : cc;
    lv = wc * cc[0] + (1.0 - wc) * pc[0];
    av = wc * cc[1] + (1.0 - wc) * pc[1];
  }
  double* r = a.robot + ((size_t)b * P + i) * 6;
  r[0] = x; r[1] = y; r[2] = yaw; r[3] = (double)((float)i * a.time_step); r[4] = lv; r[5] = av;
  a.path_xy[(size_t)b * 2 * P + i] = x;
  a.path_xy[(size_t)b * 2 * P + P + i] = y;
  if (i < a.n_blocks) {
    a.u0[((size_t)b * a.n_blocks + i) * 2] = lv;  // block b starts at the seed velocity of time index b (Q1)
    a.u0[((size_t)b * a.n_blocks + i) * 2 + 1] = av;
  }
  if (i == 0) {
    double sh, ch;
    sincos(yaw * 0.5, &sh, &ch);
    a.pose0[3 * b] = x;
    a.pose0[3 * b + 1] = y;
    a.pose0[3 * b + 2] = atan2(2.0 * (ch * sh), ch * ch - sh * sh);  // evolving_poses[0]: setRPY (:224-226) + getYaw
  }
  if (i == Pb - 1) a.goal_yaw[b] = yaw;
}

// PathTrajectorizer::trajectorize (reference src/path_trajectorizer.cpp:120-288): pure-pursuit seed of up to max_steps
// Euler steps. One WARP per robot: the time loop is sequential, but every step searches the whole global path for its
// look-ahead point ("scanning from the end, the first pose within lookahead_dist, else the nearest one"), and that
// search is done by the 32 lanes at once — the look-ahead point is the LARGEST index within reach (a ballot per 32
// points, taken from the end), else an arg-min with the serial loop's tie rule (strict '<' while walking down: the
// larger index wins). Every lane then advances the same robot state, so no broadcast is needed. Decisions are
// bit-identical to the serial scan (same sqrt(dx^2 + dy^2) per point).
__global__ void __launch_bounds__(128) smpc_trajectorize_kernel(smpc_trajectorize_args a) {
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (b >= a.n_problems) return;
  const int N = a.n_path;
  const double* path = a.global_path + (size_t)(a.path_index ? a.path_index[b] : b) * N * 2;
  double rx = a.pose[3 * b], ry = a.pose[3 * b + 1];
  double rth;
  {
    double sh, ch;
    sincos(a.pose[3 * b + 2] * 0.5, &sh, &ch);
    rth = atan2(2.0 * (ch * sh), ch * ch - sh * sh);  // tf2::getYaw(robot_pose.pose.orientation)
  }
  double* poses = a.poses + (size_t)b * (a.max_steps + 1) * 3;
  double* cmds = a.cmds + (size_t)b * a.max_steps * 3;
  if (lane == 0) {
    poses[0] = rx; poses[1] = ry; poses[2] = rth;
  }
  const double gx = path[2 * (N - 1)], gy = path[2 * (N - 1) + 1];
  double goal_dist = 1000.0;
  int steps = 0;
  while (goal_dist > 0.2 && steps < a.max_steps) {
    // look-ahead point
    int wp = -1;
    double best_d = 100.0;  // the reference's initial min_dist
    int best_i = -1;
    for (int top = N - 1; top >= 0 && wp < 0; top -= 32) {
      const int i = top - lane;
      double d = INFINITY;
      if (i >= 0) {
        const double dx = rx - path[2 * i], dy = ry - path[2 * i + 1];
        d = sqrt(dx * dx + dy * dy);
      }
      const unsigned hit = __ballot_sync(0xffffffffu, d <= a.lookahead_dist);
      if (hit) {
        wp = top - (__ffs(hit) - 1);  // lowest lane = largest index of this group of 32
      } else if (d < best_d) {        // within a lane the indices only go down: strict '<' keeps the larger one
        best_d = d;
        best_i = i;
      }
    }
    if (wp < 0) {  // nothing within reach: nearest pose, ties to the larger index
      for (int off = 16; off > 0; off >>= 1) {
        const double od = __shfl_xor_sync(0xffffffffu, best_d, off);
        const int oi = __shfl_xor_sync(0xffffffffu, best_i, off);
        if (od < best_d || (od == best_d && oi > best_i)) {
          best_d = od;
          best_i = oi;
        }
      }
      wp = best_i;
    }
    if (wp < 0) wp = N - 1;  // every pose farther than 100 m: the reference would index -1 (UB); take the goal
    const double wpx = path[2 * wp], wpy = path[2 * wp + 1];
    double st, ct;
    sincos(rth, &st, &ct);
    const double dx = (wpx - rx) * ct + (wpy - ry) * st;
    const double dy = -(wpx - rx) * st + (wpy - ry) * ct;
    const double dtheta = atan2(dy, dx);
    double vx = 0.0, vy = 0.0, wz = 0.0;
    if (a.omnidirectional) {
      vx = a.desired_linear_vel * cos(dtheta);
      vy = a.desired_linear_vel * sin(dtheta);
    } else {
      const double d2 = dx * dx + dy * dy;
      double curvature = 0.0;
      if (d2 > 0.001) curvature = 2.0 * dy / d2;
      vx = a.desired_linear_vel;
      if (fabs(dtheta) > M_PI / 2.0) {
        vx = 0.0;
        wz = a.max_angular_vel * (dtheta > 0 ? 1.0 : -1.0);
      } else {
        wz = vx * curvature;
      }
    }
    // computeNewX/Y/ThetaPosition (path_trajectorizer.hpp:106-133)
    rx = rx + (vx * ct + vy * cos(M_PI_2 + rth)) * a.time_step;
    ry = ry + (vx * st + vy * sin(M_PI_2 + rth)) * a.time_step;
    rth = rth + wz * a.time_step;
    if (lane == 0) {
      double sh, ch;
      sincos(rth * 0.5, &sh, &ch);
      poses[3 * (steps + 1)] = rx;
      poses[3 * (steps + 1) + 1] = ry;
      poses[3 * (steps + 1) + 2] = atan2(2.0 * (ch * sh), ch * ch - sh * sh);  // setRPY(0, 0, rtheta) read back by getYaw
      cmds[3 * steps] = vx;
      cmds[3 * steps + 1] = vy;
      cmds[3 * steps + 2] = wz;
    }
    const double ex = rx - gx, ey = ry - gy;
    goal_dist = sqrt(ex * ex + ey * ey);
    ++steps;
  }
  if (lane == 0) a.n_steps[b] = steps;
}

__global__ void smpc_people_status_kernel(int B, int A, const double* __restrict__ raw, const int32_t* __restrict__ n_people,
                                          double* __restrict__ init, uint8_t* __restrict__ has_people) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)B * A) return;
  const int b = (int)(t / A), k = (int)(t % A);
  const int n = n_people[b];
  double* o = init + (size_t)t * 6;
  if (k < n) {
    const double* p = raw + (size_t)t * 5;
    o[0] = p[0]; o[1] = p[1]; o[2] = atan2(p[3], p[2]); o[3] = 0.0; o[4] = sqrt(p[2] * p[2] + p[3] * p[3]); o[5] = p[4];
  } else {  // invalid agent: time = -1 (:468-474)
    o[0] = 0.0; o[1] = 0.0; o[2] = 0.0; o[3] = -1.0; o[4] = 0.0; o[5] = 0.0;
  }
  if (k == 0 && has_people) has_people[b] = n != 0;
}

__global__ void smpc_memory_update_kernel(int B, int n, const uint8_t* __restrict__ usable, const double* __restrict__ path,
                                          const double* __restrict__ cmds, double* __restrict__ prev_poses,
                                          double* __restrict__ prev_cmds) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)B * n) return;
  const int b = (int)(t / n);
  if (!usable[b]) return;
  for (int c = 0; c < 3; ++c) prev_poses[t * 3 + c] = path[t * 3 + c];
  for (int c = 0; c < 2; ++c) prev_cmds[t * 2 + c] = cmds[t * 2 + c];
}

}  // namespace

extern "C" {

int smpc_trajectorize_batch_device(smpc_handle* h, const smpc_trajectorize_args* a, void* stream) {
  if (!h || !a) return smpc_host_fail(SMPC_ERR_ARGUMENT, "NULL argument");
  if (a->n_path < 2) return smpc_host_fail(SMPC_ERR_ARGUMENT, "Path has less than 2 poses, cannot trajectorize");
  if (a->n_problems < 0 || a->max_steps < 1 || !(a->time_step > 0.0) || !a->global_path || !a->pose || !a->poses ||
      !a->cmds || !a->n_steps)
    return smpc_host_fail(SMPC_ERR_ARGUMENT, "trajectorize: bad arguments");
  if (a->n_problems == 0) return SMPC_OK;
  cudaSetDevice(smpc_handle_device(h));  // the caller may have another device current (multi-GPU processes)
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : smpc_handle_stream(h);
  smpc_trajectorize_kernel<<<(a->n_problems + 3) / 4, 128, 0, st>>>(*a);  // one warp per robot
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return smpc_host_fail(SMPC_ERR_CUDA, std::string("trajectorize kernel: ") + cudaGetErrorString(e));
  smpc_handle_count_launch(h);
  return SMPC_OK;
}

int smpc_people_to_status_device(smpc_handle* h, int n_problems, int n_agents, const double* people_raw,
                                 const int32_t* n_people, double* people_init, uint8_t* has_people, void* stream) {
  if (!h || n_problems < 0 || n_agents < 1 || !people_raw || !n_people || !people_init)
    return smpc_host_fail(SMPC_ERR_ARGUMENT, "people_to_status: bad arguments");
  if (n_problems == 0) return SMPC_OK;
  cudaSetDevice(smpc_handle_device(h));  // the caller may have another device current (multi-GPU processes)
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : smpc_handle_stream(h);
  const long long n = (long long)n_problems * n_agents;
  smpc_people_status_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n_problems, n_agents, people_raw, n_people, people_init,
                                                                       has_people);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return smpc_host_fail(SMPC_ERR_CUDA, std::string("people_status kernel: ") + cudaGetErrorString(e));
  smpc_handle_count_launch(h);
  return SMPC_OK;
}

int smpc_memory_update_device(smpc_handle* h, int n_problems, int n, const uint8_t* usable, const double* path,
                              const double* cmds, double* prev_poses, double* prev_cmds, void* stream) {
  if (!h || n_problems < 0 || n < 1 || !usable || !path || !cmds || !prev_poses || !prev_cmds)
    return smpc_host_fail(SMPC_ERR_ARGUMENT, "memory_update: bad arguments");
  if (n_problems == 0) return SMPC_OK;
  cudaSetDevice(smpc_handle_device(h));  // the caller may have another device current (multi-GPU processes)
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : smpc_handle_stream(h);
  const long long total = (long long)n_problems * n;
  smpc_memory_update_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(n_problems, n, usable, path, cmds, prev_poses,
                                                                           prev_cmds);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return smpc_host_fail(SMPC_ERR_CUDA, std::string("memory_update kernel: ") + cudaGetErrorString(e));
  smpc_handle_count_launch(h);
  return SMPC_OK;
}


int smpc_format_batch_device(smpc_handle* h, const smpc_format_args* a, void* stream) {
  if (!h || !a) return smpc_host_fail(SMPC_ERR_ARGUMENT, "NULL argument");
  if (a->n_problems < 0 || a->n_poses < 2 || a->n_blocks < 1 || a->n_blocks > a->n_poses - 1)
    return smpc_host_fail(SMPC_ERR_ARGUMENT, "format: need n_poses >= 2 and 1 <= n_blocks <= n_poses - 1");
  if (!a->poses || !a->cmds || !a->speed || !a->robot || !a->pose0 || !a->u0 || !a->path_xy || !a->goal_yaw)
    return smpc_host_fail(SMPC_ERR_ARGUMENT, "format: missing buffer");
  if (a->n_problems == 0) return SMPC_OK;
  cudaSetDevice(smpc_handle_device(h));  // the caller may have another device current (multi-GPU processes)
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : smpc_handle_stream(h);
  const long long n = (long long)a->n_problems * a->n_poses;
  smpc_format_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(*a);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return smpc_host_fail(SMPC_ERR_CUDA, std::string("format kernel: ") + cudaGetErrorString(e));
  smpc_handle_count_launch(h);
  return SMPC_OK;
}


int smpc_project_people_batch_device(smpc_handle* h, const smpc_project_args* a, void* stream) {
  if (!h || !a) return smpc_host_fail(SMPC_ERR_ARGUMENT, "NULL argument");
  if (a->n_problems < 0 || a->n_steps < 1 || a->n_agents < 1 || a->n_agents > kMaxAgents - 1)
    return smpc_host_fail(SMPC_ERR_ARGUMENT, "project_people: need n_steps >= 1 and 1 <= n_agents <= 63");
  if (!a->robot || !a->people_init || !a->agents || !a->od_indexes || !a->od_origin || a->n_grids < 1)
    return smpc_host_fail(SMPC_ERR_ARGUMENT, "project_people: missing buffer");
  if (a->od_width == 0 || a->od_height == 0) return smpc_host_fail(SMPC_ERR_ARGUMENT, "ObstacleDistance grid has invalid size");
  if (!(a->od_resolution > 0.0f)) return smpc_host_fail(SMPC_ERR_ARGUMENT, "ObstacleDistance grid has invalid resolution");
  if (a->n_problems == 0) return SMPC_OK;
  cudaSetDevice(smpc_handle_device(h));  // the caller may have another device current (multi-GPU processes)
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : smpc_handle_stream(h);
  const int ctas = (a->n_problems + kWarps - 1) / kWarps;
  const int grid = ctas < 148 * 8 ? ctas : 148 * 8;
  smpc_project_kernel<<<grid, kWarps * 32, 0, st>>>(*a);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return smpc_host_fail(SMPC_ERR_CUDA, std::string("project kernel: ") + cudaGetErrorString(e));
  smpc_handle_count_launch(h);
  return SMPC_OK;
}

int smpc_project_people_batch(smpc_handle* h, const smpc_project_args* a) {
  if (!h || !a) return smpc_host_fail(SMPC_ERR_ARGUMENT, "NULL argument");
  if (a->n_problems <= 0) return SMPC_OK;
  const size_t B = a->n_problems, S1 = (size_t)a->n_steps + 1, A = a->n_agents, M = a->n_grids;
  const size_t cells = (size_t)a->od_width * a->od_height;
  smpc_project_args d = *a;
  std::vector<void*> to_free;
  auto up = [&](const void* host, size_t bytes) -> void* {
    if (!host) return nullptr;
    void* p = nullptr;
    if (cudaMalloc(&p, bytes) != cudaSuccess) return nullptr;
    to_free.push_back(p);
    cudaMemcpy(p, host, bytes, cudaMemcpyHostToDevice);
    return p;
  };
  d.od_origin = (const double*)up(a->od_origin, M * 2 * 8);
  d.od_indexes = (const uint32_t*)up(a->od_indexes, M * cells * 4);
  d.od_index = (const int32_t*)up(a->od_index, B * 4);
  d.robot = (const double*)up(a->robot, B * S1 * 6 * 8);
  d.people_init = (const double*)up(a->people_init, B * A * 6 * 8);
  void* dout = nullptr;
  void* dstat = nullptr;
  cudaMalloc(&dout, B * A * 6 * S1 * 8);
  cudaMalloc(&dstat, B * 4);
  to_free.push_back(dout);
  to_free.push_back(dstat);
  d.agents = (double*)dout;
  d.status = (int32_t*)dstat;
  int rc = smpc_project_people_batch_device(h, &d, nullptr);
  if (rc == SMPC_OK) {
    cudaStreamSynchronize(smpc_handle_stream(h));
    cudaMemcpy(a->agents, dout, B * A * 6 * S1 * 8, cudaMemcpyDeviceToHost);
    if (a->status) cudaMemcpy(a->status, dstat, B * 4, cudaMemcpyDeviceToHost);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) rc = smpc_host_fail(SMPC_ERR_CUDA, std::string("project_people: ") + cudaGetErrorString(e));
  }
  for (void* p : to_free) cudaFree(p);
  return rc;
}

}  // extern "C"

// ===================================================================================================================
// FOV people filter of SocialMPCController::computeVelocityCommands (reference src/social_mpc_controller.cpp:198-214)
// for a fleet: a person is kept when Costmap2D::worldToMap succeeds for its position and |bearing - yaw| < fov_angle,
// with the reference's FLOAT roundings (angle_to_person, robot_yaw and relative_angle are floats there). One thread
// per robot walks its people in order (the filter is an order-preserving compaction; only the first A_out survive,
// people_to_status keeps three, src/optimizer.cpp:476-479).
// ===================================================================================================================
namespace {
__global__ void smpc_fov_filter_kernel(smpc_fov_args a) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= a.n_robots) return;
  const int mi = a.costmap_index ? a.costmap_index[b] : (b % a.n_costmaps);
  const double ox = a.costmap_origin[2 * mi], oy = a.costmap_origin[2 * mi + 1];
  const double px = a.pose[3 * b], py = a.pose[3 * b + 1];
  double sh, ch;
  sincos(a.pose[3 * b + 2] * 0.5, &sh, &ch);
  const float robot_yaw = (float)atan2(2.0 * (ch * sh), ch * ch - sh * sh);  // tf2::getYaw of the pose quaternion
  const double* in = a.people_in + (size_t)b * a.n_in_max * 5;
  double* out = a.people_out + (size_t)b * a.n_out_max * 5;
  const int n = min(a.n_people_in[b], a.n_in_max);
  int kept = 0, total = 0;
  for (int k = 0; k < n; ++k) {
    const double wx = in[5 * k], wy = in[5 * k + 1];
    // Costmap2D::worldToMap
    if (wx < ox || wy < oy) continue;
    const unsigned mx = (unsigned)((wx - ox) / a.resolution), my = (unsigned)((wy - oy) / a.resolution);
    if (!(mx < (unsigned)a.size_x && my < (unsigned)a.size_y)) continue;
    const float angle_to_person = (float)atan2(wy - py, wx - px);
    // angles::shortest_angular_distance(from, to) = normalize_angle(to - from), evaluated in double on the float values
    const double diff = (double)angle_to_person - (double)robot_yaw;
    const double norm = fmod(fmod(diff + M_PI, 2.0 * M_PI) + 2.0 * M_PI, 2.0 * M_PI) - M_PI;
    const float relative_angle = (float)norm;
    if (fabs((double)relative_angle) < a.fov_angle) {
      if (kept < a.n_out_max) {
        for (int c = 0; c < 5; ++c) out[5 * kept + c] = in[5 * k + c];
        ++kept;
      }
      ++total;
    }
  }
  for (int k = kept; k < a.n_out_max; ++k)
    for (int c = 0; c < 5; ++c) out[5 * k + c] = 0.0;
  a.n_people_out[b] = total;  // people.people.size() after the filter (has_people = total != 0, :263)
}
}  // namespace

extern "C" {
int smpc_fov_filter_batch_device(smpc_handle* h, const smpc_fov_args* a, void* stream) {
  if (!h || !a) return smpc_host_fail(SMPC_ERR_ARGUMENT, "NULL argument");
  if (a->n_robots < 0 || a->n_in_max < 1 || a->n_out_max < 1 || a->n_costmaps < 1 || !a->people_in || !a->n_people_in ||
      !a->pose || !a->costmap_origin || !a->people_out || !a->n_people_out || !(a->resolution > 0.0))
    return smpc_host_fail(SMPC_ERR_ARGUMENT, "fov_filter: bad arguments");
  if (a->n_robots == 0) return SMPC_OK;
  cudaSetDevice(smpc_handle_device(h));
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : smpc_handle_stream(h);
  smpc_fov_filter_kernel<<<(a->n_robots + 127) / 128, 128, 0, st>>>(*a);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return smpc_host_fail(SMPC_ERR_CUDA, std::string("fov filter kernel: ") + cudaGetErrorString(e));
  smpc_handle_count_launch(h);
  return SMPC_OK;
}
}  // extern "C"

// ===================================================================================================================
// Level-2 BATCH entry: smpc_optimize_batch = bool Optimizer::optimize(...) (reference src/optimizer.cpp:148-452) for a
// fleet of B robots per call, every stage a kernel on the handle's stream, per-robot horizons, per-robot warm-start
// memory (previous path / cmds) resident on the device between ticks.
// ===================================================================================================================
namespace {

// TrajectoryMemory seeding (:177-181): a robot without memory gets its CURRENT (uncut) seed as "previous".
__global__ void fleet_seed_memory_kernel(int B, int stride, const int32_t* __restrict__ n_in, const double* __restrict__ poses,
                                         const double* __restrict__ cmds, double* __restrict__ prev_poses,
                                         double* __restrict__ prev_cmds, const int32_t* __restrict__ n_prev_poses) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)B * stride) return;
  const int b = (int)(t / stride), i = (int)(t % stride);
  const int n = n_in[b];
  if (n < 2 || n_prev_poses[b] != 0) return;
  if (i < n)
    for (int c = 0; c < 3; ++c) prev_poses[t * 3 + c] = poses[t * 3 + c];
  if (i < n - 1)
    for (int c = 0; c < 2; ++c) prev_cmds[t * 2 + c] = cmds[t * 2 + c];
}

__global__ void fleet_seed_len_kernel(int B, const int32_t* __restrict__ n_in, int32_t* n_prev_poses, int32_t* n_prev_cmds) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  if (n_in[b] >= 2 && n_prev_poses[b] == 0) {
    n_prev_poses[b] = n_in[b];
    n_prev_cmds[b] = n_in[b] - 1;
  }
}

// Post-solve (:384-449): where the solve is usable the optimised path / cmds replace the seed and become the robot's
// memory; where it is not (or a person left the obstacle grid: the reference throws there) the robot keeps its cmds,
// its path is the cut + blended seed format_to_optimize left behind, and its memory stays as it was.
struct FleetFinish {
  int B, stride;
  const int32_t* n_in;
  const int32_t* n_each;  // poses optimised per robot (after the max_time cut), 0 = inactive (fewer than 2 poses)
  const uint8_t* usable;
  const int32_t* status;
  const double* robot;     // [B][stride][6] blended seed
  const double* path;      // [B][stride][3] solve output
  const double* cmds_new;  // [B][stride][2] solve output
  double* poses_io;        // [B][stride][3] in: seed, out: result
  double* cmds_io;         // [B][stride][2]
  double* prev_poses;
  double* prev_cmds;
  int32_t* n_prev_poses;
  int32_t* n_prev_cmds;
  int32_t* n_out;
  uint8_t* optimized;
};

__global__ void fleet_finish_kernel(FleetFinish a) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)a.B * a.stride) return;
  const int b = (int)(t / a.stride), i = (int)(t % a.stride);
  const int n = a.n_each[b];
  const bool active = n >= 2;
  const bool ok = active && a.usable[b] != 0 && a.status[b] == 0;
  if (i == 0) {
    a.optimized[b] = ok ? 1 : 0;
    a.n_out[b] = active ? n : a.n_in[b];
    if (ok) {
      a.n_prev_poses[b] = n;
      a.n_prev_cmds[b] = n;
    }
  }
  if (!active || i >= n) return;
  if (ok) {
    for (int c = 0; c < 3; ++c) {
      const double v = a.path[t * 3 + c];
      a.poses_io[t * 3 + c] = v;
      a.prev_poses[t * 3 + c] = v;
    }
    for (int c = 0; c < 2; ++c) {
      const double v = a.cmds_new[t * 2 + c];
      a.cmds_io[t * 2 + c] = v;
      a.prev_cmds[t * 2 + c] = v;
    }
  } else {
    for (int c = 0; c < 3; ++c) a.poses_io[t * 3 + c] = a.robot[t * 6 + c];
  }
}

using Carve = smpc_carve;
#define FLEET_CUDA SMPC_FLEET_CUDA

}  // namespace

void smpc_fleet_carve_stages(smpc_carve& c, smpc_fleet_dev* d) {
  const size_t B = d->B, BS = B * d->stride, A = d->A;
  d->init = c.take<double>(B * A * 6);
  d->has_people = c.take<uint8_t>(B);
  d->robot = c.take<double>(BS * 6);
  d->pose0 = c.take<double>(B * 3);
  d->u0 = c.take<double>(B * d->nb * 2);
  d->path_xy = c.take<double>(BS * 2);
  d->goal_yaw = c.take<double>(B);
  d->agents = c.take<double>(B * A * 6 * d->stride);
  d->cmds_new = c.take<double>(BS * 2);
  d->path_new = c.take<double>(BS * 3);
  d->usable = c.take<uint8_t>(B);
  d->term = c.take<int32_t>(B);
  d->iters = c.take<int32_t>(B);
  d->cost0 = c.take<double>(B);
  d->cost1 = c.take<double>(B);
  d->n_out = c.take<int32_t>(B);
  d->optimized = c.take<uint8_t>(B);
  d->status = c.take<int32_t>(B);
}

cudaError_t smpc_fleet_memory(smpc_fleet_state* fs, smpc_fleet_dev* d, cudaStream_t st) {
  const int B = d->B, stride = d->stride;
  if (fs->mem_robots != B || fs->mem_stride != stride) {
    const size_t bytes = (size_t)B * stride * 5 * sizeof(double) + 2 * (size_t)B * sizeof(int32_t) + 1024;
    cudaError_t e = fs->memory.reserve(bytes);
    if (e == cudaSuccess) e = cudaMemsetAsync(fs->memory.ptr, 0, bytes, st);
    if (e != cudaSuccess) return e;
    fs->mem_robots = B;
    fs->mem_stride = stride;
  }
  Carve cm(fs->memory.ptr);
  d->prev_poses = cm.take<double>((size_t)B * stride * 3);
  d->prev_cmds = cm.take<double>((size_t)B * stride * 2);
  d->n_prev_poses = cm.take<int32_t>(B);
  d->n_prev_cmds = cm.take<int32_t>(B);
  return cudaSuccess;
}

int smpc_fleet_tick_enqueue(smpc_handle* h, const smpc_fleet_dev& d, cudaStream_t st) {
  const int B = d.B, stride = d.stride, A = d.A, S = stride - 1;
  const size_t BS = (size_t)B * stride;
  FLEET_CUDA(cudaMemsetAsync(d.status, 0, (size_t)B * 4, st));

  const unsigned g_bs = (unsigned)((BS + 255) / 256), g_b = (unsigned)((B + 255) / 256);
  // ---- TrajectoryMemory seeding, people_to_status, format_to_optimize, project_people
  fleet_seed_memory_kernel<<<g_bs, 256, 0, st>>>(B, stride, d.n_in, d.poses, d.cmds, d.prev_poses, d.prev_cmds,
                                                 d.n_prev_poses);
  fleet_seed_len_kernel<<<g_b, 256, 0, st>>>(B, d.n_in, d.n_prev_poses, d.n_prev_cmds);
  smpc_people_status_kernel<<<(unsigned)(((size_t)B * A + 255) / 256), 256, 0, st>>>(B, A, d.people, d.n_people, d.init,
                                                                                    d.has_people);
  smpc_format_args fa{};
  fa.n_problems = B; fa.n_poses = stride; fa.n_prev_poses = stride; fa.n_prev_cmds = stride; fa.n_blocks = d.nb;
  fa.time_step = d.time_step; fa.current_path_w = smpc_handle_params(h)->current_path_w;
  fa.current_cmds_w = smpc_handle_params(h)->current_cmds_w;
  fa.poses = d.poses; fa.cmds = d.cmds; fa.speed = d.speed; fa.prev_poses = d.prev_poses; fa.prev_cmds = d.prev_cmds;
  fa.robot = d.robot; fa.pose0 = d.pose0; fa.u0 = d.u0; fa.path_xy = d.path_xy; fa.goal_yaw = d.goal_yaw;
  fa.n_poses_each = d.n_each; fa.n_prev_poses_each = d.n_prev_poses; fa.n_prev_cmds_each = d.n_prev_cmds;
  fa.cmds_stride = stride; fa.has_people = d.has_people;
  smpc_format_kernel<<<g_bs, 256, 0, st>>>(fa);
  smpc_project_args pa{};
  pa.n_problems = B; pa.n_steps = S; pa.n_agents = A; pa.n_grids = d.n_od_grids;
  pa.od_width = d.od_width; pa.od_height = d.od_height; pa.od_resolution = d.od_resolution;
  pa.max_time = d.max_time; pa.time_step = d.time_step;
  pa.od_origin = d.od_org; pa.od_indexes = d.od; pa.od_index = d.od_index;
  pa.robot = d.robot; pa.people_init = d.init; pa.agents = d.agents; pa.status = d.status; pa.n_steps_each = d.s_each;
  {
    const int ctas = (B + kWarps - 1) / kWarps;
    smpc_project_kernel<<<ctas < 148 * 8 ? ctas : 148 * 8, kWarps * 32, 0, st>>>(pa);
  }
  FLEET_CUDA(cudaGetLastError());
  for (int k = 0; k < 5; ++k) smpc_handle_count_launch(h);

  // ---- the solve (level-1 path, per-robot horizons) with its post-solve expansion
  smpc_batch bt{};
  bt.n_problems = B; bt.n_steps = S; bt.n_agents = A; bt.n_costmaps = d.n_costmaps;
  bt.size_x = d.size_x; bt.size_y = d.size_y; bt.resolution = d.resolution; bt.dt = (double)d.time_step;
  bt.pose0 = d.pose0; bt.u0 = d.u0; bt.path_xy = d.path_xy; bt.goal_yaw = d.goal_yaw; bt.agents = d.agents;
  bt.has_people = d.has_people; bt.costmaps = d.maps; bt.costmap_origin = d.map_org;
  bt.costmap_index = d.map_index; bt.n_steps_each = d.s_each;
  smpc_result rs{};
  rs.cmds = d.cmds_new; rs.path = d.path_new; rs.usable = d.usable; rs.termination = d.term; rs.iterations = d.iters;
  rs.cost_initial = d.cost0; rs.cost_final = d.cost1;
  const int rc = d.weights ? smpc_solve_batch_weighted(h, &bt, &rs, d.weights, d.weight_set, st)
                           : smpc_solve_batch_device(h, &bt, &rs, st);
  if (rc != SMPC_OK) return rc;

  // ---- post-solve: outputs, memory update
  FleetFinish ff{B, stride, d.n_in, d.n_each, d.usable, d.status, d.robot, d.path_new, d.cmds_new, d.poses, d.cmds,
                 d.prev_poses, d.prev_cmds, d.n_prev_poses, d.n_prev_cmds, d.n_out, d.optimized};
  fleet_finish_kernel<<<g_bs, 256, 0, st>>>(ff);
  FLEET_CUDA(cudaGetLastError());
  smpc_handle_count_launch(h);
  return SMPC_OK;
}

int smpc_check_weight_sets(const smpc_weight_sets* w, int n, const char* name) {
  const std::string pre = std::string(name) + ": ";
  if (!w) return smpc_host_fail(SMPC_ERR_ARGUMENT, pre + "NULL weight sets");
  if (w->n_sets < 1) return smpc_host_fail(SMPC_ERR_ARGUMENT, pre + "n_sets < 1");
  if (!w->weights || !w->set_index) return smpc_host_fail(SMPC_ERR_ARGUMENT, pre + "weights / set_index missing");
  for (size_t i = 0; i < (size_t)w->n_sets * 9; ++i)
    if (!std::isfinite(w->weights[i])) return smpc_host_fail(SMPC_ERR_ARGUMENT, pre + "a weight is not finite");
  for (int b = 0; b < n; ++b)
    if (w->set_index[b] < 0 || w->set_index[b] >= w->n_sets)
      return smpc_host_fail(SMPC_ERR_ARGUMENT, pre + "set_index[b] outside 0..n_sets-1");
  return SMPC_OK;
}

int smpc_optimize_batch_on(smpc_handle* h, smpc_fleet_state* fs, smpc_fleet_io* io, const smpc_weight_sets* w) {
  if (!h || !io || !fs) return smpc_host_fail(SMPC_ERR_ARGUMENT, "NULL argument");
  const int B = io->n_robots, stride = io->max_poses, A = io->n_agents;
  if (B < 0 || stride < 2 || A < 1 || A > kMaxAgents - 1)
    return smpc_host_fail(SMPC_ERR_ARGUMENT, "optimize_batch: need n_robots >= 0, max_poses >= 2, 1 <= n_agents <= 63");
  if (B == 0) return SMPC_OK;
  if (!io->n_poses || !io->poses || !io->cmds || !io->people || !io->n_people || !io->speed || !io->costmaps ||
      !io->costmap_origin || io->n_costmaps < 1 || io->size_x < 1 || io->size_y < 1 || !(io->resolution > 0.0))
    return smpc_host_fail(SMPC_ERR_ARGUMENT, "optimize_batch: missing buffer");
  if (!io->od_indexes || !io->od_origin || io->n_od_grids < 1)
    return smpc_host_fail(SMPC_ERR_ARGUMENT, "ObstacleDistance is empty");  // reference: std::runtime_error (:676-680)
  if (io->od_width == 0 || io->od_height == 0) return smpc_host_fail(SMPC_ERR_ARGUMENT, "ObstacleDistance grid has invalid size");
  if (!(io->od_resolution > 0.0f)) return smpc_host_fail(SMPC_ERR_ARGUMENT, "ObstacleDistance grid has invalid resolution");
  if (!io->n_out || !io->optimized) return smpc_host_fail(SMPC_ERR_ARGUMENT, "optimize_batch: n_out / optimized missing");
  if (w) {
    const int rc = smpc_check_weight_sets(w, B, "optimize_batch_weighted");
    if (rc != SMPC_OK) return rc;
  }
  const smpc_params* prm = smpc_handle_params(h);
  if (prm->omni_solve)  // the reference's Optimizer::optimize is unicycle-only (update_state.hpp:46-61)
    return smpc_host_fail(SMPC_ERR_UNSUPPORTED, "the level-2 entries mirror Optimizer::optimize, which has no omnidirectional solve");
  std::lock_guard<std::mutex> lk(fs->mu);
  FLEET_CUDA(cudaSetDevice(smpc_handle_device(h)));
  cudaStream_t st = smpc_handle_stream(h);

  // ---- per-robot sizes on the host (O(B) integer work): the max_time cut of format_to_optimize (:492-497)
  const float timestep = io->time_step > 0.0f ? io->time_step : prm->time_step, maxtime = prm->max_time;
  const int maxsize = (int)std::round(maxtime / timestep);
  std::vector<int32_t>& n_each = fs->host_n_each;
  std::vector<int32_t>& s_each = fs->host_s_each;
  n_each.assign(B, 0);
  s_each.assign(B, 1);
  int n_max = 0;
  for (int b = 0; b < B; ++b) {
    int n = io->n_poses[b];
    if (n > stride) return smpc_host_fail(SMPC_ERR_ARGUMENT, "optimize_batch: n_poses[b] > max_poses");
    if (n < 2) continue;  // "Path has less than 2 points, cannot optimize" -> false for this robot (:158-162)
    if (n > maxsize) n = maxsize - 1;
    if (n < 2) return smpc_host_fail(SMPC_ERR_ARGUMENT, "max_time / time_step leaves fewer than 2 poses");
    n_each[b] = n;
    s_each[b] = n - 1;
    n_max = std::max(n_max, n);
  }
  const int S = stride - 1;  // array stride of the level-1 batch; every robot solves its own S_b = n_b - 1 <= S
  int nb = 0;
  int rc = smpc_problem_dims(prm, S, nullptr, nullptr, &nb, nullptr);
  if (rc != SMPC_OK) return rc;

  smpc_fleet_dev d{};
  d.B = B; d.stride = stride; d.A = A; d.nb = nb; d.time_step = timestep; d.max_time = maxtime;

  // ---- persistent per-robot memory (TrajectoryMemory per robot): re-created only when the fleet shape changes
  FLEET_CUDA(smpc_fleet_memory(fs, &d, st));

  // ---- costmaps and obstacle-distance grids stay on the device between ticks: re-sent only when maps_version changes
  const size_t map_bytes = (size_t)io->n_costmaps * io->size_x * io->size_y;
  const size_t od_cells = (size_t)io->od_width * io->od_height;
  const size_t od_bytes = (size_t)io->n_od_grids * od_cells * sizeof(uint32_t);
  const size_t maps_total = ((map_bytes + 255) & ~(size_t)255) + ((od_bytes + 255) & ~(size_t)255) +
                            (((size_t)io->n_costmaps * 16 + 255) & ~(size_t)255) + (((size_t)io->n_od_grids * 16 + 255) & ~(size_t)255);
  const bool resend = io->maps_version == 0 || io->maps_version != fs->maps_version || fs->maps_bytes != maps_total;
  FLEET_CUDA(fs->maps.reserve(maps_total));
  Carve cmaps(fs->maps.ptr);
  uint8_t* d_maps = cmaps.take<uint8_t>(map_bytes);
  uint32_t* d_od = cmaps.take<uint32_t>((size_t)io->n_od_grids * od_cells);
  double* d_map_org = cmaps.take<double>((size_t)io->n_costmaps * 2);
  double* d_od_org = cmaps.take<double>((size_t)io->n_od_grids * 2);
  // Small ticks (one robot: Optimizer::optimize itself) are dominated by per-copy driver overhead, not bytes: their
  // inputs, maps and results travel as ONE staged page-locked block each instead of ~14 + 4 + 10 separate copies.
  constexpr size_t kPackedTick = 256u << 10;
  if (resend && maps_total <= kPackedTick) {
    FLEET_CUDA(fs->pin_maps.reserve(maps_total));
    char* stage = static_cast<char*>(fs->pin_maps.ptr);
    const char* dev0 = static_cast<const char*>(fs->maps.ptr);
    std::memcpy(stage + (reinterpret_cast<const char*>(d_maps) - dev0), io->costmaps, map_bytes);
    std::memcpy(stage + (reinterpret_cast<const char*>(d_od) - dev0), io->od_indexes, od_bytes);
    std::memcpy(stage + (reinterpret_cast<const char*>(d_map_org) - dev0), io->costmap_origin, (size_t)io->n_costmaps * 16);
    std::memcpy(stage + (reinterpret_cast<const char*>(d_od_org) - dev0), io->od_origin, (size_t)io->n_od_grids * 16);
    FLEET_CUDA(cudaMemcpyAsync(fs->maps.ptr, stage, maps_total, cudaMemcpyHostToDevice, st));
    fs->maps_version = io->maps_version;
    fs->maps_bytes = maps_total;
  } else if (resend) {
    FLEET_CUDA(cudaMemcpyAsync(d_maps, io->costmaps, map_bytes, cudaMemcpyHostToDevice, st));
    FLEET_CUDA(cudaMemcpyAsync(d_od, io->od_indexes, od_bytes, cudaMemcpyHostToDevice, st));
    FLEET_CUDA(cudaMemcpyAsync(d_map_org, io->costmap_origin, (size_t)io->n_costmaps * 16, cudaMemcpyHostToDevice, st));
    FLEET_CUDA(cudaMemcpyAsync(d_od_org, io->od_origin, (size_t)io->n_od_grids * 16, cudaMemcpyHostToDevice, st));
    fs->maps_version = io->maps_version;
    fs->maps_bytes = maps_total;
  }
  d.n_costmaps = io->n_costmaps; d.size_x = io->size_x; d.size_y = io->size_y; d.resolution = io->resolution;
  d.maps = d_maps; d.map_org = d_map_org;
  d.n_od_grids = io->n_od_grids; d.od_width = io->od_width; d.od_height = io->od_height;
  d.od_resolution = io->od_resolution; d.od = d_od; d.od_org = d_od_org;

  // ---- per-tick scratch (one allocation that only ever grows): the ten input arrays, then the stage buffers and
  // outputs of the tick
  const size_t BS = (size_t)B * stride;
  auto carve_inputs = [&](Carve& c) {
    d.poses = c.take<double>(BS * 3);
    d.cmds = c.take<double>(BS * 2);
    d.people = c.take<double>((size_t)B * A * 5);
    d.n_people = c.take<int32_t>(B);
    d.speed = c.take<double>((size_t)B * 2);
    d.n_in = c.take<int32_t>(B);
    d.n_each = c.take<int32_t>(B);
    d.s_each = c.take<int32_t>(B);
    d.map_index = c.take<int32_t>(B);
    d.od_index = c.take<int32_t>(B);
    d.weights = c.take<double>(w ? (size_t)w->n_sets * 9 : 0);  // unweighted: no bytes, the layout is unchanged
    d.weight_set = c.take<int32_t>(w ? B : 0);
    smpc_fleet_carve_stages(c, &d);
  };
  size_t need = 0;
  {
    Carve probe(nullptr);
    carve_inputs(probe);
    need = probe.off;
  }
  FLEET_CUDA(fs->scratch.reserve(need));
  Carve cs(fs->scratch.ptr);
  carve_inputs(cs);
  double* d_poses = d.poses;
  double* d_cmds = d.cmds;
  double* d_people = const_cast<double*>(d.people);
  int32_t* d_map_index = const_cast<int32_t*>(d.map_index);
  int32_t* d_od_index = const_cast<int32_t*>(d.od_index);
  // the scratch starts with the ten input arrays (d_poses .. d_od_index) and ends with the result scalars
  // (usable .. status): each group is one contiguous span
  const char* scratch0 = static_cast<const char*>(fs->scratch.ptr);
  const size_t in_span = reinterpret_cast<const char*>(d.init) - scratch0;
  const size_t tail_off = reinterpret_cast<const char*>(d.usable) - scratch0, tail_span = need - tail_off;
  const size_t io_span = reinterpret_cast<const char*>(d_people) - scratch0;  // d_poses + d_cmds: in/out
  const bool packed = in_span <= kPackedTick && tail_span + io_span <= kPackedTick;

  // ---- inputs up
  struct Src { const void* dev; const void* host; size_t bytes; };
  const Src srcs[] = {
      {d_poses, io->poses, BS * 3 * 8},          {d_cmds, io->cmds, BS * 2 * 8},
      {d_people, io->people, (size_t)B * A * 5 * 8}, {d.n_people, io->n_people, (size_t)B * 4},
      {d.speed, io->speed, (size_t)B * 16},      {d.n_in, io->n_poses, (size_t)B * 4},
      {d.n_each, n_each.data(), (size_t)B * 4},  {d.s_each, s_each.data(), (size_t)B * 4},
      {d_map_index, io->costmap_index, (size_t)B * 4}, {d_od_index, io->od_index, (size_t)B * 4},
      {d.weights, w ? w->weights : nullptr, w ? (size_t)w->n_sets * 72 : 0},
      {d.weight_set, w ? w->set_index : nullptr, (size_t)B * 4},
  };
  if (packed) {
    FLEET_CUDA(fs->pin_in.reserve(in_span));
    char* stage = static_cast<char*>(fs->pin_in.ptr);
    for (const Src& c : srcs)
      if (c.host) std::memcpy(stage + (static_cast<const char*>(c.dev) - scratch0), c.host, c.bytes);
    FLEET_CUDA(cudaMemcpyAsync(fs->scratch.ptr, stage, in_span, cudaMemcpyHostToDevice, st));
  } else {
    for (const Src& c : srcs)
      if (c.host) FLEET_CUDA(cudaMemcpyAsync(const_cast<void*>(c.dev), c.host, c.bytes, cudaMemcpyHostToDevice, st));
  }
  if (!io->costmap_index) d.map_index = nullptr;
  if (!io->od_index) d.od_index = nullptr;
  if (!w) {
    d.weights = nullptr;
    d.weight_set = nullptr;
  }

  rc = smpc_fleet_tick_enqueue(h, d, st);
  if (rc != SMPC_OK) return rc;

  // ---- results down
  struct Dst { void* host; const void* dev; size_t bytes; };
  const Dst dsts[] = {
      {io->poses, d_poses, BS * 3 * 8},           {io->cmds, d_cmds, BS * 2 * 8},
      {io->n_out, d.n_out, (size_t)B * 4},        {io->optimized, d.optimized, (size_t)B},
      {io->termination, d.term, (size_t)B * 4},   {io->iterations, d.iters, (size_t)B * 4},
      {io->cost_initial, d.cost0, (size_t)B * 8}, {io->cost_final, d.cost1, (size_t)B * 8},
      {io->project_status, d.status, (size_t)B * 4},
  };
  if (io->people_proj)
    FLEET_CUDA(cudaMemcpyAsync(io->people_proj, d.agents, (size_t)B * A * 6 * stride * 8, cudaMemcpyDeviceToHost, st));
  if (packed) {  // [d_poses, d_cmds] and [d_usable .. d_status] into one staging block, then scattered on the host
    FLEET_CUDA(fs->pin_out.reserve(io_span + tail_span));
    char* stage = static_cast<char*>(fs->pin_out.ptr);
    FLEET_CUDA(cudaMemcpyAsync(stage, fs->scratch.ptr, io_span, cudaMemcpyDeviceToHost, st));
    FLEET_CUDA(cudaMemcpyAsync(stage + io_span, scratch0 + tail_off, tail_span, cudaMemcpyDeviceToHost, st));
    FLEET_CUDA(cudaStreamSynchronize(st));
    for (const Dst& c : dsts) {
      if (!c.host) continue;
      const size_t off = static_cast<const char*>(c.dev) - scratch0;
      std::memcpy(c.host, stage + (off < io_span ? off : io_span + (off - tail_off)), c.bytes);
    }
    return SMPC_OK;
  }
  for (const Dst& c : dsts)
    if (c.host) FLEET_CUDA(cudaMemcpyAsync(c.host, c.dev, c.bytes, cudaMemcpyDeviceToHost, st));
  FLEET_CUDA(cudaStreamSynchronize(st));
  return SMPC_OK;
}

extern "C" {

int smpc_optimize_batch(smpc_handle* h, smpc_fleet_io* io) {
  if (!h) return smpc_host_fail(SMPC_ERR_ARGUMENT, "handle is NULL");
  return smpc_optimize_batch_on(h, smpc_handle_fleet(h), io);
}

int smpc_optimize_batch_weighted(smpc_handle* h, smpc_fleet_io* io, const smpc_weight_sets* w) {
  if (!h) return smpc_host_fail(SMPC_ERR_ARGUMENT, "handle is NULL");
  const int rc = smpc_check_weight_sets(w, 0, "optimize_batch_weighted");  // the indices: once B is known
  if (rc != SMPC_OK) return rc;
  return smpc_optimize_batch_on(h, smpc_handle_fleet(h), io, w);
}

}  // extern "C"
