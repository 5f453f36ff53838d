// smpc_crowd.cu — the reactive crowd of the closed-loop episodes (smpc_run_crowd_episodes, smpc_run_shared_episodes):
// the people of every scene walk to their own goals under the lightsfm social force model (reference
// include/nav2_social_mpc_controller/sfm.hpp, the same model and constants the controller's people projection uses,
// smpc_sfm.cuh), avoid the walls of the scene's obstacle-distance grid and each other, and give way to the scene's
// robots, which exert force as extra agents but are moved by the world step, not by the model. One warp per scene,
// lanes over people (two slots per lane), the agent states of the current substep in shared memory, laid out like
// smpc_project_kernel: the people in slots 0 .. n-1, the R robots in slots n .. n+R-1.
#include <cuda_runtime.h>

#include <cmath>
#include <string>

#include "../../include/smpc.h"
#include "smpc_host_state.h"
#include "smpc_sfm.cuh"

namespace {

constexpr int kMaxAgents = 64;  // people + robots
constexpr int kMaxRobots = 8;   // robots per scene
constexpr int kWarps = 4;

struct CrowdSmem {  // structure of arrays, one slot per agent of the current substep
  double px[kMaxAgents], py[kMaxAgents], vx[kMaxAgents], vy[kMaxAgents];
  double nx[kMaxAgents], ny[kMaxAgents], nvx[kMaxAgents], nvy[kMaxAgents];  // next-substep staging
  double dist[kMaxRobots][32];  // per robot and lane: sum of |F(robot -> person)| dt_s over this lane's people
};

// One controller tick k of the crowd of scene b: `substeps` synchronous lightsfm updates of dt_s = dt_c / substeps,
// every force from the state at the start of its substep. Robot r is at x_k + (s dt_s) v_k (cos th_k, sin th_k) at
// substep s for its own pose and command of tick k; a robot whose episode is done stands still (v = 0).
// Forces on person i (sfm.hpp:188-281): desired force to its goal at its own desired speed (braking -v / 0.5 once the
// goal is cleared), the obstacle force of the nearest obstacle cell of the grid at the person's current position
// (radius 0.5; none outside the grid), and the pair force of every other person and of the robot. Unlike the
// reference's projection (SURVEY Q10) the obstacle enters as a position, so people are pushed away from the walls.
// The pair forces come from the people first, then from robots 0 .. R-1 in order (R = 1: the arithmetic of one robot).
// updatePosition (sfm.hpp:512-545): velocity capped at the desired speed, the goal cleared for good the first time the
// updated position is within 0.25 m of it; vz carries lightsfm's angular velocity. Robot r's pair term,
// |F(robot -> i)| dt_s, accumulates into disturbance[b * R + r] while that robot runs. The people move while any robot
// of the scene runs.
__global__ void __launch_bounds__(kWarps * 32) smpc_crowd_step_kernel(smpc_crowd_step_args a) {
  __shared__ CrowdSmem sm[kWarps];
  CrowdSmem& s = sm[threadIdx.x >> 5];
  const int lane = threadIdx.x & 31;
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;  // scene
  if (b >= a.B) return;  // warp-uniform
  const int R = a.R, r0 = b * R;
  bool running = false;
  for (int r = 0; r < R; ++r) running |= a.active[r0 + r] != 0;
  if (!running) return;  // warp-uniform
  const double kDesired = 2.0, kObstacle = 20.0, kSigma = 0.2, kRelax = 0.5, kRadius = 0.5, kGoalRadius = 0.25;
  const int K = a.K, n = K > 0 ? a.n_people[b] : 0;
  const double dts = a.dt_c / (double)a.substeps;
  double* P = a.people + (size_t)b * K * 5;
  const int gi = a.od_index ? a.od_index[r0] : (r0 % a.n_od_grids);
  const uint32_t* idx = a.od + (size_t)gi * a.od_width * a.od_height;
  const double ox = a.od_org[2 * gi], oy = a.od_org[2 * gi + 1];

  // lane r < R: robot r's pose and command of tick k (the world step applies the same command)
  double rx = 0.0, ry = 0.0, rvx = 0.0, rvy = 0.0;
  if (lane < R) {
    const int rb = r0 + lane;
    const double v = a.active[rb] ? a.cmds[(size_t)rb * a.stride * 2] : 0.0;
    rx = a.pose[3 * rb];
    ry = a.pose[3 * rb + 1];
    double rs, rc;
    sincos(a.pose[3 * rb + 2], &rs, &rc);
    rvx = __dmul_rn(v, rc);
    rvy = __dmul_rn(v, rs);
  }
  for (int r = 0; r < R; ++r) s.dist[r][lane] = 0.0;

  double yaw[2], vz[2], gx[2], gy[2], vdes[2];
  bool goal[2], mine[2];
  for (int q = 0; q < 2; ++q) {
    const int slot = lane + 32 * q;
    mine[q] = slot < n;
    yaw[q] = vz[q] = gx[q] = gy[q] = 0.0;
    vdes[q] = 1.0;
    goal[q] = false;
    if (!mine[q]) continue;
    const double* p = P + (size_t)slot * 5;
    s.px[slot] = p[0];
    s.py[slot] = p[1];
    s.vx[slot] = p[2];
    s.vy[slot] = p[3];
    vz[q] = p[4];
    yaw[q] = atan2(p[3], p[2]);
    gx[q] = a.goals[((size_t)b * K + slot) * 2];
    gy[q] = a.goals[((size_t)b * K + slot) * 2 + 1];
    vdes[q] = a.vdes[(size_t)b * K + slot];
    goal[q] = a.has_goal[(size_t)b * K + slot] != 0;
  }
  if (a.people_log && a.k == 0)  // row 0 = the input state
    for (int e = lane; e < K * 5; e += 32) a.people_log[(size_t)b * (a.T + 1) * K * 5 + e] = P[e];

  for (int sub = 0; sub < a.substeps; ++sub) {
    if (lane < R) {  // robot r as agent n + r
      const double ts = __dmul_rn((double)sub, dts);
      s.px[n + lane] = __dadd_rn(rx, __dmul_rn(ts, rvx));
      s.py[n + lane] = __dadd_rn(ry, __dmul_rn(ts, rvy));
      s.vx[n + lane] = rvx;
      s.vy[n + lane] = rvy;
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
        if (goal[q] && dn > kGoalRadius) {
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
      // social force from every other person, then from the robots (sfm.hpp:239-281)
      double2 f = make_double2(0.0, 0.0);
      for (int k = 0; k < n; ++k) {
        if (k == slot) continue;
        f = smpc::sfm_pair(s.px[k] - px, s.py[k] - py, vx - s.vx[k], vy - s.vy[k], f.x, f.y);
      }
      for (int r = 0; r < R; ++r) {
        const int j = n + r;
        const double2 fr = smpc::sfm_pair(s.px[j] - px, s.py[j] - py, vx - s.vx[j], vy - s.vy[j], 0.0, 0.0);
        f.x += fr.x;
        f.y += fr.y;
        s.dist[r][lane] += sqrt(fr.x * fr.x + fr.y * fr.y) * dts;
      }
      fx += f.x;
      fy += f.y;
      // obstacle force (sfm.hpp:206-221) of the nearest obstacle cell at the current position; none outside the grid
      // (nearest_obstacle alone would read a point left of or below the origin as column / row 0)
      double mx, my;
      if (px >= ox && py >= oy &&
          smpc::nearest_obstacle(a.od_width, a.od_height, a.od_resolution, idx, ox, oy, px, py, &mx, &my)) {
        const double mn = sqrt(mx * mx + my * my);
        const double distance = mn - kRadius;
        const double z = mx * mx + my * my;
        double ex = mx, ey = my;
        if (z > 0.0) {
          const double sq = sqrt(z);
          ex = mx / sq;
          ey = my / sq;
        }
        const double k = kObstacle * exp(-distance / kSigma);
        fx += k * ex;
        fy += k * ey;
      }
      // updatePosition (sfm.hpp:512-545)
      double nvx = vx + fx * dts, nvy = vy + fy * dts;
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
      yaw[q] = smpc::wrap_pi(atan2(nvy, nvx));
      vz[q] = smpc::wrap_pi(yaw[q] - y0) / dts;
      const double npx = px + nvx * dts, npy = py + nvy * dts;
      if (goal[q]) {
        const double dx = gx[q] - npx, dy = gy[q] - npy;
        if (sqrt(dx * dx + dy * dy) <= kGoalRadius) goal[q] = false;
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
    }
    __syncwarp();
  }

  for (int r = 0; r < R; ++r) {
    double dist = s.dist[r][lane];
    for (int off = 16; off > 0; off >>= 1) dist += __shfl_xor_sync(0xffffffffu, dist, off);
    if (lane == 0 && a.active[r0 + r]) a.disturbance[r0 + r] += dist;
  }
  double* log = a.people_log ? a.people_log + ((size_t)b * (a.T + 1) + a.k + 1) * K * 5 : nullptr;
  for (int q = 0; q < 2; ++q) {
    const int slot = lane + 32 * q;
    if (slot >= K) continue;
    double st[5];
    if (mine[q]) {
      st[0] = s.px[slot]; st[1] = s.py[slot]; st[2] = s.vx[slot]; st[3] = s.vy[slot]; st[4] = vz[q];
      for (int c = 0; c < 5; ++c) P[(size_t)slot * 5 + c] = st[c];
      a.has_goal[(size_t)b * K + slot] = goal[q];
    } else {  // padding beyond the scene's people: unchanged
      for (int c = 0; c < 5; ++c) st[c] = P[(size_t)slot * 5 + c];
    }
    if (log)
      for (int c = 0; c < 5; ++c) log[(size_t)slot * 5 + c] = st[c];
  }
}

}  // namespace

int smpc_crowd_step_enqueue(smpc_handle* h, const smpc_crowd_step_args& a, cudaStream_t st) {
  if (a.B == 0) return SMPC_OK;
  smpc_crowd_step_kernel<<<(unsigned)((a.B + kWarps - 1) / kWarps), kWarps * 32, 0, st>>>(a);
  SMPC_FLEET_CUDA(cudaGetLastError());
  smpc_handle_count_launch(h);
  return SMPC_OK;
}
