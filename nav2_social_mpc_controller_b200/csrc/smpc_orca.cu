// smpc_orca.cu — the ORCA crowd of the closed-loop episodes (smpc_run_orca_episodes): the people of every scene choose
// velocities by optimal reciprocal collision avoidance (van den Berg et al., "Reciprocal n-body collision avoidance";
// RVO2's Agent::computeNewVelocity, linearProgram1/2/3 and Agent::update), a model the controller's people projection
// does not contain. Laid out like smpc_crowd_step_kernel: one warp per scene, lanes over people (two slots per lane),
// the agent states of the current substep in shared memory (people in slots 0 .. n-1, the R robots in n .. n+R-1),
// next-substep staging, and the per-robot disturbance reduced across the warp. A person's ORCA lines (at most 16
// agents + 1 obstacle) and linearProgram3's projected lines live in per-thread local arrays.
// Compiled with -fmad=false (Makefile): no contraction, so tests/orca_ref.py reproduces every line bit for bit.
#include <cuda_runtime.h>

#include <cmath>
#include <string>

#include "../../include/smpc.h"
#include "smpc_host_state.h"
#include "smpc_sfm.cuh"

namespace {

constexpr int kMaxAgents = 64;  // people + robots
constexpr int kMaxRobots = 8;   // robots per scene
constexpr int kMaxNeighbors = 16;
constexpr int kMaxLines = kMaxNeighbors + 1;  // + the obstacle line
constexpr int kWarps = 4;
constexpr double kEps = 1e-5;  // RVO_EPSILON

struct OrcaSmem {  // structure of arrays, one slot per agent of the current substep
  double px[kMaxAgents], py[kMaxAgents], vx[kMaxAgents], vy[kMaxAgents];
  double nx[kMaxAgents], ny[kMaxAgents], nvx[kMaxAgents], nvy[kMaxAgents];  // next-substep staging
  double dist[kMaxRobots][32];  // per robot and lane: robot_responsibility |u| dt_s over this lane's people
};

struct Line {  // the half-plane left of `point + t dir`
  double px, py, dx, dy;
};

__device__ __forceinline__ double det2(double ax, double ay, double bx, double by) { return ax * by - ay * bx; }

// linearProgram1: the optimum on line `no` within the circle of `radius` and the lines before it; false if none
__device__ bool lp1(const Line* L, int no, double radius, double ox, double oy, bool dir_opt, double* rx, double* ry) {
  const Line& l = L[no];
  const double dot = l.px * l.dx + l.py * l.dy;
  const double disc = dot * dot + radius * radius - (l.px * l.px + l.py * l.py);
  if (disc < 0.0) return false;
  const double sq = sqrt(disc);
  double tl = -dot - sq, tr = -dot + sq;
  for (int i = 0; i < no; ++i) {
    const double den = det2(l.dx, l.dy, L[i].dx, L[i].dy);
    const double num = det2(L[i].dx, L[i].dy, l.px - L[i].px, l.py - L[i].py);
    if (fabs(den) <= kEps) {  // (almost) parallel
      if (num < 0.0) return false;
      continue;
    }
    const double t = num / den;
    if (den >= 0.0) tr = fmin(tr, t);
    else tl = fmax(tl, t);
    if (tl > tr) return false;
  }
  double t;
  if (dir_opt) {
    t = (ox * l.dx + oy * l.dy > 0.0) ? tr : tl;
  } else {
    t = l.dx * (ox - l.px) + l.dy * (oy - l.py);
    if (t < tl) t = tl;
    else if (t > tr) t = tr;
  }
  *rx = l.px + t * l.dx;
  *ry = l.py + t * l.dy;
  return true;
}

// linearProgram2: returns n on success, else the first line it could not satisfy (the result then satisfies the lines
// before it)
__device__ int lp2(const Line* L, int n, double radius, double ox, double oy, bool dir_opt, double* rx, double* ry) {
  if (dir_opt) {
    *rx = ox * radius;
    *ry = oy * radius;
  } else if (ox * ox + oy * oy > radius * radius) {
    const double len = sqrt(ox * ox + oy * oy);
    *rx = ox / len * radius;
    *ry = oy / len * radius;
  } else {
    *rx = ox;
    *ry = oy;
  }
  for (int i = 0; i < n; ++i) {
    if (det2(L[i].dx, L[i].dy, L[i].px - *rx, L[i].py - *ry) > 0.0) {
      const double sx = *rx, sy = *ry;
      if (!lp1(L, i, radius, ox, oy, dir_opt, rx, ry)) {
        *rx = sx;
        *ry = sy;
        return i;
      }
    }
  }
  return n;
}

// linearProgram3: from line `begin` on, minimise the largest violation of the soft lines (n_obst hard lines first)
__device__ void lp3(const Line* L, int n, int n_obst, int begin, double radius, double* rx, double* ry) {
  Line proj[kMaxLines];
  double distance = 0.0;
  for (int i = begin; i < n; ++i) {
    if (det2(L[i].dx, L[i].dy, L[i].px - *rx, L[i].py - *ry) > distance) {
      int np = 0;
      for (int j = 0; j < n_obst; ++j) proj[np++] = L[j];
      for (int j = n_obst; j < i; ++j) {
        Line pl;
        const double dt = det2(L[i].dx, L[i].dy, L[j].dx, L[j].dy);
        if (fabs(dt) <= kEps) {  // parallel
          if (L[i].dx * L[j].dx + L[i].dy * L[j].dy > 0.0) continue;  // same direction
          pl.px = 0.5 * (L[i].px + L[j].px);
          pl.py = 0.5 * (L[i].py + L[j].py);
        } else {
          const double s = det2(L[j].dx, L[j].dy, L[i].px - L[j].px, L[i].py - L[j].py) / dt;
          pl.px = L[i].px + s * L[i].dx;
          pl.py = L[i].py + s * L[i].dy;
        }
        const double ddx = L[j].dx - L[i].dx, ddy = L[j].dy - L[i].dy;
        const double len = sqrt(ddx * ddx + ddy * ddy);
        pl.dx = ddx / len;
        pl.dy = ddy / len;
        proj[np++] = pl;
      }
      const double sx = *rx, sy = *ry;
      if (lp2(proj, np, radius, -L[i].dy, L[i].dx, true, rx, ry) < np) {  // floating-point failure: keep the result
        *rx = sx;
        *ry = sy;
      }
      distance = det2(L[i].dx, L[i].dy, L[i].px - *rx, L[i].py - *ry);
    }
  }
}

// The ORCA line of one agent (or the obstacle point) at relative position (rpx, rpy) = other - me with relative velocity
// (rvx, rvy) = mine - other's and combined radius cr; my velocity (vx, vy), my share resp. False (no line) for a
// collision with |w| == 0. u: the smallest change of the relative velocity that leaves the velocity obstacle.
__device__ bool orca_line(double rpx, double rpy, double rvx, double rvy, double cr, double inv_t, double inv_dt,
                          double vx, double vy, double resp, Line* l, double* ux, double* uy) {
  const double dist_sq = rpx * rpx + rpy * rpy;
  const double cr_sq = cr * cr;
  if (dist_sq > cr_sq) {  // no collision
    const double wx = rvx - inv_t * rpx, wy = rvy - inv_t * rpy;
    const double wl_sq = wx * wx + wy * wy;
    const double dp1 = wx * rpx + wy * rpy;
    if (dp1 < 0.0 && dp1 * dp1 > cr_sq * wl_sq) {  // cut-off circle
      const double wl = sqrt(wl_sq);
      const double uwx = wx / wl, uwy = wy / wl;
      l->dx = uwy;
      l->dy = -uwx;
      const double s = cr * inv_t - wl;
      *ux = s * uwx;
      *uy = s * uwy;
    } else {  // legs
      const double leg = sqrt(dist_sq - cr_sq);
      if (det2(rpx, rpy, wx, wy) > 0.0) {  // left leg
        l->dx = (rpx * leg - rpy * cr) / dist_sq;
        l->dy = (rpx * cr + rpy * leg) / dist_sq;
      } else {  // right leg
        l->dx = -(rpx * leg + rpy * cr) / dist_sq;
        l->dy = -(-rpx * cr + rpy * leg) / dist_sq;
      }
      const double dp2 = rvx * l->dx + rvy * l->dy;
      *ux = dp2 * l->dx - rvx;
      *uy = dp2 * l->dy - rvy;
    }
  } else {  // collision: cut-off circle of one substep
    const double wx = rvx - inv_dt * rpx, wy = rvy - inv_dt * rpy;
    const double wl = sqrt(wx * wx + wy * wy);
    if (wl == 0.0) return false;
    const double uwx = wx / wl, uwy = wy / wl;
    l->dx = uwy;
    l->dy = -uwx;
    const double s = cr * inv_dt - wl;
    *ux = s * uwx;
    *uy = s * uwy;
  }
  l->px = vx + resp * *ux;
  l->py = vy + resp * *uy;
  return true;
}

// One controller tick k of the ORCA crowd of scene b: `substeps` synchronous updates of dt_s = dt_c / substeps, every
// line from the state at the start of its substep (include/smpc.h states the model). Robot r is at
// x_k + (s dt_s) v_k (cos th_k, sin th_k) at substep s with that velocity; a robot whose episode is done stands still.
// With robot_responsibility == 0 the robots are no agents. The people move while any robot of the scene runs.
__global__ void __launch_bounds__(kWarps * 32) smpc_orca_step_kernel(smpc_crowd_step_args a, smpc_orca_params o) {
  __shared__ OrcaSmem sm[kWarps];
  OrcaSmem& s = sm[threadIdx.x >> 5];
  const int lane = threadIdx.x & 31;
  const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;  // scene
  if (b >= a.B) return;  // warp-uniform
  const int R = a.R, r0 = b * R;
  bool running = false;
  for (int r = 0; r < R; ++r) running |= a.active[r0 + r] != 0;
  if (!running) return;  // warp-uniform
  const double kGoalRadius = 0.25;
  const int K = a.K, n = K > 0 ? a.n_people[b] : 0;
  const int n_robots = o.robot_responsibility > 0.0 ? R : 0;  // robots as agents
  const double dts = a.dt_c / (double)a.substeps;
  const double inv_t = 1.0 / o.time_horizon, inv_to = 1.0 / o.time_horizon_obst, inv_dt = 1.0 / dts;
  const double range0 = o.neighbor_dist * o.neighbor_dist;
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
      const double vmax = vdes[q];
      double prefx = 0.0, prefy = 0.0;  // preferred velocity
      if (goal[q]) {
        const double dx = gx[q] - px, dy = gy[q] - py;
        const double z = dx * dx + dy * dy;
        if (z > 0.0) {
          const double sq = sqrt(z);
          prefx = vmax * (dx / sq);
          prefy = vmax * (dy / sq);
        }
      }
      // neighbours: people in slot order, then robots; RVO2's insertion into a list sorted by distSq
      double nd[kMaxNeighbors];
      int ni[kMaxNeighbors];
      int nn = 0;
      double range = range0;
      for (int j = 0; j < n + n_robots; ++j) {
        if (j == slot) continue;
        const double dx = s.px[j] - px, dy = s.py[j] - py;
        const double d = dx * dx + dy * dy;
        if (!(d < range)) continue;
        if (nn < o.max_neighbors) ++nn;
        int i = nn - 1;
        while (i != 0 && d < nd[i - 1]) {
          nd[i] = nd[i - 1];
          ni[i] = ni[i - 1];
          --i;
        }
        nd[i] = d;
        ni[i] = j;
        if (nn == o.max_neighbors) range = nd[nn - 1];
      }
      Line L[kMaxLines];
      int nl = 0;
      double ux, uy;
      // the nearest obstacle cell as a static point (hard line); none outside the grid
      double mx, my;
      if (px >= ox && py >= oy &&
          smpc::nearest_obstacle(a.od_width, a.od_height, a.od_resolution, idx, ox, oy, px, py, &mx, &my)) {
        const double rpx = -mx, rpy = -my;  // cell - p
        const double reach = o.time_horizon_obst * vmax + o.person_radius;
        if (rpx * rpx + rpy * rpy < reach * reach &&
            orca_line(rpx, rpy, vx, vy, o.person_radius, inv_to, inv_dt, vx, vy, 1.0, &L[nl], &ux, &uy))
          ++nl;
      }
      const int n_obst = nl;
      for (int i = 0; i < nn; ++i) {
        const int j = ni[i];
        const bool robot = j >= n;
        const double cr = o.person_radius + (robot ? o.robot_radius : o.person_radius);
        const double resp = robot ? o.robot_responsibility : 0.5;
        if (!orca_line(s.px[j] - px, s.py[j] - py, vx - s.vx[j], vy - s.vy[j], cr, inv_t, inv_dt, vx, vy, resp, &L[nl],
                       &ux, &uy))
          continue;
        if (robot && det2(L[nl].dx, L[nl].dy, L[nl].px - vx, L[nl].py - vy) > 0.0)
          s.dist[j - n][lane] += resp * sqrt(ux * ux + uy * uy) * dts;
        ++nl;
      }
      double nvx, nvy;
      const int fail = lp2(L, nl, vmax, prefx, prefy, false, &nvx, &nvy);
      if (fail < nl) lp3(L, nl, n_obst, fail, vmax, &nvx, &nvy);
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

int smpc_orca_step_enqueue(smpc_handle* h, const smpc_crowd_step_args& a, const smpc_orca_params& o, cudaStream_t st) {
  if (a.B == 0) return SMPC_OK;
  smpc_orca_step_kernel<<<(unsigned)((a.B + kWarps - 1) / kWarps), kWarps * 32, 0, st>>>(a, o);
  SMPC_FLEET_CUDA(cudaGetLastError());
  smpc_handle_count_launch(h);
  return SMPC_OK;
}
