// smpc_device.cuh — device-side social-MPC solver for sm_100a (B200), FP64 CUDA cores.
//
// A GROUP of G lanes (4, 8, 16 or 32) solves one MPC problem: lane gl owns horizon steps gl, gl+G, ...
//   * rollout: heading in closed form from the block-held angular rates, positions by warp inclusive
//     scans; forward sensitivities dX/du, dY/du by the same scans (reference update_state.hpp:37-63
//     re-rolls-out 0..i inside every functor, O(S^2); here it is one O(S) pass per evaluation).
//   * residuals + ANALYTIC gradients wrt the lane's pose (X, Y, Theta, v_block) for the eight active
//     critics (reference include/nav2_social_mpc_controller/critics/*.hpp), accumulated per lane as a
//     4x4 Gauss-Newton block M = sum c c^T and q = sum c r, then g_lane = D^T q and — only when the trial point can
//     become the next iterate — H_lane = D^T M D with the 4xP sensitivity matrix D; a shared-memory column sum
//     gives cost, J^T r, J^T J of the group.
//   * the bounded trust-region Levenberg-Marquardt loop of ceres::Solve (reference src/optimizer.cpp:381
//     with the options of :117-131) is run by the group's FIRST lane on the group's shared-memory state (the other
//     lanes wait at a __syncwarp): Jacobi scaling, LM diagonal, PxP Cholesky, projected Armijo line search with
//     cubic / quintic interpolation, tolerance tests, radius update.
// No CPU fallback exists; this header is the product path.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cfloat>
#include <cmath>
#include <type_traits>

#include "smpc_math.cuh"

namespace smpc {

constexpr unsigned kFullMask = 0xffffffffu;
constexpr int kMaxSteps = 64;  // S <= 64 steps (the reference parameter sets give 13, 28, 38)

struct DevParams {
  double w_distance, w_social, w_velocity, w_angle, w_agent_angle, w_prox, w_vf, w_obstacle, w_goal;
  double param_tol, fn_tol, gradient_tol;
  int max_iterations, ceres_compat, max_evaluations;
  int ch, bl, nb, n_bounded;  // of the batch's longest horizon (nb = template NB of the kernel)
  int dof;  // parameters per block: 2 = (v, w) reference unicycle, 3 = (vx, vy, w) omnidirectional extension
  int control_horizon, block_length;  // yaml values: per-problem dims are derived from them (src/optimizer.cpp:248-249)
};

struct DevBatch {
  int B, S, A, M, size_x, size_y;
  double resolution, dt;
  const double* pose0;
  const double* u0;
  const double* path_xy;
  const double* goal_yaw;
  const double* agents;
  const double* agents_packed;  // [B][A][S+1][4] = x, y, vx, vy (built once per batch by smpc_pack_agents_kernel)
  const uint8_t* agents_valid;  // [B][A][S+1]   = (t != -1)
  const uint8_t* has_people;
  const uint8_t* costmaps;
  const double* costmap_origin;
  const int32_t* costmap_index;
  const int32_t* n_steps_each;  // [B] per-problem horizon S_b <= S, NULL = S for all
  // Host-buffer pipeline only (else NULL): arrival[0] = number of leading problems whose costmap has landed in device
  // memory (written by the copy stream after each map chunk), arrival[1] = set by the kernel if it gave up waiting.
  unsigned* arrival;
  // Time slicing of the solve queue (NULL = off; smpc_host.cu enables it for batches of a few waves, where the tail of
  // late-started long solves dominates): a group that has spent `park_quantum` evaluations on a problem while fresh
  // problems are still waiting parks it — saves its shared-memory state to park_state[b], publishes b in park_ring —
  // and starts a fresh one; parked problems are resumed, to completion, once the main queue has drained.
  double* park_state;  // [B][Layout::total(S)]
  int* park_ring;      // [B] problem ids in parking order, -1 = not published yet
  int* park_counters;  // [0] = published slots reserved (tail), [1] = slots claimed by resumers (head)
  int park_quantum;
  // 1 = the warps of a CTA meet at a CTA barrier before every evaluation (they then walk the large evaluation code
  // together and share its instruction-cache lines); 0 = warps run free and leave on their own
  int cta_sync;
  // scenario sharing: problem b reads row scenario[b] of the per-scene arrays (NULL: row b); n_rows = rows of those arrays
  const int32_t* scenario;
  int n_rows;
  // per-problem critic weights (the weighted solve kernel only; NULL = DevParams' w_*): problem b uses row
  // weight_set[b] of weights [P][9], in DevParams order w_distance .. w_goal
  const double* weights;
  const int32_t* weight_set;
};

struct DevResult {
  double* u;
  double* cmds;
  double* path;
  double* cost_initial;
  double* cost_final;
  int32_t* iterations;
  int32_t* termination;
  uint8_t* usable;
  int32_t* n_evals;
  double* trace;  // [B][trace_rows][8], NULL = off (include/smpc.h)
  int trace_rows;
};

struct DevEvalOut {
  double* cost;
  double* cost_plain;
  double* grad;
  double* hess;
  uint8_t* ok;
};

// Group-uniform view of one problem (lives in the group's shared memory).
struct Prob {
  double x0, y0, yaw0, goal_yaw, fin_x, fin_y, org_x, org_y;
  const double* px;
  const double* py;
  const double* agents;  // [A][6][S+1]
  const double* packed;  // [A][S+1][4]
  const uint8_t* valid;  // [A][S+1]
  const uint8_t* map;
  // per-problem sizes (src/optimizer.cpp:248-249, :373): S_b steps, ch = min(control_horizon, S_b),
  // bl = min(block_length, ch), nb = ceil(ch / bl) blocks in use (<= NB of the kernel), nbd = ch / bl bounded blocks
  int S, ch, bl, nb, nbd;
  bool has_people;
};

enum EvalFlags : unsigned { kResidualBad = 1u, kJacobianBad = 2u, kNoHessian = 4u };

// std::max / std::min as Ceres and the reference use them: one compare + select, and a NaN in the FIRST argument
// propagates (CUDA's fmax / fmin return the other operand and cost ~8 instructions each for that).
// One Kogge-Stone step v += (lane takes part ? t : 0) as ONE DFMA with the 0 / 1 mask m: fma(t, 1, v) is v + t exactly
// and fma(t, 0, v) is v (the compiler's form of `if (on) v += t` is DADD + two FSEL, and ptxas turns a predicated
// add back into that; the scans are 14 x log2(G) such steps per evaluation). A non-finite t poisons the masked lanes
// too — their own value is non-finite already (out-of-range shuffles return the lane's own value).
__device__ __forceinline__ void add_masked(double& v, double t, double m) { v = fma(t, m, v); }

__device__ __forceinline__ double std_max(double a, double b) { return (a < b) ? b : a; }
__device__ __forceinline__ double std_min(double a, double b) { return (b < a) ? b : a; }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(kFullMask, v, d);
  return v;
}

// ---------------------------------------------------------------------------------------------------
// Social force of `me` caused by `other` (reference social_work_cost_function.hpp:165-223, constants
// social_work_cost_function.cpp:38-43) as a function of d = me.xy - other.xy and w = me.vel - other.vel,
// with its 2x4 Jacobian wrt (d.x, d.y, w.x, w.y).
// ---------------------------------------------------------------------------------------------------
struct PairOut {
  double fx, fy;
  double dfx[4], dfy[4];
  bool degenerate;  // theta came from the reference's two-atan2 branch (the pair is then not odd in (d, w))
};

__device__ __forceinline__ double wrap_to_pi(double a) {
  // reference social_work_cost_function.hpp:39-46
  while (a > M_PI) a -= 2.0 * M_PI;
  while (a <= -M_PI) a += 2.0 * M_PI;
  return a;
}

// gamma, 1/gamma, force factor, coincident-position |d| and |d|^2, degenerate |sin theta|
static __constant__ double kPairTab[6] = {0.35, 1.0 / 0.35, 2.1, 1e-6, 1e-12, 1e-9};

// kReferenceAngle = false: theta always from the one-atan2 form (the caller re-evaluates degenerate pairs through
// social_pair_reference, an out-of-line call, so the two general atan2 expansions stay out of the hot loop body).
template <bool kReferenceAngle>
__device__ __forceinline__ void social_pair(double dx, double dy, double wx, double wy, PairOut& o) {
  const double kLambda = 2.0, kNPrime = 3.0, kN = 2.0;
  const double kGamma = kPairTab[0], kInvGamma = kPairTab[1], kFactor = kPairTab[2];
  double d2 = dx * dx + dy * dy;
  const bool tiny = d2 < kPairTab[4];  // |d| < 1e-6
  if (kReferenceAngle && tiny) {  // coincident: fixed direction (1e-6, 0), a constant for the derivative
    dx = kPairTab[3];           // (the hot instantiation only FLAGS such a pair as degenerate: its caller re-evaluates
    dy = 0.0;                   //  it through social_pair_reference)
    d2 = dx * dx;
  }
  const double inv_rho = rsqrt_pos(d2);
  const double rho = d2 * inv_rho;
  const double ex = dx * inv_rho, ey = dy * inv_rho;  // Eigen normalized() (|d|^2 > 0 always holds here)
  const double Ix = kLambda * wx + ex, Iy = kLambda * wy + ey;
  const double L2 = Ix * Ix + Iy * Iy;
  const double inv_L = rsqrt_pos(L2);
  const double L = L2 * inv_L;
  const double ix = Ix * inv_L, iy = Iy * inv_L;
  // theta = wrapToPi(atan2(e) - atan2(i)), the signed angle from i to e. Generic geometry: one atan2 of
  // (cross, dot) (same value to ~1 ulp, and sgn(theta) = sgn(cross) robustly). Near-degenerate geometry
  // (|sin theta| < 1e-9: exactly (anti)parallel set-ups such as a person dead ahead): the model is discontinuous
  // at theta = 0 and +-pi and the reference's own rounding decides the branch, so its formulation is used verbatim.
  const double cross = ey * ix - ex * iy, dot = ex * ix + ey * iy;
  double theta;
  o.degenerate = tiny || !(fabs(cross) > kPairTab[5]);  // the coincident-position fix-up is not odd in d either
  if (!kReferenceAngle || !o.degenerate) {
    theta = atan2_unit(cross, dot);
  } else {
    theta = wrap_to_pi(atan2(ey, ex) - atan2(iy, ix));
  }
  const double Bq = kGamma * L;
  const double inv_B = inv_L * kInvGamma;
  const double Bth = Bq * theta;
  const double t1 = kNPrime * Bth, t2 = kN * Bth;
  const double base = -rho * inv_B;
  const double E1 = exp_nonpos(base - t1 * t1);
  const double E2 = exp_nonpos(base - t2 * t2);
  // fa = -sgn(theta) exp(.), sgn(0) = -1 as in the reference; the hot instantiation never sees theta == 0 (that is
  // cross == 0: degenerate), so the sign is a bit operation there
  const double fv = -E1, fa = kReferenceAngle ? ((theta > 0.0) ? -E2 : E2) : copysign(E2, -theta);
  const double Fix = kFactor * ix, Fiy = kFactor * iy;
  const double a = Fix * fv, b = Fiy * fa, c = Fiy * fv, d = Fix * fa;
  o.fx = a - b;
  o.fy = c + d;

  // Gradients wrt (dx, dy, wx, wy) by the chain rule through the four scalars the force depends on: rho = |d|, phi_e
  // (direction of d), L = |I|, phi_i (direction of I), with theta = phi_e - phi_i, B = gamma L and
  //   u_n = -rho / B - (n B theta)^2,   fv = -exp(u_3),  fa = -sgn(theta) exp(u_2),   f = F Rot(phi_i) (fv, fa):
  //   d u_n = -d rho / B + (rho / (B L)) dL + k_n (gamma theta dL + B (d phi_e - d phi_i)),   k_n = -2 n^2 B theta.
  // First the partials of (fx, fy) wrt (rho, L, phi_e, phi_i) — X*, Y* below — then the 2x4 Jacobian from
  //   d rho = e,  d phi_e = e_perp / rho,  dL = (i . e_perp) d phi_e + lambda i dw,
  //   d phi_i = ((i . e) / L) d phi_e + (lambda / L) i_perp dw.
  const double zd = (kReferenceAngle && tiny) ? 0.0 : 1.0;  // coincident fix-up: d is a constant
  const double gr0 = zd * ex, gr1 = zd * ey;
  const double ge0 = -zd * ey * inv_rho, ge1 = zd * ex * inv_rho;
  const double k1 = -2.0 * t1 * kNPrime, k2 = -2.0 * t2 * kN;
  const double m1 = fma(a, k1, -(b * k2)), m2 = fma(c, k1, d * k2);
  const double thg = theta * kGamma;
  const double rho_BL = -base * inv_L;  // d(-rho / B) / dL
  const double Xr = -inv_B * o.fx, Yr = -inv_B * o.fy;
  const double XL = fma(thg, m1, rho_BL * o.fx), YL = fma(thg, m2, rho_BL * o.fy);
  const double Xe = Bq * m1, Ye = Bq * m2;
  const double Xi = -Xe - o.fy, Yi = o.fx - Ye;  // through theta, and through the rotation of f itself
  const double cil = dot * inv_L;                // (i . e) / L;  i . e_perp = -cross
  const double Xd = fma(Xi, cil, fma(XL, -cross, Xe)), Yd = fma(Yi, cil, fma(YL, -cross, Ye));  // total d / d phi_e
  o.dfx[0] = fma(Xd, ge0, Xr * gr0);
  o.dfx[1] = fma(Xd, ge1, Xr * gr1);
  o.dfy[0] = fma(Yd, ge0, Yr * gr0);
  o.dfy[1] = fma(Yd, ge1, Yr * gr1);
  const double lil = kLambda * inv_L;
  const double XLl = kLambda * XL, Xil = lil * Xi, YLl = kLambda * YL, Yil = lil * Yi;
  o.dfx[2] = fma(XLl, ix, -(Xil * iy));
  o.dfx[3] = fma(XLl, iy, Xil * ix);
  o.dfy[2] = fma(YLl, ix, -(Yil * iy));
  o.dfy[3] = fma(YLl, iy, Yil * ix);
}

// Near-degenerate pair (see above), evaluated with the reference's two-atan2 angle. Rare (exactly (anti)parallel
// set-ups), so it is a real call: out = {fx, fy, dfx[4], dfy[4]} scaled by `sign` on the gradient.
static __device__ __noinline__ void social_pair_reference(double dx, double dy, double wx, double wy, double sign,
                                                          double* out) {
  PairOut o;
  social_pair<true>(dx, dy, wx, wy, o);
  out[0] = o.fx;
  out[1] = o.fy;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    out[2 + c] = sign * o.dfx[c];
    out[6 + c] = sign * o.dfy[c];
  }
}

// ---------------------------------------------------------------------------------------------------
// ceres::BiCubicInterpolator<Grid2D<u_char>> (SURVEY Appendix B): value + d/drow + d/dcol.
// NC = the map may be read through the non-coherent (read-only) path. People-free batches can stream their costmaps
// into the RUNNING kernel (host-buffer pipeline, wait_for_costmap); PTX allows ld.global.nc only for data that is
// read-only for the whole kernel, so those kernels read the maps with coherent ld.global.ca instead.
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void hermite(double p0, double p1, double p2, double p3, double x, double& f, double& dfdx) {
  const double a = 0.5 * (-p0 + 3.0 * p1 - 3.0 * p2 + p3);
  const double b = 0.5 * (2.0 * p0 - 5.0 * p1 + 4.0 * p2 - p3);
  const double c = 0.5 * (-p0 + p2);
  f = p1 + x * (c + x * (b + x * a));
  dfdx = c + x * (2.0 * b + 3.0 * a * x);
}

template <bool NC, class T>
__device__ __forceinline__ T ld_in(const T* p) {
  if (NC) return __ldg(p);
  return __ldca(p);
}

template <bool NC>
__device__ __forceinline__ void bicubic(const uint8_t* map, int size_x, int size_y, double r, double c, double& f,
                                        double& dfdr, double& dfdc) {
  // clamp the cell index so that a non-finite / huge coordinate cannot overflow the int conversion
  const double rf = floor(std_min(std_max(r, -4.0), (double)size_y + 4.0));
  const double cf = floor(std_min(std_max(c, -4.0), (double)size_x + 4.0));
  const int row = (int)rf, col = (int)cf;
  const double xr = r - (double)row, xc = c - (double)col;
  int cc[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) cc[k] = min(max(col - 1 + k, 0), size_x - 1);
  double fr[4], dfr[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int rr = min(max(row - 1 + k, 0), size_y - 1);
    const uint8_t* line = map + (size_t)rr * size_x;
    hermite((double)ld_in<NC>(line + cc[0]), (double)ld_in<NC>(line + cc[1]), (double)ld_in<NC>(line + cc[2]),
            (double)ld_in<NC>(line + cc[3]), xc, fr[k], dfr[k]);
  }
  double unused;
  hermite(fr[0], fr[1], fr[2], fr[3], xr, f, dfdr);
  hermite(dfr[0], dfr[1], dfr[2], dfr[3], xr, dfdc, unused);
}

// steps k < j that belong to block beta: blocks hold bl steps, block `last` (= the problem's last block) extends to the
// horizon end, blocks beyond it do not exist for this problem
__device__ __forceinline__ int steps_in_block_before(int j, int beta, int bl, int last) {
  const int n = j - beta * bl;
  if (beta > last) return 0;
  if (beta == last) return max(n, 0);
  return min(max(n, 0), bl);
}

// AgentAngleCost branch selection (reference agent_angle_cost_function.hpp:125-195): depends only on
// constants of the problem, so it is evaluated once per solve. Returns the steering target angle or NaN
// when the residual is identically zero for this step.
__device__ __forceinline__ double agent_angle_target(const DevBatch& bt, const Prob& pb, int step_plus_1) {
  const int stride = bt.S + 1;
  int closest = -1;
  double best = INFINITY;
  for (int k = 0; k < bt.A; ++k) {
    const double* a = pb.agents + (size_t)k * 6 * stride + step_plus_1;
    const double dx = a[0] - pb.x0, dy = a[stride] - pb.y0;
    const double d2 = dx * dx + dy * dy;
    if (d2 < best && a[4 * stride] > 0.05) {
      best = d2;
      closest = k;
    }
  }
  if (closest < 0 || best > 4.0) return NAN;
  const double* a = pb.agents + (size_t)closest * 6 * stride + step_plus_1;
  const double bearing = atan2(a[stride] - pb.y0, a[0] - pb.x0);
  const double hd_arg = a[2 * stride] - pb.yaw0;
  const double hd = atan2(sin(hd_arg), cos(hd_arg));
  const double wb_arg = bearing - pb.yaw0;
  const double wb = atan2(sin(wb_arg), cos(wb_arg));
  if (hd <= -(5 * M_PI / 6.0) || hd >= (M_PI / 6.0)) {
    if (wb < 0.0) return NAN;
    return pb.yaw0 + (-(M_PI / 6.0));
  }
  if (wb > 0.0) return NAN;
  return pb.yaw0 + (M_PI / 6.0);
}
#define SMPC_UNROLL _Pragma("unroll")
// The log2(G) levels of the Kogge-Stone scans stay a loop: unrolled, the shuffle ladder of the 2 + 4 NB scans is ~16 kB of
// SASS per evaluation, and the evaluation is instruction-fetch bound (its code does not fit the 32 kB L1.5 I-cache)
// (measured: -16 kB; +3..5 % with people). Small groups have 2 - 3 levels and 7 chunks per evaluation: there the loop
// overhead costs more than the code (-25 % on 65536 people-free problems at G = 4), so they keep the ladder unrolled.
template <int G, class F>
__device__ __forceinline__ void scan_levels(F level) {
  if (G <= 8) {
    SMPC_UNROLL for (int d = 1; d < G; d <<= 1) level(d);
  } else {
    _Pragma("unroll 1") for (int d = 1; d < G; d <<= 1) level(d);
  }
}

// ---------------------------------------------------------------------------------------------------
// Work mapping: a GROUP of G lanes (G = 4, 8, 16 or 32) solves one problem, so a warp holds 32/G problems.
// Lane gl of the group owns horizon steps gl, gl+G, gl+2G, ... ("chunks" of G consecutive steps are scanned
// across the group, carries go through shared memory). G = 32 is the latency mapping (one step per lane);
// small G is the throughput mapping: the scan / reduction overheads and the group-leader solver logic are then
// shared by 32/G problems per warp.
// ---------------------------------------------------------------------------------------------------

// Per-group shared-memory state. Buffers hold [cost_diff, cost_plain, g[P], H[NH]] (H row-major lower triangle,
// H[a(a+1)/2 + b], a >= b) of the current iterate and of the trial point; the LM vectors follow.
//   cost_diff  = 1/2 sum r^2 as a DIFFERENTIATED evaluation of the reference computes it (Jets),
//   cost_plain = the same sum as a cost-only (double) evaluation computes it.
// They differ only under ceres_compat < 210, where ProxemicsCost evaluates differently under Jets (evaluate()).
constexpr int kRedStride = 33;  // odd stride of the per-warp reduction scratch: conflict-free rows and columns

// D = parameters per block: 2 = (v, w), the reference's unicycle (update_state.hpp:46-61); 3 = (vx, vy, w), the
// omnidirectional extension (holonomic Euler step x += (vx cos th - vy sin th) dt, consistent with the reference's
// trajectorizer, path_trajectorizer.hpp:106-123; the reference has no omnidirectional SOLVE).
// WT = the weighted solve kernel: the group's problem carries its own critic weights in a 9-double slot (kWt).
template <int NB, int D = 2, bool WT = false>
struct Layout {
  static constexpr int P = D * NB;
  static constexpr int NH = P * (P + 1) / 2;
  static constexpr int NG = 2 + P;       // cost_diff, cost_plain, g[P]: the part every evaluation reduces
  static constexpr int NE = NG + NH;     // ... plus J^T J
  static constexpr int NC = 4 + 4 * NB;  // scan carries: X, Y, sin, cos of the heading, 4 NB sensitivities
  static constexpr int kBuf0 = 0;
  static constexpr int kBuf1 = NE;
  static constexpr int kX = 2 * NE;
  static constexpr int kBest = kX + P;
  static constexpr int kScale = kBest + P;
  static constexpr int kDiag = kScale + P;
  static constexpr int kDelta = kDiag + P;
  static constexpr int kCand = kDelta + P;
  static constexpr int kCarry = kCand + P;
  static constexpr int kYaw = kCarry + NC;  // sin, cos of yaw0
  static constexpr int kState = kYaw + 2;    // LmState (solver scalars parked here across the evaluation)
  static constexpr int kProb = kState + 22;  // Prob (group-uniform problem view)
  static constexpr int kWt = kProb + 18;  // critic weights of the problem [9] (WT only)
  static constexpr int kAa = kWt + (WT ? 9 : 0);  // agent-angle steering target per step [S]
  __host__ __device__ static constexpr int total(int S) { return ((kAa + S) | 1); }  // odd stride: no bank conflicts
  static constexpr int kRedDoubles = NE * kRedStride;  // per-WARP scratch behind the per-group regions
  __host__ __device__ static constexpr int g(int c) { return 2 + c; }
  __host__ __device__ static constexpr int h(int a, int b) { return NG + a * (a + 1) / 2 + b; }
};

// Layout<NB>::total(S) for a run-time NB (the host sizes the parking area of the time-sliced queue with it).
__host__ __device__ constexpr int layout_total(int nb, int S, int dof = 2) {
  const int P = dof * nb, NE = 2 + P + P * (P + 1) / 2, NC = 4 + 4 * nb;
  return ((2 * NE + 6 * P + NC + 2 + 22 + 18 + S) | 1);
}
static_assert(layout_total(3, 28) == Layout<3>::total(28) && layout_total(5, 38) == Layout<5>::total(38) &&
                  layout_total(18, 18) == Layout<18>::total(18) && layout_total(3, 28, 3) == Layout<3, 3>::total(28),
              "layout_total must mirror Layout<NB>::total");

template <int G>
struct Group {
  static constexpr int kLog2 = (G == 32) ? 5 : (G == 16) ? 4 : (G == 8) ? 3 : (G == 4) ? 2 : (G == 2) ? 1 : 0;
  static constexpr int kPerWarp = 32 / G;
  __device__ static __forceinline__ unsigned mask(int lane) {
    return (G == 32) ? kFullMask : (((1u << G) - 1u) << (lane & ~(G - 1)));
  }
};

__device__ __forceinline__ double wrap_angle(double a) {
  // atan2(sin a, cos a) of the reference critics, evaluated as a - 2 pi round(a / 2 pi) (|difference| ~ 1 ulp of pi)
  return a - (2.0 * M_PI) * rint(a * (0.5 / M_PI));
}

// Solver scalars of one group, resident in shared memory and touched ONLY by the group's first lane (between
// __syncwarp pairs), so that no update depends on the lanes of a group running in lock-step.
enum Phase { kFetch = 0, kInit = 1, kLineSearch = 2, kFullStep = 3 };
struct LmState {
  double x_cost, x_norm, gmax, radius, decrease_factor, minimum_cost, it_cost, cost_initial, cost_final,
      model_cost_change, g0, dmax, t, prev_x, prev_value, prev_gradient;
  double se_cost;  // TrustRegionStepEvaluator::current_cost_: iteration-zero cost, then the last accepted CANDIDATE cost
  int iteration, n_invalid, n_eval, n_light, ls_iters, term, phase, b, flags, pad_;
};
static_assert(sizeof(LmState) == 22 * sizeof(double), "Layout::kState reserves 22 doubles");
static_assert(sizeof(Prob) <= 18 * sizeof(double), "Layout::kProb reserves 18 doubles");
enum StateFlags {
  kReuseDiagonal = 1, kItSuccessful = 2, kAnySuccess = 4, kPrevOk = 8, kLive = 16, kExhausted = 32, kSwapped = 64,
  kDrained = 128,  // this group has seen the main queue empty
  kClosed = 256,   // ... and the parked queue closed and empty: nothing will ever come again
  kFinished = 512  // the leader has terminated the solve: all lanes write the results, then the group fetches again
};

// ---------------------------------------------------------------------------------------------------
// Evaluation at block values xs[P] (group shared memory): cost = 1/2 sum r^2, g = J^T r and (when wanted) H = J^T J,
// written to out[NE] (group shared memory). Residual set and order of reference src/optimizer.cpp:251-371
// (SURVEY Appendix D). Must be called by all 32 lanes of the warp (scans use full-mask shuffles of width G);
// `live` = this group holds a problem.
// `st` (solve kernel) lets the evaluation stop early: a line-search sample that fails the Armijo test is used for
// its cost and directional derivative only (Ceres evaluates exactly cost + gradient there, line_search.cc), so its
// J^T J is not built and kNoHessian is returned. st == nullptr: always build J^T J.
// ---------------------------------------------------------------------------------------------------
// Critic weight k of DevParams' w_* order: the kernel parameter, or (WT) the problem's row in the group's workspace.
#define SMPC_W(field, k) (WT ? ws[L::kWt + (k)] : prm.field)
template <int NB, int G, bool PPL, int D = 2, bool WT = false>
__device__ __forceinline__ unsigned evaluate(const DevParams& prm, const DevBatch& bt, const Prob& pb, bool live,
                                             double* ws, double* red, const double* xs, int lane, double* out,
                                             const LmState* st) {
  using L = Layout<NB, D, WT>;
  constexpr int P = L::P;
  const int gl = lane & (G - 1);
  const unsigned gmask = Group<G>::mask(lane);
  const int Sb = live ? pb.S : 0;
  // the scans are warp-wide shuffles: every group of the warp walks as many chunks as the longest horizon among them
  const int Sw = (G == 32) ? Sb : __reduce_max_sync(kFullMask, Sb);
  const int bl = pb.bl, last_b = pb.nb - 1, ch = pb.ch;
  const double dt = bt.dt;
  const int stride = bt.S + 1;
  const double inv_res = 1.0 / bt.resolution;
  double* carry = ws + L::kCarry;
  const double* aa = ws + L::kAa;
  const int col0 = lane & ~(G - 1);
  unsigned flags = 0;
  bool need_h = true;
  bool bad_res = false, bad_jac = false;

  // heading before the group's first step: sin / cos of yaw0 (stored at problem set-up), then carried chunk to chunk
  const double s0 = ws[L::kYaw], c0 = ws[L::kYaw + 1];

#pragma unroll 1
  for (int base = 0; base < Sw; base += G) {
    const int j = base + gl;
    const bool act = j < Sb;
    const bool first = (base == 0);
    const bool last = (base + G >= Sw);
    // block of step j (j / bl capped at the problem's last block) and d theta_j / d w_b = dt #{steps < j in block b}
    int bj = 0;
    SMPC_UNROLL for (int b = 1; b < NB; ++b) bj += (j >= b * bl && b <= last_b) ? 1 : 0;
    double vj = xs[0], wj = xs[D - 1];
    double vyj = 0.0;     // lateral velocity of the step's block (omnidirectional blocks only)
    double Th = pb.yaw0;  // heading AFTER step j = yaw0 + sum_b w_b dt #{steps <= j in block b}
    double tau[NB];       // d theta_j / d w_b (heading before step j)
    SMPC_UNROLL for (int b = 0; b < NB; ++b) {
      if (b == bj) {
        vj = xs[D * b];
        wj = xs[D * b + D - 1];
        if (D == 3) vyj = xs[D * b + 1];
      }
      tau[b] = dt * (double)steps_in_block_before(j, b, bl, last_b);
      Th += xs[D * b + D - 1] * tau[b];
    }
    Th += wj * dt;
    // one sincos per step: lane j evaluates the heading after its step; the heading before it is the
    // previous lane's (the previous chunk's last lane / yaw0 for the group's first lane)
    double sT, cT;
    sincos(Th, &sT, &cT);
    double sn = __shfl_up_sync(kFullMask, sT, 1, G);
    double cs = __shfl_up_sync(kFullMask, cT, 1, G);
    if (gl == 0) {
      sn = first ? s0 : carry[2];
      cs = first ? c0 : carry[3];
    }
    const double cdt = act ? cs * dt : 0.0, sdt = act ? sn * dt : 0.0;
    // displacement of step j: unicycle v (cos, sin) dt; omnidirectional R(theta) (vx, vy) dt
    const double aj = (D == 3) ? vj * cdt - vyj * sdt : vj * cdt;
    const double bjv = (D == 3) ? vj * sdt + vyj * cdt : vj * sdt;

    // ---- positions: two scans -----------------------------------------------------------------------------
    double sx = aj, sy = bjv;
    scan_levels<G>([&](int d) {
      const double tx = __shfl_up_sync(kFullMask, sx, d, G);
      const double ty = __shfl_up_sync(kFullMask, sy, d, G);
      const double m = (gl >= d) ? 1.0 : 0.0;
      add_masked(sx, tx, m);
      add_masked(sy, ty, m);
    });
    const double X = (first ? pb.x0 : carry[0]) + sx;
    const double Y = (first ? pb.y0 : carry[1]) + sy;

    // ---- people critics (k = 0, 1, 2), BEFORE the sensitivity scans: the pair loop and the 4 NB scan registers are
    //      never live together. Each critic leaves its residual and its gradient wrt (X, Y, Theta, lv). ----------
    double ra = 0.0, caT = 0.0;                                // AgentAngle: residual, d/dTheta
    double rs = 0.0, sX = 0.0, sY = 0.0, sTh = 0.0, sL = 0.0;  // SocialWork
    double sM = 0.0;                                           // ... d/d(lateral velocity), omnidirectional only
    double rp = 0.0, pX = 0.0, pY = 0.0;                       // Proxemics (differentiated evaluation)
    double cprox_plain = 0.0;                                  // 1/2 r^2 of Proxemics as a cost-only evaluation sees it
    if (PPL && act && pb.has_people) {  // PPL == false: the people critics are compiled out (people-free batch)
      // --- AgentAngle (k=0): w * wrap(Theta - target)^2 ------------------------------------------
      const double tgt = aa[j];
      if (tgt == tgt) {
        const double del = wrap_angle(Th - tgt);
        ra = SMPC_W(w_agent_angle, 4) * (del * del);
        caT = 2.0 * SMPC_W(w_agent_angle, 4) * del;
      }
      // --- SocialWork (k=1) and Proxemics (k=2) ----------------------------------------------------
      // robot velocity uses lv = v_{b(i)} and the NEW heading (omnidirectional: the body velocity rotated into the world)
      const double rvx = (D == 3) ? vj * cT - vyj * sT : vj * cT;
      const double rvy = (D == 3) ? vj * sT + vyj * cT : vj * sT;
      double Frx = 0.0, Fry = 0.0;
      double JFx[4] = {0, 0, 0, 0}, JFy[4] = {0, 0, 0, 0};
      double wp = 0.0;
      double G4[4] = {0, 0, 0, 0};  // gradient of (wr + wp) wrt (dX, dY, dvx, dvy) of the robot
      double dmin = DBL_MAX, pdx = 0.0, pdy = 0.0;
      const bool do_social = SMPC_W(w_social, 1) != 0.0;
      // agent records (x, y, vx, vy) of step j+1, one 32-byte sector each; the next agent's record is fetched
      // while the current pair interaction is evaluated
      const double2* rec = reinterpret_cast<const double2*>(pb.packed) + ((size_t)(j + 1)) * 2;
      const uint8_t* vld = pb.valid + (j + 1);
      double2 nxt_p = __ldg(rec);
      double2 nxt_v = __ldg(rec + 1);
      unsigned char nxt_valid = __ldg(vld);  // tested only in the NEXT iteration: no wait on the load here
#ifndef SMPC_PAIR_UNROLL
#define SMPC_PAIR_UNROLL 1
#endif
      constexpr int kPairUnroll = SMPC_PAIR_UNROLL;
#pragma unroll kPairUnroll
      for (int k = 0; k < bt.A; ++k) {
        const double ax = nxt_p.x, ay = nxt_p.y, avx = nxt_v.x, avy = nxt_v.y;
        const bool valid = nxt_valid != 0;
        if (k + 1 < bt.A) {
          rec += (size_t)stride * 2;
          vld += stride;
          nxt_p = __ldg(rec);
          nxt_v = __ldg(rec + 1);
          nxt_valid = __ldg(vld);
        }
        const double ddx = X - ax, ddy = Y - ay;
        {  // closest valid agent (proxemics), branch-free
          const double d2 = ddx * ddx + ddy * ddy;
          const bool closer = valid && d2 < dmin;
          dmin = closer ? d2 : dmin;
          pdx = closer ? ddx : pdx;
          pdy = closer ? ddy : pdy;
        }
        if (do_social) {
          // F(robot <- agent k) = pair(d, w) with d = robot - agent, w = v_robot - v_agent, and
          // F(agent k <- robot) = pair(-d, -w). The pair function is odd, pair(-d, -w) = -pair(d, w) (e, I and
          // their unit vectors flip, theta / B / |d| do not), so ONE evaluation serves both terms of the
          // residual; only the near-degenerate branch (reference rounding decides theta = +-pi / 0) is evaluated
          // per role. Padded agents (SURVEY Q5) only have the agent <- robot term.
          PairOut po;
          social_pair<false>(ddx, ddy, rvx - avx, rvy - avy, po);
          const bool degenerate = po.degenerate;
          if (degenerate) {
            double ref[10];
            social_pair_reference(ddx, ddy, rvx - avx, rvy - avy, 1.0, ref);
            po.fx = ref[0];
            po.fy = ref[1];
            SMPC_UNROLL for (int c = 0; c < 4; ++c) {
              po.dfx[c] = ref[2 + c];
              po.dfy[c] = ref[6 + c];
            }
          }
          {  // robot <- agent term of valid agents only: fma(1, f, F) is F + f exactly, fma(0, f, F) is F
            const double m = valid ? 1.0 : 0.0;
            Frx = fma(m, po.fx, Frx);
            Fry = fma(m, po.fy, Fry);
            SMPC_UNROLL for (int c = 0; c < 4; ++c) {
              JFx[c] = fma(m, po.dfx[c], JFx[c]);
              JFy[c] = fma(m, po.dfy[c], JFy[c]);
            }
          }
          if (degenerate) {
            double ref[10];
            social_pair_reference(-ddx, -ddy, avx - rvx, avy - rvy, -1.0, ref);  // d(-d)/dX = -1: gradient sign
            po.fx = ref[0];
            po.fy = ref[1];
            SMPC_UNROLL for (int c = 0; c < 4; ++c) {
              po.dfx[c] = ref[2 + c];
              po.dfy[c] = ref[6 + c];
            }
          }
          wp = fma(po.fy, po.fy, fma(po.fx, po.fx, wp));
          SMPC_UNROLL for (int c = 0; c < 4; ++c) G4[c] = fma(po.fy, po.dfy[c], fma(po.fx, po.dfx[c], G4[c]));  // (x 2 below)
        }
      }
      if (do_social) {
        const double wr = Frx * Frx + Fry * Fry;
        SMPC_UNROLL for (int c = 0; c < 4; ++c) G4[c] = 2.0 * fma(Fry, JFy[c], fma(Frx, JFx[c], G4[c]));
        rs = SMPC_W(w_social, 1) * (wr + wp + 1e-6);
        sX = SMPC_W(w_social, 1) * G4[0];
        sY = SMPC_W(w_social, 1) * G4[1];
        sL = SMPC_W(w_social, 1) * (G4[2] * cT + G4[3] * sT);
        if (D == 3) {
          sM = SMPC_W(w_social, 1) * (-G4[2] * sT + G4[3] * cT);
          sTh = SMPC_W(w_social, 1) * (-G4[2] * rvy + G4[3] * rvx);
        } else {
          sTh = SMPC_W(w_social, 1) * vj * (-G4[2] * sT + G4[3] * cT);
        }
      }
      // Proxemics: w * 3 * exp(-dmin / 0.25), proxemics_cost_function.hpp:128-149.
      //  * Ceres >= 2.1: std::numeric_limits<Jet>::max() is DBL_MAX. With no valid agent the value is 0 but the jet
      //    derivative is (-inf) * 0 = NaN, i.e. the differentiated evaluation fails (SURVEY Q7).
      //  * Ceres 2.0.0 (ceres_compat < 210) has no numeric_limits specialisation for Jets: the primary template returns
      //    Jet() = 0, std::min keeps it, and every DIFFERENTIATED evaluation sees the constant residual 3 w with a zero
      //    Jacobian row, while cost-only evaluations (candidate cost) see the true minimum distance.
      const double r_true = (dmin == DBL_MAX) ? 0.0 : SMPC_W(w_prox, 5) * (3.0 * exp(-dmin / (0.5 * 0.5)));
      cprox_plain = 0.5 * r_true * r_true;
      if (prm.ceres_compat < 210) {
        rp = SMPC_W(w_prox, 5) * 3.0;
      } else if (dmin == DBL_MAX) {
        flags |= kJacobianBad;
      } else {
        rp = r_true;
        const double k = -r_true * (2.0 / (0.5 * 0.5));
        pX = k * pdx;
        pY = k * pdy;
      }
    }

    // ---- forward sensitivities: 4 NB scans ---------------------------------------------------------------------
    double sd[4 * NB];
    SMPC_UNROLL for (int b = 0; b < NB; ++b) {
      sd[4 * b + 0] = (b == bj) ? cdt : 0.0;  // dX/dv_b
      sd[4 * b + 1] = (b == bj) ? sdt : 0.0;  // dY/dv_b
      sd[4 * b + 2] = -bjv * tau[b];          // dX/dw_b
      sd[4 * b + 3] = aj * tau[b];            // dY/dw_b
    }
    scan_levels<G>([&](int d) {
      const double m = (gl >= d) ? 1.0 : 0.0;
      SMPC_UNROLL for (int e = 0; e < 4 * NB; ++e) add_masked(sd[e], __shfl_up_sync(kFullMask, sd[e], d, G), m);
    });
    if (!first) {
      SMPC_UNROLL for (int e = 0; e < 4 * NB; ++e) sd[e] += carry[4 + e];
    }
    if (!last) {  // hand the inclusive totals to the next chunk
      __syncwarp(gmask);
      if (gl == G - 1) {
        carry[0] = X;
        carry[1] = Y;
        carry[2] = sT;
        carry[3] = cT;
        SMPC_UNROLL for (int e = 0; e < 4 * NB; ++e) carry[4 + e] = sd[e];
      }
      __syncwarp(gmask);
    }

    // Column pa of the lane's sensitivity matrix D (rows X, Y, Theta, L, M), as (dX, dY, third component) + its kind:
    //   kind 0  v_b / vx_b : (sum cos dt, sum sin dt, [b == bj] on L)
    //   kind 1  vy_b       : (-sum sin dt, sum cos dt, [b == bj] on M)          (omnidirectional blocks only)
    //   kind 2  w_b        : (dX/dw_b, dY/dw_b, dTheta/dw_b on Theta)
    // pa is a compile-time constant wherever this is called (unrolled loops), so the selects fold away.
    auto column = [&](int pa, double& cx, double& cy, double& c3) -> int {
      const int ba = pa / D, k = pa % D;
      if (k == D - 1) {
        cx = sd[4 * ba + 2];
        cy = sd[4 * ba + 3];
        c3 = tau[ba] + ((ba == bj) ? dt : 0.0);  // d Theta_j / d w_ba (heading after step j)
        return 2;
      }
      c3 = (ba == bj) ? 1.0 : 0.0;
      if (k == 0) {
        cx = sd[4 * ba + 0];
        cy = sd[4 * ba + 1];
        return 0;
      }
      cx = -sd[4 * ba + 1];
      cy = sd[4 * ba + 0];
      return 1;
    };
    // per-lane Gauss-Newton block wrt (X, Y, Theta, lv): M = sum c c^T (10 entries), q = sum c r
    double mXX = 0, mXY = 0, mXT = 0, mXL = 0, mYY = 0, mYT = 0, mYL = 0, mTT = 0, mTL = 0, mLL = 0;
    double qX = 0, qY = 0, qT = 0, qL = 0;
    // omnidirectional blocks add the lateral velocity M as a fifth coordinate of the lane block
    double mXM = 0, mYM = 0, mTM = 0, mLM = 0, mMM = 0, qM = 0;
    if (act) {
      double cost = 0.0;
      if (PPL) {  // fold the people critics in (all zero for a problem without people)
        cost += 0.5 * ra * ra;
        mTT += caT * caT;
        qT += caT * ra;
        cost += 0.5 * rs * rs;
        mXX += sX * sX; mXY += sX * sY; mXT += sX * sTh; mXL += sX * sL;
        mYY += sY * sY; mYT += sY * sTh; mYL += sY * sL;
        mTT += sTh * sTh; mTL += sTh * sL; mLL += sL * sL;
        qX += sX * rs; qY += sY * rs; qT += sTh * rs; qL += sL * rs;
        if (D == 3) {
          mXM += sX * sM; mYM += sY * sM; mTM += sTh * sM; mLM += sL * sM; mMM += sM * sM;
          qM += sM * rs;
        }
        mXX += pX * pX; mXY += pX * pY; mYY += pY * pY;
        qX += pX * rp; qY += pY * rp;
      }
      // --- Velocity (k=3): w (0.6 - v_b)^2 for i < ch ---------------------------------------------------
      if (j < ch) {
        const double e = 0.6 - vj;
        if (D == 3) {  // omnidirectional extension: w ((0.6 - vx)^2 + vy^2)
          const double r = SMPC_W(w_velocity, 2) * e * e + SMPC_W(w_velocity, 2) * vyj * vyj;
          const double cL = -2.0 * SMPC_W(w_velocity, 2) * e, cM = 2.0 * SMPC_W(w_velocity, 2) * vyj;
          cost += 0.5 * r * r;
          mLL += cL * cL; mLM += cL * cM; mMM += cM * cM;
          qL += cL * r; qM += cM * r;
        } else {
          const double r = SMPC_W(w_velocity, 2) * e * e;
          const double cL = -2.0 * SMPC_W(w_velocity, 2) * e;
          cost += 0.5 * r * r;
          mLL += cL * cL;
          qL += cL * r;
        }
      }
      // --- GoalAlign (k=4): w * wrap(psi - Theta)^2 -----------------------------------------------------
      {
        const double turn = wrap_angle(pb.goal_yaw - Th);
        const double r = SMPC_W(w_goal, 8) * turn * turn;
        const double cTh = -2.0 * SMPC_W(w_goal, 8) * turn;
        cost += 0.5 * r * r;
        mTT += cTh * cTh;
        qT += cTh * r;
      }
      // --- PathFollow (k=5, final seed point) and PathAlign (k=6, seed point i+1): w (|p - t|^2)^2 -----
      {
        const double ex = X - pb.fin_x, ey = Y - pb.fin_y;
        const double q2 = ex * ex + ey * ey;
        const double r = SMPC_W(w_distance, 0) * q2 * q2;
        const double k = 4.0 * SMPC_W(w_distance, 0) * q2;
        const double cX = k * ex, cY = k * ey;
        cost += 0.5 * r * r;
        mXX += cX * cX; mXY += cX * cY; mYY += cY * cY;
        qX += cX * r; qY += cY * r;
      }
      {
        const double ex = X - ld_in<PPL>(pb.px + j + 1), ey = Y - ld_in<PPL>(pb.px + stride + j + 1);
        const double q2 = ex * ex + ey * ey;
        const double r = SMPC_W(w_angle, 3) * q2 * q2;
        const double k = 4.0 * SMPC_W(w_angle, 3) * q2;
        const double cX = k * ex, cY = k * ey;
        cost += 0.5 * r * r;
        mXX += cX * cX; mXY += cX * cY; mYY += cY * cY;
        qX += cX * r; qY += cY * r;
      }
      // --- Obstacle (k=7): w * bicubic(costmap) 0.25 m ahead ---------------------------------------------
      {
        const double fxw = X + 0.25 * cT, fyw = Y + 0.25 * sT;
        const double gx = (fxw - pb.org_x) * inv_res, gy = (fyw - pb.org_y) * inv_res;
        double f, dfdr, dfdc;
        bicubic<PPL>(pb.map, bt.size_x, bt.size_y, gy, gx, f, dfdr, dfdc);
        const double r = SMPC_W(w_obstacle, 7) * f;
        const double kx = SMPC_W(w_obstacle, 7) * dfdc * inv_res, ky = SMPC_W(w_obstacle, 7) * dfdr * inv_res;
        const double cTh = 0.25 * (-kx * sT + ky * cT);
        cost += 0.5 * r * r;
        mXX += kx * kx; mXY += kx * ky; mXT += kx * cTh;
        mYY += ky * ky; mYT += ky * cTh; mTT += cTh * cTh;
        qX += kx * r; qY += ky * r; qT += cTh * r;
      }

      // --- cost and g = D^T q into column `lane` of the warp's scratch red[NE][33]. First chunk: plain stores (no
      //     zero fill, no read-modify-write); later chunks accumulate (`first` is warp-uniform, so the two store
      //     flavours are a branch, not a select per entry). Column of v_b: (dX, dY, 0, [b == bj]); of w_b:
      //     (dX, dY, dTheta, 0). -----------------------------------------------------------------------------
      {
        const double c_diff = cost + 0.5 * rp * rp, c_plain = cost + cprox_plain;
        double* r0 = red + lane;
        auto put_g = [&](auto is_first) {
          constexpr bool kFirst = decltype(is_first)::value;
          r0[0 * kRedStride] = (kFirst ? 0.0 : r0[0 * kRedStride]) + c_diff;
          r0[1 * kRedStride] = (kFirst ? 0.0 : r0[1 * kRedStride]) + c_plain;
          SMPC_UNROLL for (int pa = 0; pa < P; ++pa) {
            double cx, cy, cs3;
            const int kind = column(pa, cx, cy, cs3);
            double* gp = r0 + L::g(pa) * kRedStride;
            *gp = (kFirst ? 0.0 : *gp) + (qX * cx + qY * cy + ((kind == 0) ? qL : (kind == 1) ? qM : qT) * cs3);
          }
        };
        if (first) put_g(std::true_type{}); else put_g(std::false_type{});
      }
    } else if (first) {  // a lane without a step in the first chunk still owns a column of the column sums
      SMPC_UNROLL for (int e = 0; e < L::NG; ++e) red[e * kRedStride + lane] = 0.0;
    }

    if (last) {
      // --- VelocityFeasibility (k=8), cost and gradient part: w ((v_i - v_{i-1})^2 + (w_i - w_{i-1})^2),
      //     0 < i < ch/bl, on blocks i, i-1. Parameter-space residuals: the group's first lane adds them. -------
      if (gl == 0 && live) {
        SMPC_UNROLL for (int i = 1; i < NB; ++i) {
          if (i < pb.nbd) {
            double dk[D], r = 0.0;
            SMPC_UNROLL for (int k = 0; k < D; ++k) {
              dk[k] = xs[D * i + k] - xs[D * (i - 1) + k];
              r += SMPC_W(w_vf, 6) * dk[k] * dk[k];
            }
            red[0 * kRedStride + lane] += 0.5 * r * r;
            red[1 * kRedStride + lane] += 0.5 * r * r;
            SMPC_UNROLL for (int k = 0; k < D; ++k) {
              const double jk = 2.0 * SMPC_W(w_vf, 6) * dk[k];
              red[L::g(D * (i - 1) + k) * kRedStride + lane] -= jk * r;
              red[L::g(D * i + k) * kRedStride + lane] += jk * r;
            }
          }
        }
      }
      // --- group column sums of [cost_diff, cost_plain, g]: lane r of the group sums entries r, r + G, ... -----
      __syncwarp();
      for (int e = gl; e < L::NG; e += G) {
        const double* row = red + e * kRedStride + col0;
        double t0 = 0.0, t1 = 0.0;
        SMPC_UNROLL for (int t = 0; t < G; t += 2) {
          t0 += row[t];
          t1 += row[t + 1];
        }
        const double tot = t0 + t1;
        out[e] = tot;
        if (!isfinite(tot)) {
          if (e < 2) bad_res = true; else bad_jac = true;
        }
      }
      if (__any_sync(gmask, bad_res)) flags |= kResidualBad;
      if (__any_sync(gmask, bad_jac)) flags |= kJacobianBad;
      flags = __reduce_or_sync(gmask, flags);
      __syncwarp(gmask);
      // --- does this point need J^T J? Not if it is a line-search sample that fails the sufficient-decrease test
      //     (group-uniform: every lane reads the same shared-memory words) ---------------------------------------
      if (st != nullptr && live && st->phase == kLineSearch) {
        const bool armijo_ok = (flags == 0) && !(out[0] > st->x_cost + 1e-4 * st->g0 * st->t);
        need_h = armijo_ok;
      }
    }

    // --- lane block -> J^T J, one column at a time (T = M D[:,a] is never stored) ---------------------------------
    if (need_h) {
      if (act) {
        double* r0 = red + lane;
        auto put_h = [&](auto is_first) {
          constexpr bool kFirst = decltype(is_first)::value;
          SMPC_UNROLL for (int pa = 0; pa < P; ++pa) {
            double ax, ay, as3;
            const int ka = column(pa, ax, ay, as3);
            // T = M d_a over (X, Y, Theta, L, M); the third component of d_a sits on L (kind 0), M (1) or Theta (2)
            const double t0 = mXX * ax + mXY * ay + ((ka == 0) ? mXL : (ka == 1) ? mXM : mXT) * as3;
            const double t1 = mXY * ax + mYY * ay + ((ka == 0) ? mYL : (ka == 1) ? mYM : mYT) * as3;
            const double t2 = mXT * ax + mYT * ay + ((ka == 0) ? mTL : (ka == 1) ? mTM : mTT) * as3;
            const double t3 = mXL * ax + mYL * ay + ((ka == 0) ? mLL : (ka == 1) ? mLM : mTL) * as3;
            const double t4 = mXM * ax + mYM * ay + ((ka == 0) ? mLM : (ka == 1) ? mMM : mTM) * as3;
            SMPC_UNROLL for (int pb2 = 0; pb2 <= pa; ++pb2) {
              double bx, by, bs3;
              const int kb = column(pb2, bx, by, bs3);
              double* p = r0 + L::h(pa, pb2) * kRedStride;
              *p = (kFirst ? 0.0 : *p) + (bx * t0 + by * t1 + bs3 * ((kb == 0) ? t3 : (kb == 1) ? t4 : t2));
            }
          }
        };
        if (first) put_h(std::true_type{}); else put_h(std::false_type{});
      } else if (first) {
        SMPC_UNROLL for (int e = L::NG; e < L::NE; ++e) red[e * kRedStride + lane] = 0.0;
      }
    }
  }

  if (need_h) {
    // VelocityFeasibility, J^T J part. Row of residual i: -j_k at block i-1, +j_k at block i, j_k = 2 w (u_i - u_{i-1})_k
    if (gl == 0 && live) {
      SMPC_UNROLL for (int i = 1; i < NB; ++i) {
        if (i < pb.nbd) {
          double jk[D];
          SMPC_UNROLL for (int k = 0; k < D; ++k) jk[k] = 2.0 * SMPC_W(w_vf, 6) * (xs[D * i + k] - xs[D * (i - 1) + k]);
          SMPC_UNROLL for (int k = 0; k < D; ++k) {
            SMPC_UNROLL for (int l = 0; l < D; ++l) {
              const double v = jk[k] * jk[l];
              if (l <= k) {
                red[(L::h(D * i + k, D * i + l)) * kRedStride + lane] += v;
                red[(L::h(D * (i - 1) + k, D * (i - 1) + l)) * kRedStride + lane] += v;
              }
              red[(L::h(D * i + k, D * (i - 1) + l)) * kRedStride + lane] -= v;
            }
          }
        }
      }
    }
  }
  // (full-warp barrier: groups that skip J^T J still take part; their rows are simply not summed)
  __syncwarp();
  if (need_h) {
    bool bad_h = false;
    for (int e = L::NG + gl; e < L::NE; e += G) {
      const double* row = red + e * kRedStride + col0;
      double t0 = 0.0, t1 = 0.0;
      SMPC_UNROLL for (int t = 0; t < G; t += 2) {
        t0 += row[t];
        t1 += row[t + 1];
      }
      const double tot = t0 + t1;
      out[e] = tot;
      if (!isfinite(tot)) bad_h = true;
    }
    if (__any_sync(gmask, bad_h)) flags |= kJacobianBad;
  } else {
    flags |= kNoHessian;
  }
  __syncwarp();
  return flags;
}
#undef SMPC_W

// ---------------------------------------------------------------------------------------------------
// Interpolating-polynomial minimiser of the Armijo line search (ceres polynomial.cc, SURVEY Appendix A).
// Ceres fits the polynomial with a pivoted LU and finds the critical points as companion-matrix eigenvalues;
// the same polynomial is fitted here in closed form (Hermite data) and the roots of its derivative in closed
// form too (quadratic: Ceres' own formula; quartic: Ferrari + Newton polish, Aberth-Ehrlich as the safety net).
// Warp-uniform scalar code; called only when a trial step fails the sufficient-decrease test.
// ---------------------------------------------------------------------------------------------------
struct LsSample {
  double x, value, gradient;
  bool ok;
};

__device__ __forceinline__ double horner5(const double (&m)[6], double x) {
  return m[0] + x * (m[1] + x * (m[2] + x * (m[3] + x * (m[4] + x * m[5]))));
}

// Real parts of the 4 roots of c[0] + c[1] x + ... + c[4] x^4 by Aberth-Ehrlich (slow, robust).
static __device__ __noinline__ void quartic_aberth(const double* c, double* re) {
  double m[5];  // monic, highest first
  for (int i = 0; i <= 4; ++i) m[i] = c[4 - i] / c[4];
  double radius = 0.0;
  for (int i = 1; i <= 4; ++i) radius = fmax(radius, pow(fabs(m[i]), 1.0 / i));
  radius = 2.0 * radius + 1e-300;
  double zr[4], zi[4];
  for (int i = 0; i < 4; ++i) {
    double s, co;
    sincos(2.0 * M_PI * i / 4 + 0.35, &s, &co);
    zr[i] = 0.7 * radius * co;
    zi[i] = 0.7 * radius * s;
  }
  for (int it = 0; it < 60; ++it) {
    double moved = 0.0;
    for (int i = 0; i < 4; ++i) {
      double pr = m[0], pi = 0.0, dr = 0.0, di = 0.0;
      for (int j = 1; j <= 4; ++j) {
        const double ndr = dr * zr[i] - di * zi[i] + pr, ndi = dr * zi[i] + di * zr[i] + pi;
        const double npr = pr * zr[i] - pi * zi[i] + m[j], npi = pr * zi[i] + pi * zr[i];
        dr = ndr; di = ndi; pr = npr; pi = npi;
      }
      if (pr == 0.0 && pi == 0.0) continue;
      const double dn = dr * dr + di * di;
      const double rr = (pr * dr + pi * di) / dn, ri = (pi * dr - pr * di) / dn;  // p / p'
      double sr = 0.0, si = 0.0;
      for (int j = 0; j < 4; ++j) {
        if (j == i) continue;
        const double er = zr[i] - zr[j], ei = zi[i] - zi[j];
        const double en = er * er + ei * ei;
        sr += er / en;
        si -= ei / en;
      }
      const double qr = 1.0 - (rr * sr - ri * si), qi = -(rr * si + ri * sr);
      const double qn = qr * qr + qi * qi;
      const double stepr = (rr * qr + ri * qi) / qn, stepi = (ri * qr - rr * qi) / qn;
      zr[i] -= stepr;
      zi[i] -= stepi;
      moved = fmax(moved, (fabs(stepr) + fabs(stepi)) / (fabs(zr[i]) + fabs(zi[i]) + 1e-300));
    }
    if (moved < 1e-13) break;
  }
  for (int i = 0; i < 4; ++i) re[i] = zr[i];
}

// Real parts of the roots of c[0] + c[1] x + c[2] x^2 + c[3] x^3 + c[4] x^4 (c[4] != 0). Returns 4.
// `width` lanes starting at the caller's group base (mask `gmask`) call this together with identical arguments; with
// width >= 4 the four roots are polished by four lanes at once (lane gl polishes root gl & 3, the same arithmetic as
// the serial loop, gathered by shuffles); width == 1 = a lone thread (unit-test kernel).
__device__ __forceinline__ int quartic_real_parts(const double (&c)[5], double xlo, double xhi, double (&re)[4], int gl,
                                                  unsigned gmask, int width) {
  const double inv = 1.0 / c[4];
  const double a = c[3] * inv, b = c[2] * inv, cc = c[1] * inv, d = c[0] * inv;
  const double a2 = a * a;
  const double p = b - 0.375 * a2;
  const double q = cc - 0.5 * a * b + 0.125 * a2 * a;
  const double r = d - 0.25 * a * cc + 0.0625 * a2 * b - (3.0 / 256.0) * a2 * a2;
  double yr[4], yi[4];
  bool ok = true;
  if (q == 0.0) {
    // biquadratic: w^2 + p w + r = 0, y = +-sqrt(w)
    const double disc = p * p - 4.0 * r;
    double wr[2], wi[2];
    if (disc >= 0.0) {
      const double sq = sqrt(disc);
      wr[0] = 0.5 * (-p + sq); wr[1] = 0.5 * (-p - sq);
      wi[0] = wi[1] = 0.0;
    } else {
      wr[0] = wr[1] = -0.5 * p;
      wi[0] = 0.5 * sqrt(-disc); wi[1] = -wi[0];
    }
    for (int k = 0; k < 2; ++k) {  // principal complex square root
      const double mod = sqrt(wr[k] * wr[k] + wi[k] * wi[k]);
      const double sr = sqrt(fmax(0.5 * (mod + wr[k]), 0.0));
      double si = sqrt(fmax(0.5 * (mod - wr[k]), 0.0));
      if (wi[k] < 0.0) si = -si;
      yr[2 * k] = sr; yi[2 * k] = si;
      yr[2 * k + 1] = -sr; yi[2 * k + 1] = -si;
    }
  } else {
    // resolvent cubic z^3 + 2p z^2 + (p^2 - 4r) z - q^2 = 0: largest real root (positive)
    const double A = 2.0 * p, B = p * p - 4.0 * r, C = -q * q;
    const double Pd = B - A * A * (1.0 / 3.0);
    const double Qd = (2.0 / 27.0) * A * A * A - (1.0 / 3.0) * A * B + C;
    const double disc = 0.25 * Qd * Qd + (1.0 / 27.0) * Pd * Pd * Pd;
    double t;
    if (disc > 0.0) {
      const double sq = sqrt(disc);
      const double u = cbrt((-0.5 * Qd >= 0.0) ? (-0.5 * Qd + sq) : (-0.5 * Qd - sq));
      t = (u != 0.0) ? (u - Pd / (3.0 * u)) : 0.0;
    } else {
      const double mm = 2.0 * sqrt(fmax(-Pd * (1.0 / 3.0), 0.0));
      const double arg = (mm > 0.0) ? fmin(fmax(3.0 * Qd / (Pd * mm), -1.0), 1.0) : 0.0;
      t = mm * cos(acos(arg) * (1.0 / 3.0));
    }
    double z = t - A * (1.0 / 3.0);
    SMPC_UNROLL for (int it = 0; it < 3; ++it) {  // Newton polish on the resolvent
      const double f = ((z + A) * z + B) * z + C;
      const double fp = (3.0 * z + 2.0 * A) * z + B;
      if (fp != 0.0) z -= f / fp;
    }
    if (!(z > 0.0) || !isfinite(z)) ok = false;
    const double s = sqrt(fmax(z, 0.0));
    const double qs = (s > 0.0) ? q / s : 0.0;
    const double u = 0.5 * (p + z - qs), v = 0.5 * (p + z + qs);
    // y^2 + s y + u = 0 and y^2 - s y + v = 0
    const double d1 = s * s - 4.0 * u, d2 = s * s - 4.0 * v;
    if (d1 >= 0.0) {
      const double sq = sqrt(d1);
      yr[0] = 0.5 * (-s + sq); yr[1] = 0.5 * (-s - sq); yi[0] = yi[1] = 0.0;
    } else {
      yr[0] = yr[1] = -0.5 * s; yi[0] = 0.5 * sqrt(-d1); yi[1] = -yi[0];
    }
    if (d2 >= 0.0) {
      const double sq = sqrt(d2);
      yr[2] = 0.5 * (s + sq); yr[3] = 0.5 * (s - sq); yi[2] = yi[3] = 0.0;
    } else {
      yr[2] = yr[3] = 0.5 * s; yi[2] = 0.5 * sqrt(-d2); yi[3] = -yi[2];
    }
  }
  // back to x. Only roots whose real part can land in [xlo, xhi] matter to the caller: those get a complex
  // Newton polish on the monic quartic; the others only get a residual check (a wrong factorisation must not
  // hide an in-range root).
  const double shift = 0.25 * a;
  const double margin = 0.05 * (xhi - xlo) + 1e-3 * fabs(xhi);
  const double co[4] = {a, b, cc, d};
  // (inlined four times on purpose: the four Newton chains are independent and interleave in the leader lane; the
  // phase logic is on the critical path of the CTA's lock-step round, so its LATENCY matters, not its instruction count)
  auto polish = [&](double xr, double xi, double& out_re) -> bool {
    const bool near = (xr >= xlo - margin) && (xr <= xhi + margin);
    double res = 0.0;
    const int n_it = near ? 3 : 1;
    for (int it = 0; it < n_it; ++it) {
      double pr = 1.0, pi = 0.0, dr = 0.0, di = 0.0;  // p(x) and p'(x) by Horner, complex
      SMPC_UNROLL for (int j = 0; j < 4; ++j) {
        const double ndr = dr * xr - di * xi + pr, ndi = dr * xi + di * xr + pi;
        const double npr = pr * xr - pi * xi + co[j], npi = pr * xi + pi * xr;
        dr = ndr; di = ndi; pr = npr; pi = npi;
      }
      res = fabs(pr) + fabs(pi);
      if (it == n_it - 1) break;
      const double dn = dr * dr + di * di;
      if (dn > 0.0) {
        const double idn = 1.0 / dn;
        xr -= (pr * dr + pi * di) * idn;
        xi -= (pi * dr - pr * di) * idn;
      }
    }
    const double ax = fabs(xr) + fabs(xi);
    const double scale = fabs(d) + ax * (fabs(cc) + ax * (fabs(b) + ax * (fabs(a) + ax)));
    out_re = xr;
    return res <= (near ? 1e-10 : 1e-6) * scale + 1e-300;
  };
  if (width >= 4) {
    const int k = gl & 3;
    const double myr = (k == 0) ? yr[0] : (k == 1) ? yr[1] : (k == 2) ? yr[2] : yr[3];
    const double myi = (k == 0) ? yi[0] : (k == 1) ? yi[1] : (k == 2) ? yi[2] : yi[3];
    double mine;
    const bool mine_ok = polish(myr - shift, myi, mine);
    SMPC_UNROLL for (int kk = 0; kk < 4; ++kk) re[kk] = __shfl_sync(gmask, mine, kk, width);
    ok = __all_sync(gmask, ok && mine_ok);
  } else {
    SMPC_UNROLL for (int k = 0; k < 4; ++k) {
      if (!polish(yr[k] - shift, yi[k], re[k])) ok = false;
    }
  }
  if (!ok) quartic_aberth(c, re);
  return 4;
}

// Minimiser on [lo, hi] of the cubic through (0, f0, g0), (t, f1, g1).
static __device__ __noinline__ double cubic_interp_min(double f0, double g0, double t, double f1, double g1, double lo,
                                                   double hi) {
  const double A = f1 - f0 - g0 * t, Bv = g1 - g0;
  const double inv_t = 1.0 / t;
  const double a = (Bv * t - 2.0 * A) * inv_t * inv_t * inv_t;
  const double b = (3.0 * A - Bv * t) * inv_t * inv_t;
  auto pv = [&](double x) { return f0 + x * (g0 + x * (b + x * a)); };
  double ox = (lo + hi) / 2.0, ov = pv(ox);
  const double vlo = pv(lo);
  if (vlo < ov) { ov = vlo; ox = lo; }
  const double vhi = pv(hi);
  if (vhi < ov) { ov = vhi; ox = hi; }
  // critical points: roots of 3a x^2 + 2b x + g0 (leading zeros removed as Ceres does)
  const double qa = 3.0 * a, qb = 2.0 * b, qc = g0;
  double r0 = NAN, r1 = NAN;
  if (qa != 0.0) {
    const double D = qb * qb - 4.0 * qa * qc;
    const double sD = sqrt(fabs(D));
    if (D >= 0.0) {
      if (qb >= 0.0) {
        r0 = (-qb - sD) / (2.0 * qa);
        r1 = (2.0 * qc) / (-qb - sD);
      } else {
        r0 = (2.0 * qc) / (-qb + sD);
        r1 = (-qb + sD) / (2.0 * qa);
      }
    } else {
      r0 = r1 = -qb / (2.0 * qa);
    }
  } else if (qb != 0.0) {
    r0 = -qc / qb;
  }
  if (r0 >= lo && r0 <= hi) {
    const double v = pv(r0);
    if (v < ov) { ov = v; ox = r0; }
  }
  if (r1 >= lo && r1 <= hi) {
    const double v = pv(r1);
    if (v < ov) { ov = v; ox = r1; }
  }
  return ox;
}

// Minimiser on [lo, hi] of the quintic through (0, f0, g0), (t1, f1, g1), (t2, f2, g2), 0 < t1 < t2.
static __device__ __noinline__ double quintic_interp_min(double f0, double g0, double t1, double f1, double g1, double t2,
                                                        double f2, double g2, double lo, double hi, int gl, unsigned gmask,
                                                        int width) {
  // work in xi = x / t2: nodes 0, tau, 1 (Hermite divided differences), then expand to monomials
  const double tau = t1 / t2;
  const double d0 = g0 * t2, d1 = g1 * t2, d2 = g2 * t2;
  const double inv_tau = 1.0 / tau, inv_om = 1.0 / (1.0 - tau);
  const double e01 = (f1 - f0) * inv_tau, e12 = (f2 - f1) * inv_om;
  const double s0 = (e01 - d0) * inv_tau, s1 = (d1 - e01) * inv_tau, s2 = (e12 - d1) * inv_om, s3 = (d2 - e12) * inv_om;
  const double h0 = (s1 - s0) * inv_tau, h1 = (s2 - s1), h2 = (s3 - s2) * inv_om;
  const double k0 = h1 - h0, k1 = h2 - h1;
  const double c5 = k1 - k0;
  const double c0 = f0, c1 = d0, c2 = s0, c3 = h0, c4 = k0;
  const double tau2 = tau * tau;
  double m[6];
  m[5] = c5;
  m[4] = c4 - (2.0 * tau + 1.0) * c5;
  m[3] = c3 - 2.0 * tau * c4 + (tau2 + 2.0 * tau) * c5;
  m[2] = c2 - tau * c3 + tau2 * c4 - tau2 * c5;
  m[1] = c1;
  m[0] = c0;
  const double xlo = lo / t2, xhi = hi / t2;
  double ox = (xlo + xhi) / 2.0, ov = horner5(m, ox);
  const double vlo = horner5(m, xlo);
  if (vlo < ov) { ov = vlo; ox = xlo; }
  const double vhi = horner5(m, xhi);
  if (vhi < ov) { ov = vhi; ox = xhi; }
  const double dq[5] = {m[1], 2.0 * m[2], 3.0 * m[3], 4.0 * m[4], 5.0 * m[5]};
  double roots[4];
  int nr = 0;
  if (dq[4] != 0.0) {
    nr = quartic_real_parts(dq, xlo, xhi, roots, gl, gmask, width);
  } else if (dq[3] != 0.0) {
    // exactly-zero leading coefficient (never seen on real data): x * cubic has the cubic's roots plus 0,
    // and 0 lies outside [xlo, xhi]
    const double dq2[5] = {0.0, dq[0], dq[1], dq[2], dq[3]};
    quartic_aberth(dq2, roots);
    nr = 4;
  } else if (dq[2] != 0.0) {
    const double dq2[5] = {0.0, 0.0, dq[0], dq[1], dq[2]};
    quartic_aberth(dq2, roots);
    nr = 4;
  } else if (dq[1] != 0.0) {
    roots[0] = -dq[0] / dq[1];
    nr = 1;
  }
  for (int i = 0; i < nr; ++i) {
    if (roots[i] >= xlo && roots[i] <= xhi) {
      const double v = horner5(m, roots[i]);
      if (v < ov) { ov = v; ox = roots[i]; }
    }
  }
  return ox * t2;
}

// Box projection of ParameterBlock::Plus: only the first n_bounded blocks carry bounds
// (reference src/optimizer.cpp:373-379: v in [0, 0.6], w in [-1.4, 1.4]; SURVEY Q2, Q9).
// Omnidirectional blocks (extension): the lateral velocity is bounded by the same speed, vy in [-0.6, 0.6].
template <int D>
__device__ __forceinline__ double project_param(double v, int c, int n_bounded) {
  if ((c / D) < n_bounded) {
    const int k = c % D;
    const double hi = (k == D - 1) ? 1.4 : 0.6;
    const double lo = (k == D - 1) ? -1.4 : ((k == 0) ? 0.0 : -0.6);
    return std_min(std_max(v, lo), hi);  // SetParameterLowerBound / UpperBound projection of Ceres' Plus
  }
  return v;
}

enum Termination {
  kConvGradient = 0,
  kConvParameter = 1,
  kConvFunction = 2,
  kConvRadius = 3,
  kNoConvergence = 4,
  kFailInvalidSteps = 5,
  kFailEvaluation = 6
};

// Host-buffer pipeline: the per-problem costmaps stream in on a second stream WHILE the solve kernel runs. Problems are
// handed out in index order, so a group only has to wait until the arrival counter has passed its problem. The copy
// engine needs no SM, so the wait cannot deadlock; it still gives up after 2 s and reports through arrival[1].
__device__ __forceinline__ void wait_for_costmap(unsigned* arrival, int b) {
  unsigned long long t0 = 0;
  for (;;) {
    unsigned seen;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(seen) : "l"(arrival) : "memory");
    if (seen > (unsigned)b) return;
    unsigned gave_up;
    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(gave_up) : "l"(arrival + 1) : "memory");
    if (gave_up) return;  // another group already timed out: the call fails, do not wait again
    unsigned long long now;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
    if (t0 == 0) t0 = now;
    if (now - t0 > 2000000000ull) {
      atomicExch(arrival + 1, 1u);
      return;
    }
    __nanosleep(200);
  }
}

// Load the group-uniform problem view. NC = the inputs are read-only for the whole kernel (see bicubic).
template <bool NC>
__device__ __forceinline__ void load_problem(const DevParams& prm, const DevBatch& bt, int b, Prob& pb) {
  const int S1 = bt.S + 1;
  if (bt.scenario) b = ld_in<NC>(bt.scenario + b);  // row of the per-scene arrays; u0 and the outputs stay per problem
  const int Sb = bt.n_steps_each ? min(max(__ldg(bt.n_steps_each + b), 1), bt.S) : bt.S;
  pb.S = Sb;
  pb.ch = min(prm.control_horizon, Sb);   // src/optimizer.cpp:248
  pb.bl = min(prm.block_length, pb.ch);   // src/optimizer.cpp:249
  pb.nb = (pb.ch + pb.bl - 1) / pb.bl;
  pb.nbd = pb.ch / pb.bl;
  pb.x0 = ld_in<NC>(bt.pose0 + 3 * (size_t)b);
  pb.y0 = ld_in<NC>(bt.pose0 + 3 * (size_t)b + 1);
  pb.yaw0 = ld_in<NC>(bt.pose0 + 3 * (size_t)b + 2);
  pb.goal_yaw = ld_in<NC>(bt.goal_yaw + b);
  pb.px = bt.path_xy + (size_t)b * 2 * S1;
  pb.py = pb.px + S1;
  pb.fin_x = ld_in<NC>(pb.px + Sb);
  pb.fin_y = ld_in<NC>(pb.py + Sb);
  pb.agents = (bt.A > 0 && bt.agents) ? bt.agents + (size_t)b * bt.A * 6 * S1 : nullptr;
  pb.packed = pb.agents ? bt.agents_packed + (size_t)b * bt.A * S1 * 4 : nullptr;
  pb.valid = pb.agents ? bt.agents_valid + (size_t)b * bt.A * S1 : nullptr;
  pb.has_people = (bt.has_people != nullptr) && (bt.has_people[b] != 0);
  const int mi = bt.costmap_index ? ld_in<NC>(bt.costmap_index + b) : (b % bt.M);
  pb.map = bt.costmaps + (size_t)mi * bt.size_x * bt.size_y;
  pb.org_x = ld_in<NC>(bt.costmap_origin + 2 * mi);
  pb.org_y = ld_in<NC>(bt.costmap_origin + 2 * mi + 1);
}

// Agent-angle steering targets of every step -> group shared memory (once per problem).
template <int NB, int G, bool PPL, int D = 2, bool WT = false>
__device__ __forceinline__ void agent_angle_setup(const DevBatch& bt, const Prob& pb, int lane, double* ws) {
  using L = Layout<NB, D, WT>;
  const int gl = lane & (G - 1);
  if (gl == 0) {
    double s0, c0;
    sincos(pb.yaw0, &s0, &c0);
    ws[L::kYaw] = s0;
    ws[L::kYaw + 1] = c0;
  }
  if (PPL) {
    for (int j = gl; j < pb.S; j += G) {
      double tgt = NAN;
      if (pb.has_people && bt.A > 0 && pb.agents != nullptr) tgt = agent_angle_target(bt, pb, j + 1);
      ws[L::kAa + j] = tgt;
    }
  }
}

// Post-solve expansion (reference src/optimizer.cpp:390-446): cmds[S+1] hold block min(i/bl, nb-1) for i < ch
// and the last block afterwards; the path is the Euler rollout of those cmds from pose0 (pose0 excluded).
template <int NB, int G, int D = 2>
__device__ __forceinline__ void expand_outputs(const DevBatch& bt, const DevResult& rs, const Prob& pb, int b,
                                               const double (&x)[D * NB], int lane) {
  const int gl = lane & (G - 1);
  const unsigned gmask = Group<G>::mask(lane);
  const int S = pb.S, S1 = bt.S + 1, last_b = pb.nb - 1;
  double s0, c0;
  sincos(pb.yaw0 * 0.5, &s0, &c0);
  const double yaw_rt = atan2(2.0 * (c0 * s0), c0 * c0 - s0 * s0);  // evolving_poses[0] went through setRPY/getYaw
  double carry_x = pb.x0, carry_y = pb.y0;
  for (int base = 0; base <= S; base += G) {
    const int i = base + gl;
    const bool act = i <= S;
    const int bi = (i < pb.ch) ? min(i / pb.bl, last_b) : last_b;
    double v = x[0], w = x[D - 1], vy = 0.0;
    double th = yaw_rt, th_next = yaw_rt;
    SMPC_UNROLL for (int bb = 0; bb < NB; ++bb) {
      if (bb == bi) {
        v = x[D * bb];
        w = x[D * bb + D - 1];
        if (D == 3) vy = x[D * bb + 1];
      }
      th += x[D * bb + D - 1] * (bt.dt * (double)steps_in_block_before(i, bb, pb.bl, last_b));
      th_next += x[D * bb + D - 1] * (bt.dt * (double)steps_in_block_before(i + 1, bb, pb.bl, last_b));
    }
    if (act && rs.cmds) {  // cmds [B][S+1][D]: (v, w) or (vx, vy, w)
      rs.cmds[((size_t)b * S1 + i) * D] = v;
      if (D == 3) rs.cmds[((size_t)b * S1 + i) * D + 1] = vy;
      rs.cmds[((size_t)b * S1 + i) * D + D - 1] = w;
    }
    if (rs.path) {
      double sn, cs;
      sincos(th, &sn, &cs);
      double sx = act ? v * cs * bt.dt : 0.0, sy = act ? v * sn * bt.dt : 0.0;
      if (D == 3 && act) {
        sx = (v * cs - vy * sn) * bt.dt;
        sy = (v * sn + vy * cs) * bt.dt;
      }
      SMPC_UNROLL for (int d = 1; d < G; d <<= 1) {
        const double tx = __shfl_up_sync(gmask, sx, d, G), ty = __shfl_up_sync(gmask, sy, d, G);
        if (gl >= d) {
          sx += tx;
          sy += ty;
        }
      }
      const double X = carry_x + sx, Y = carry_y + sy;
      carry_x = __shfl_sync(gmask, X, G - 1, G);
      carry_y = __shfl_sync(gmask, Y, G - 1, G);
      if (act) {
        double sh, chh;
        sincos(th_next * 0.5, &sh, &chh);
        double* o = rs.path + ((size_t)b * S1 + i) * 3;
        o[0] = X;
        o[1] = Y;
        o[2] = atan2(2.0 * (chh * sh), chh * chh - sh * sh);  // tf2 setRPY -> getYaw (SURVEY Q14)
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// ceres::Solve restated (SURVEY Appendix A) as a per-group state machine around ONE evaluation site.
// Every trial point (iteration zero, each line-search sample, the un-shortened step after a failed line search)
// is evaluated once: an accepted point needs no second pass — its plain cost is the candidate cost, its
// differentiated cost the next iterate's cost and its J^T J / J^T r the next iterate's normal equations. Groups of a
// warp run different problems in different phases; they meet at the evaluation (warp-convergent) and diverge only in
// the scalar phase logic, which the group's first lane runs alone. A group that finishes its problem writes the
// results and pulls the next problem from the atomic queue.
// ---------------------------------------------------------------------------------------------------

// Claim the next parked problem (lane 0 of a group that has seen the main queue empty). Parks in flight are counted
// in park_counters[2] (raised BEFORE the parker tries to fetch its fresh problem, lowered after it has published or
// failed to fetch), so "main queue empty and nothing in flight" means the published count can no longer change: from
// then on a plain atomicAdd hands out the slots (no compare-and-swap storm when thousands of groups go idle at once)
// and a ticket beyond the final count means the queue is closed for good.
// Returns the problem id, -1 = parks still in flight (ask again next iteration), -2 = closed and empty.
__device__ __forceinline__ int park_pop(const DevBatch& bt) {
  volatile int* cnt = bt.park_counters;
  if (cnt[2] != 0) return -1;
  __threadfence();
  const int tail = cnt[0];
  const int h = atomicAdd(bt.park_counters + 1, 1);
  if (h >= tail) return -2;
  const int id = atomicAdd(bt.park_ring + h, 0);
  __threadfence();
  return id;
}

// One trace row (include/smpc.h smpc_result.trace), written by the group leader when tracing is on.
__device__ __forceinline__ void trace_row(const DevResult& rs, int b, int row, double iteration, double phase, double t,
                                          double cost_diff, double cost_plain, double aux, double code, double radius) {
  if (rs.trace == nullptr || row < 0 || row >= rs.trace_rows) return;
  double* o = rs.trace + ((size_t)b * rs.trace_rows + row) * 8;
  o[0] = iteration; o[1] = phase; o[2] = t; o[3] = cost_diff;
  o[4] = cost_plain; o[5] = aux; o[6] = code; o[7] = radius;
}

template <int NB, int G, bool PPL, int D = 2, bool WT = false>
__device__ __forceinline__ void solve_loop(const DevParams& prm, const DevBatch& bt, const DevResult& rs, int* queue,
                                           double* ws, double* red, int lane) {
  using L = Layout<NB, D, WT>;
  constexpr int P = L::P;
  const int gl = lane & (G - 1);
  const unsigned gmask = Group<G>::mask(lane);
  // every piece of group state is addressed as ws + constant so that only `ws` stays live across the evaluation
#define xs (ws + L::kX)
#define best (ws + L::kBest)
#define scale (ws + L::kScale)
#define diag (ws + L::kDiag)
#define delta (ws + L::kDelta)
#define cand (ws + L::kCand)
#define gs (reinterpret_cast<LmState*>(ws + L::kState))
#define pbs (reinterpret_cast<Prob*>(ws + L::kProb))

  if (gl == 0) {
    gs->phase = kFetch;
    gs->flags = 0;
    gs->b = -1;
    gs->n_eval = 0;
  }
  __syncwarp(gmask);

  unsigned loop_count = 0;
  for (;;) {
    // ---- work acquisition. An idle group takes the next fresh problem, else (time slicing) the next parked one. A
    //      group whose live problem reaches a quantum boundary while fresh problems are still waiting parks it and
    //      takes a fresh one: long solves no longer start late behind short ones (the tail of a few-wave batch).
    const int fl0 = gs->flags;
    const bool slicing = !PPL && bt.park_state != nullptr;  // people kernels: compiled out (register budget)
    const bool idle = gs->phase == kFetch;
    const bool at_quantum = slicing && !idle && (fl0 & kLive) && !(fl0 & kDrained) && gs->n_eval > 0 &&
                            (gs->n_eval % bt.park_quantum) == 0;
    __syncwarp(gmask);  // every lane has read the state words the leader rewrites below
    if ((idle && !(fl0 & kClosed) && (slicing || !(fl0 & kExhausted))) || at_quantum) {
      int nb_ = bt.B, resume = -2;
      if (gl == 0) {
        if (at_quantum) {  // announce the park before trying to fetch (see park_pop)
          atomicAdd(bt.park_counters + 2, 1);
          __threadfence();
        }
        if (!(fl0 & kDrained)) nb_ = atomicAdd(queue, 1);
        if (at_quantum && nb_ >= bt.B) atomicSub(bt.park_counters + 2, 1);
        if (nb_ >= bt.B && idle && slicing) {
          __threadfence();
          resume = park_pop(bt);
        }
      }
      nb_ = __shfl_sync(gmask, nb_, 0, G);
      resume = __shfl_sync(gmask, resume, 0, G);
      __syncwarp(gmask);
      const int stride = L::total(bt.S);
      if (nb_ >= bt.B && resume >= 0) {
        // resume a parked problem: its whole group state comes back from L2 (never through a stale L1 line)
        const double* src = bt.park_state + (size_t)resume * stride;
        for (int i = gl; i < stride; i += G) ws[i] = __ldcg(src + i);
        __syncwarp(gmask);
        if (gl == 0) gs->flags |= kDrained;
      } else if (nb_ >= bt.B) {
        if (gl == 0)
          gs->flags = idle ? (kExhausted | kDrained | ((resume == -2) ? kClosed : 0)) : (fl0 | kDrained);
      } else {
        if (at_quantum) {  // park the live problem: state -> global, then publish its id
          const int self = gs->b;
          double* dst = bt.park_state + (size_t)self * stride;
          for (int i = gl; i < stride; i += G) dst[i] = ws[i];
          __threadfence();
          __syncwarp(gmask);
          if (gl == 0) {
            atomicExch(bt.park_ring + atomicAdd(bt.park_counters, 1), self);
            __threadfence();
            atomicSub(bt.park_counters + 2, 1);
          }
          __syncwarp(gmask);
        }
        if (gl == 0) {
          if (!PPL && bt.arrival != nullptr) wait_for_costmap(bt.arrival, nb_);
          load_problem<PPL>(prm, bt, nb_, *pbs);
          if (WT) {  // the problem's critic weights: row weight_set[b] of the batch's table
            const double* row = bt.weights + 9 * (size_t)ld_in<PPL>(bt.weight_set + nb_);
            SMPC_UNROLL for (int k = 0; k < 9; ++k) ws[L::kWt + k] = ld_in<PPL>(row + k);
          }
        }
        __syncwarp(gmask);
        agent_angle_setup<NB, G, PPL, D, WT>(bt, *pbs, lane, ws);
        if (gl == 0) {
          // IterationZero: project the start point onto the box. Blocks the problem does not use (shorter horizon than
          // the batch's) stay exactly zero: no residual touches them, so their rows of J^T J and J^T r are zero, the LM
          // diagonal keeps their pivot positive and their step is exactly zero.
          const int Pb = D * pbs->nb, nbd = pbs->nbd;
          for (int c = 0; c < P; ++c) {
            const double v = (c < Pb) ? ld_in<PPL>(bt.u0 + (size_t)nb_ * P + c) : 0.0;
            xs[c] = v;
            best[c] = v;
            cand[c] = project_param<D>(v, c, nbd);
          }
          LmState z;
          z.x_cost = z.x_norm = z.gmax = 0.0;
          z.radius = 1e4;
          z.decrease_factor = 2.0;
          z.minimum_cost = DBL_MAX;
          z.it_cost = z.cost_initial = z.cost_final = z.model_cost_change = z.g0 = z.dmax = 0.0;
          z.t = 1.0;
          z.prev_x = z.prev_value = z.prev_gradient = 0.0;
          z.se_cost = 0.0;
          z.iteration = z.n_invalid = z.n_eval = z.n_light = z.ls_iters = 0;
          z.term = kNoConvergence;
          z.phase = kInit;
          z.b = nb_;
          z.flags = kLive | kItSuccessful;
          z.pad_ = 0;
          *gs = z;
        }
      }
      __syncwarp(gmask);
    }
    // CTA barrier per evaluation: the warps of a CTA walk the large unrolled evaluation code together and share its
    // instruction-cache lines (measured +15..40 %); it also ends the loop once every group of the CTA is out of work
    // (a barrier every 2nd / 3rd / 4th evaluation measured -8 / -17 / -20 %: SMPC_SYNC_EVERY stays 1; two / three
    // independent lock-step teams per CTA on named barriers, so that one team's single-lane phase logic could run under
    // another team's FP64-bound evaluation, measured -3 / -6 % with 20 agents and -4 / -8 % without people)
#ifndef SMPC_SYNC_EVERY
#define SMPC_SYNC_EVERY 1
#endif
    if (bt.cta_sync) {
      if ((loop_count++ % SMPC_SYNC_EVERY) == 0) {
        if (__syncthreads_and((gs->flags & kExhausted) != 0)) break;
      }
    } else if (__all_sync(kFullMask, (gs->flags & kExhausted) != 0)) {
      break;
    }

    const bool live = (gs->flags & kLive) != 0;
    const unsigned fl = evaluate<NB, G, PPL, D, WT>(prm, bt, *pbs, live, ws, red, cand, lane,
                                             ws + ((gs->flags & kSwapped) ? L::kBuf0 : L::kBuf1), gs);

    // ---- phase logic: the group's first lane alone, on the group's shared-memory state -----------------------
    if (gl == 0 && live) {
      LmState& st = *gs;
      const int nbd = pbs->nbd;
      double* cur = ws + ((st.flags & kSwapped) ? L::kBuf1 : L::kBuf0);    // normal equations at x
      double* trial = ws + ((st.flags & kSwapped) ? L::kBuf0 : L::kBuf1);  // normal equations at the trial point
      const double t_cost = trial[0];        // cost of the differentiated evaluation (line search, next x_cost)
      const double t_cost_plain = trial[1];  // cost of the plain evaluation (candidate cost)
      const bool eval_ok = (fl & (kResidualBad | kJacobianBad)) == 0;
      bool take_step = false;    // proceed to accept/reject with `cand`
      bool finished = false;     // the solve of this problem has terminated
      bool next_sample = false;  // another trial point has been set up in `cand`
      const int row = st.n_eval;  // trace row of this evaluation
      const double tr_iter = (double)st.iteration, tr_phase = (double)st.phase, tr_t = (st.phase == kInit) ? 0.0 : st.t;
      double tr_aux = NAN, tr_code = 0.0;
      ++st.n_eval;
      if (fl & kNoHessian) ++st.n_light;

      // ===== part A: classify the evaluated point (init / line-search sample / full step), accept or reject
      if (st.phase == kInit) {
        st.cost_initial = st.cost_final = t_cost;
        if (!eval_ok) {
          st.term = kFailEvaluation;
          finished = true;
        } else {
          // x <- projected seed; cur <- trial; Jacobi scaling from the column norms (= sqrt of diag(J^T J))
          for (int c = 0; c < P; ++c) {
            xs[c] = cand[c];
            scale[c] = 1.0 / (1.0 + sqrt(trial[L::h(c, c)]));
          }
          st.flags ^= kSwapped;
          { double* tmp = cur; cur = trial; trial = tmp; }
          st.x_cost = t_cost;
          st.se_cost = t_cost;
          st.it_cost = t_cost;
          st.flags |= kItSuccessful;
        }
      } else if (st.phase == kLineSearch) {
        // Armijo sufficient decrease at step t along delta (projected); the evaluation has already tested it
        // (kNoHessian <=> rejected), so both sides use one and the same comparison
        if (!(fl & kNoHessian)) {
          take_step = true;  // success: delta <- t * delta, candidate = this trial point
          tr_code = 1.0;
        } else {
          tr_aux = t_cost - (st.x_cost + 1e-4 * st.g0 * st.t);
          double gd = 0.0;
          for (int c = 0; c < P; ++c) gd += delta[c] * trial[L::g(c)];
          ++st.ls_iters;
          bool ls_failed = st.ls_iters >= 20;
          double t_new = st.t;
          if (!ls_failed) {
            const double lo = 1e-3 * st.t, hi = 0.6 * st.t;
            if (!eval_ok) {
              t_new = std_min(std_max(st.t * 0.5, lo), hi);
            } else if (st.flags & kPrevOk) {
              t_new = quintic_interp_min(st.x_cost, st.g0, st.t, t_cost, gd, st.prev_x, st.prev_value, st.prev_gradient,
                                         lo, hi, 0, 0u, 1);
            } else {
              t_new = cubic_interp_min(st.x_cost, st.g0, st.t, t_cost, gd, lo, hi);
            }
            if (t_new * st.dmax < 1e-9) ls_failed = true;
          }
          if (!ls_failed) {
            st.prev_x = st.t;
            st.prev_value = t_cost;
            st.prev_gradient = gd;
            st.flags = eval_ok ? (st.flags | kPrevOk) : (st.flags & ~kPrevOk);
            st.t = t_new;
            for (int c = 0; c < P; ++c) cand[c] = project_param<D>(xs[c] + t_new * delta[c], c, nbd);
            next_sample = true;  // evaluate the next line-search sample
          } else {
            // line search failed: the un-shortened TR step Plus(x, delta) is the candidate (delta unchanged). It needs
            // a full evaluation — also when t is still 1 and this very point was just sampled without its J^T J.
            st.t = 1.0;
            for (int c = 0; c < P; ++c) cand[c] = project_param<D>(xs[c] + delta[c], c, nbd);
            st.phase = kFullStep;
            next_sample = true;
          }
        }
      } else {  // kFullStep: evaluation of Plus(x, delta) after a failed line search
        take_step = true;
      }

      if (take_step) {
        tr_code += 2.0;
        const double cand_cost = (fl & kResidualBad) ? DBL_MAX : t_cost_plain;
        const bool tol_armed = (prm.ceres_compat < 210) || (st.flags & kAnySuccess);
        double step_norm = 0.0;
        for (int c = 0; c < P; ++c) {
          const double dd = xs[c] - cand[c];
          step_norm += dd * dd;
        }
        step_norm = sqrt(step_norm);
        const double cost_change = st.x_cost - cand_cost;
        if (tol_armed && step_norm <= prm.param_tol * (st.x_norm + prm.param_tol)) {
          tr_aux = step_norm / (prm.param_tol * (st.x_norm + prm.param_tol)) - 1.0;
          --st.iteration;
          st.term = kConvParameter;
          finished = true;
        } else if (tol_armed && fabs(cost_change) <= prm.fn_tol * st.x_cost) {
          tr_aux = fabs(cost_change) - prm.fn_tol * st.x_cost;
          --st.iteration;
          st.term = kConvFunction;
          finished = true;
        } else {
          // TrustRegionStepEvaluator::StepQuality (monotonic steps): measured from the step evaluator's current cost
          const double rho = (cand_cost >= DBL_MAX) ? -DBL_MAX : (st.se_cost - cand_cost) / st.model_cost_change;
          tr_aux = rho;
          if (rho > 1e-3) {  // HandleSuccessfulStep
            if (fl & kJacobianBad) {
              --st.iteration;
              st.term = kFailEvaluation;
              finished = true;
            } else {
              tr_code += 4.0;
              for (int c = 0; c < P; ++c) xs[c] = cand[c];
              st.flags ^= kSwapped;
              { double* tmp = cur; cur = trial; trial = tmp; }
              st.x_cost = t_cost;
              st.se_cost = cand_cost;
              st.flags |= kAnySuccess | kItSuccessful;
              st.flags &= ~kReuseDiagonal;
              st.it_cost = t_cost;
              const double qq = 2.0 * rho - 1.0;
              st.radius = std_min(1e16, st.radius / std_max(1.0 / 3.0, 1.0 - qq * qq * qq));
              st.decrease_factor = 2.0;
            }
          } else {
            st.flags &= ~kItSuccessful;
            st.flags |= kReuseDiagonal;
            st.it_cost = cand_cost;
            st.radius = st.radius / st.decrease_factor;
            st.decrease_factor *= 2.0;
          }
        }
      }

      // ===== part B: a new outer iteration starts here (after iteration zero or after accept / reject)
      if (!finished && !next_sample) {
        if (st.flags & kItSuccessful) {  // x changed: refresh |x| and the projected-gradient max norm
          double xn = 0.0, gm = 0.0;
          for (int c = 0; c < P; ++c) {
            const double xv = xs[c];
            xn += xv * xv;
            gm = std_max(gm, fabs(xv - project_param<D>(xv - cur[L::g(c)], c, nbd)));
          }
          st.x_norm = sqrt(xn);
          st.gmax = gm;
        }
        for (;;) {
          // FinalizeIterationAndCheckIfMinimizerCanContinue
          if ((st.flags & kItSuccessful) && st.x_cost < st.minimum_cost) {
            st.minimum_cost = st.x_cost;
            for (int c = 0; c < P; ++c) best[c] = xs[c];
          }
          st.cost_final = std_min(st.cost_final, st.it_cost);
          if (prm.max_evaluations > 0 && st.n_eval >= prm.max_evaluations) { st.term = kNoConvergence; finished = true; break; }
          if (st.iteration >= prm.max_iterations) { st.term = kNoConvergence; finished = true; break; }
          if ((st.flags & kItSuccessful) && st.gmax <= prm.gradient_tol) { st.term = kConvGradient; finished = true; break; }
          if (st.radius <= 1e-32) { st.term = kConvRadius; finished = true; break; }
          ++st.iteration;

          // LevenbergMarquardtStrategy::ComputeStep on the column-scaled normal equations
          if (!(st.flags & kReuseDiagonal)) {
            for (int c = 0; c < P; ++c) {
              const double scv = scale[c];
              diag[c] = std_min(std_max(scv * scv * cur[L::h(c, c)], 1e-6), 1e32);
            }
          }
          st.flags |= kReuseDiagonal;
          double sc[P], Lc[L::NH], step[P];
          const double inv_radius = 1.0 / st.radius;
          SMPC_UNROLL for (int c = 0; c < P; ++c) sc[c] = scale[c];
          SMPC_UNROLL for (int a = 0; a < P; ++a) {
            SMPC_UNROLL for (int bq = 0; bq <= a; ++bq) Lc[a * (a + 1) / 2 + bq] = sc[a] * sc[bq] * cur[L::h(a, bq)];
            Lc[a * (a + 1) / 2 + a] += diag[a] * inv_radius;  // (sqrt(diag / radius))^2 of the LM strategy
          }
          bool step_ok = true;
          SMPC_UNROLL for (int jc = 0; jc < P; ++jc) {  // Cholesky, in place, lower triangle
            double d = Lc[jc * (jc + 1) / 2 + jc];
            SMPC_UNROLL for (int k = 0; k < jc; ++k) d -= Lc[jc * (jc + 1) / 2 + k] * Lc[jc * (jc + 1) / 2 + k];
            if (!(d > 0.0)) step_ok = false;
            const double inv_d = rsqrt(d);
            Lc[jc * (jc + 1) / 2 + jc] = inv_d;  // store 1/L_jj
            SMPC_UNROLL for (int i = jc + 1; i < P; ++i) {
              double sacc = Lc[i * (i + 1) / 2 + jc];
              SMPC_UNROLL for (int k = 0; k < jc; ++k) sacc -= Lc[i * (i + 1) / 2 + k] * Lc[jc * (jc + 1) / 2 + k];
              Lc[i * (i + 1) / 2 + jc] = sacc * inv_d;
            }
          }
          SMPC_UNROLL for (int i = 0; i < P; ++i) {  // forward substitution
            double sacc = sc[i] * cur[L::g(i)];
            SMPC_UNROLL for (int k = 0; k < i; ++k) sacc -= Lc[i * (i + 1) / 2 + k] * step[k];
            step[i] = sacc * Lc[i * (i + 1) / 2 + i];
          }
          SMPC_UNROLL for (int i = P - 1; i >= 0; --i) {  // back substitution
            double sacc = step[i];
            SMPC_UNROLL for (int k = i + 1; k < P; ++k) sacc -= Lc[k * (k + 1) / 2 + i] * step[k];
            step[i] = sacc * Lc[i * (i + 1) / 2 + i];
          }
          SMPC_UNROLL for (int c = 0; c < P; ++c) {
            step_ok = step_ok && isfinite(step[c]);
            step[c] = -step[c];
          }
          // model_cost_change = -(Js s)'(r + Js s / 2) = -s'(Js' r) - s'(Js' Js) s / 2
          double lin = 0.0, quad = 0.0;
          SMPC_UNROLL for (int a = 0; a < P; ++a) {
            const double sa = sc[a] * step[a];
            lin += sa * cur[L::g(a)];
            double rowv = 0.0;
            SMPC_UNROLL for (int bq = 0; bq < a; ++bq) rowv += cur[L::h(a, bq)] * (sc[bq] * step[bq]);
            quad += sa * (2.0 * rowv + cur[L::h(a, a)] * sa);
          }
          st.model_cost_change = -lin - 0.5 * quad;
          const bool valid = step_ok && (st.model_cost_change > 0.0);
          if (valid) {
            st.n_invalid = 0;
            double g0 = 0.0, dmax = 0.0;
            SMPC_UNROLL for (int c = 0; c < P; ++c) {
              const double dl = step[c] * sc[c];
              g0 += cur[L::g(c)] * dl;
              dmax = std_max(dmax, fabs(dl));
              delta[c] = dl;
              cand[c] = project_param<D>(xs[c] + dl, c, nbd);
            }
            st.g0 = g0;
            st.dmax = dmax;
            break;
          }
          // HandleInvalidStep
          if (++st.n_invalid >= 5) {
            --st.iteration;
            st.term = kFailInvalidSteps;
            finished = true;
            break;
          }
          st.radius /= st.decrease_factor;
          st.decrease_factor *= 2.0;
          st.flags &= ~kItSuccessful;
          st.it_cost = st.x_cost;
        }
        if (!finished) {
          st.phase = kLineSearch;
          st.t = 1.0;
          st.ls_iters = 0;
          st.flags &= ~kPrevOk;
        }
      }
      if (finished) {
        st.flags |= kFinished;
        tr_code += 8.0 + 16.0 * (double)st.term;
      }
      if (rs.trace != nullptr)
        trace_row(rs, st.b, row, tr_iter, tr_phase, tr_t, t_cost, take_step ? t_cost_plain : NAN, tr_aux, tr_code, st.radius);
    }
    __syncwarp(gmask);

    if (live && (gs->flags & kFinished)) {
      // results. Solution = best accepted iterate when usable (Solver::Summary::IsSolutionUsable), else the seed.
      const LmState& st = *gs;
      const bool usable = st.term <= kNoConvergence;
      const int b = st.b;
      const int Pb = D * pbs->nb;
      double x[P];
      SMPC_UNROLL for (int c = 0; c < P; ++c)
        x[c] = (c < Pb) ? (usable ? best[c] : ld_in<PPL>(bt.u0 + (size_t)b * P + c)) : 0.0;
      if (gl == 0) {
        if (rs.u) {
          SMPC_UNROLL for (int c = 0; c < P; ++c)
            if (c < Pb) rs.u[(size_t)b * P + c] = x[c];
        }
        if (rs.cost_initial) rs.cost_initial[b] = st.cost_initial;
        if (rs.cost_final) rs.cost_final[b] = st.cost_final;
        if (rs.iterations) rs.iterations[b] = st.iteration;
        if (rs.termination) rs.termination[b] = st.term;
        if (rs.usable) rs.usable[b] = usable ? 1 : 0;
        if (rs.n_evals) {
          rs.n_evals[2 * b] = st.n_eval - st.n_light;
          rs.n_evals[2 * b + 1] = st.n_light;
        }
      }
      if (rs.cmds || rs.path) expand_outputs<NB, G, D>(bt, rs, *pbs, b, x, lane);
      __syncwarp(gmask);
      if (gl == 0) {
        gs->phase = kFetch;
        gs->flags &= ~(kLive | kFinished);
      }
    }
    __syncwarp(gmask);
  }
}

#undef xs
#undef best
#undef scale
#undef diag
#undef delta
#undef cand
#undef gs
#undef pbs

}  // namespace smpc
