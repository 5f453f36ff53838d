// smpc_local_costmap.cu — rolling local costmaps of the closed-loop episodes (smpc_run_local_costmap_episodes): one
// robot-centred window per robot, cropped from its static costmap at whole cells, with the cells around the people in it
// raised to a fixed inflation stencil, as Nav2's local costmap marks them with its obstacle layer and inflates them with
// its inflation layer. The FOV filter and the fleet tick read the windows in place of the static maps.
// One CTA per running robot. Warp 0 compacts the rows of the robot's list whose static cell lies inside the window into
// shared memory (ballot / popc, 64 rows per pass), the stencil sits in shared memory, and every thread owns 4-byte words
// of the window: it reads their static bytes and maxes in each marked row whose stencil box covers them. Owner-computes
// with no atomics, and integer-only after the floor of each position, so a build is deterministic and
// tests/local_costmap_ref.py reproduces it byte for byte (-fmad=false in the Makefile keeps the floors' operands and
// the origin IEEE-rounded).
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

#include "../../include/smpc.h"
#include "smpc_host_state.h"

namespace {

constexpr int kThreads = 256;
constexpr int kMaxHalf = 32;
constexpr int kStencilMax = (2 * kMaxHalf + 1) * (2 * kMaxHalf + 1);
constexpr int kRowsPerPass = 64;  // two rows per lane of warp 0
constexpr double kCellLimit = 1e15;  // |cell index| bound before the conversion to an integer (far beyond any map)

__global__ void __launch_bounds__(kThreads) smpc_local_costmap_kernel(smpc_local_costmap_args a) {
  __shared__ uint8_t sten[kStencilMax];
  __shared__ int row_x[kRowsPerPass], row_y[kRowsPerPass];
  __shared__ int n_marked;
  const int b = blockIdx.x;
  if (!a.active[b]) return;  // block-uniform: a finished robot keeps its last window
  const int mi = a.map_index ? a.map_index[b] : b % a.n_costmaps;
  const double ox = a.map_org[2 * mi], oy = a.map_org[2 * mi + 1], res = a.resolution;
  const double cx = floor((a.pose[3 * b] - ox) / res), cy = floor((a.pose[3 * b + 1] - oy) / res);
  const long long c0x = (long long)fmin(fmax(cx, -kCellLimit), kCellLimit) - a.sx / 2;
  const long long c0y = (long long)fmin(fmax(cy, -kCellLimit), kCellLimit) - a.sy / 2;
  const int half = a.half, w = 2 * half + 1;
  for (int i = threadIdx.x; i < w * w; i += kThreads) sten[i] = a.stencil[i];

  const int n = a.n_list ? min(a.n_list[b], a.L) : 0;
  const uint8_t* map = a.maps + (size_t)mi * a.size_y * a.size_x;
  const int cells = a.sx * a.sy, words = (cells + 3) >> 2;
  const bool aligned = (cells & 3) == 0;  // then every window (and log row) starts on a 4-byte boundary
  uint8_t* win = a.window + (size_t)b * cells;
  uint8_t* log = a.window_log ? a.window_log + ((size_t)b * a.n_builds + a.build) * cells : nullptr;
  int total = 0;
  for (int base = 0; base == 0 || base < n; base += kRowsPerPass) {
    __syncthreads();  // the stencil is staged; the previous pass's rows are consumed
    if (threadIdx.x < 32) {
      const int lane = threadIdx.x;
      // row j of this pass -> (window column, window row), or (-1, -1) when its static cell is not in the window
      auto cell_of = [&](int j) {
        if (j >= n) return make_int2(-1, -1);
        const double* p = a.list + ((size_t)b * a.L + j) * 5;
        const double fx = floor((p[0] - ox) / res) - (double)c0x, fy = floor((p[1] - oy) / res) - (double)c0y;
        const bool in = fx >= 0.0 && fx < (double)a.sx && fy >= 0.0 && fy < (double)a.sy;  // NaN: not marked
        return in ? make_int2((int)fx, (int)fy) : make_int2(-1, -1);
      };
      const int2 r0 = cell_of(base + lane), r1 = cell_of(base + lane + 32);
      const unsigned m0 = __ballot_sync(0xffffffffu, r0.x >= 0), m1 = __ballot_sync(0xffffffffu, r1.x >= 0);
      const unsigned below = (1u << lane) - 1u;
      const int n0 = __popc(m0);
      if (r0.x >= 0) {
        const int o = __popc(m0 & below);
        row_x[o] = r0.x;
        row_y[o] = r0.y;
      }
      if (r1.x >= 0) {
        const int o = n0 + __popc(m1 & below);
        row_x[o] = r1.x;
        row_y[o] = r1.y;
      }
      if (lane == 0) n_marked = n0 + __popc(m1);
    }
    __syncthreads();
    const int nm = n_marked;
    total += nm;
    for (int wd = threadIdx.x; wd < words; wd += kThreads) {
      unsigned packed = 0u;
      for (int q = 0; q < 4; ++q) {
        const int i = 4 * wd + q;
        if (i >= cells) break;
        const int wy = i / a.sx, wx = i - wy * a.sx;
        int v = 0;
        if (base == 0) {  // the static layer
          const long long gx = c0x + wx, gy = c0y + wy;
          if (gx >= 0 && gx < a.size_x && gy >= 0 && gy < a.size_y) v = map[(size_t)gy * a.size_x + (size_t)gx];
        } else {  // a later pass maxes into what this thread wrote
          v = win[i];
        }
        for (int m = 0; m < nm; ++m) {
          const int dx = wx - row_x[m], dy = wy - row_y[m];
          if (abs(dx) <= half && abs(dy) <= half) v = max(v, (int)sten[(dy + half) * w + dx + half]);
        }
        packed |= (unsigned)v << (8 * q);
      }
      if (aligned) {
        reinterpret_cast<unsigned*>(win)[wd] = packed;
        if (log) reinterpret_cast<unsigned*>(log)[wd] = packed;
      } else {
        for (int q = 0; q < 4 && 4 * wd + q < cells; ++q) {
          win[4 * wd + q] = (uint8_t)(packed >> (8 * q));
          if (log) log[4 * wd + q] = (uint8_t)(packed >> (8 * q));
        }
      }
    }
  }
  if (threadIdx.x == 0) {
    const double wox = __dadd_rn(ox, __dmul_rn((double)c0x, res)), woy = __dadd_rn(oy, __dmul_rn((double)c0y, res));
    a.origin[2 * b] = wox;
    a.origin[2 * b + 1] = woy;
    a.marked[b] += total;
    if (a.origin_log) {
      double* o = a.origin_log + ((size_t)b * a.n_builds + a.build) * 2;
      o[0] = wox;
      o[1] = woy;
    }
  }
}

}  // namespace

int smpc_local_costmap_enqueue(smpc_handle* h, const smpc_local_costmap_args& a, cudaStream_t st) {
  if (a.B == 0) return SMPC_OK;
  smpc_local_costmap_kernel<<<(unsigned)a.B, kThreads, 0, st>>>(a);
  SMPC_FLEET_CUDA(cudaGetLastError());
  smpc_handle_count_launch(h);
  return SMPC_OK;
}

int smpc_local_costmap_build_stencil(const smpc_local_costmap* l, double res, std::vector<uint8_t>* stencil, int* half,
                                     const char* name) {
  auto fail_arg = [name](const char* msg) {
    return smpc_host_fail(SMPC_ERR_ARGUMENT, std::string(name) + ": " + msg);
  };
  auto finite_ge0 = [](double x) { return std::isfinite(x) && x >= 0.0; };
  if (l->size_x < 8 || l->size_x > 256 || l->size_y < 8 || l->size_y > 256)
    return fail_arg("local costmap size_x or size_y outside 8..256");
  if (l->update_period_ticks < 1 || l->update_period_ticks > 20) return fail_arg("update_period_ticks outside 1..20");
  if (l->mark_people != 0 && l->mark_people != 1) return fail_arg("mark_people not 0 or 1");
  if (!finite_ge0(l->agent_radius) || !finite_ge0(l->inscribed_radius))
    return fail_arg("agent_radius or inscribed_radius not finite and >= 0");
  if (!(std::isfinite(l->cost_scaling_factor) && l->cost_scaling_factor > 0.0))
    return fail_arg("cost_scaling_factor not finite and > 0");
  if (!(std::isfinite(l->inflation_radius) && l->inflation_radius >= l->inscribed_radius))
    return fail_arg("inflation_radius not finite and >= inscribed_radius");
  if (!(std::isfinite(res) && res > 0.0)) return fail_arg("resolution not finite and > 0");

  // Computed on a grid one cell wider than the largest stencil: a non-zero entry on its rim means a half-width above 32
  // (cost falls with the distance to the disc, so a wider non-zero stencil is non-zero on this rim too).
  constexpr int H = kMaxHalf + 1, W = 2 * H + 1;
  const double rho = l->agent_radius / res + 1e-9, rho2 = rho * rho;
  auto lethal = [rho2](int dx, int dy) {
    return dx < -H || dx > H || dy < -H || dy > H ? false : (double)(dx * dx + dy * dy) <= rho2;
  };
  std::vector<int> edge;  // lethal cells with a non-lethal 4-neighbour: the nearest lethal cell is always one of them
  for (int dy = -H; dy <= H; ++dy)
    for (int dx = -H; dx <= H; ++dx)
      if (lethal(dx, dy) && !(lethal(dx - 1, dy) && lethal(dx + 1, dy) && lethal(dx, dy - 1) && lethal(dx, dy + 1))) {
        edge.push_back(dx);
        edge.push_back(dy);
      }
  std::vector<uint8_t> grid((size_t)W * W, 0);
  int hw = 0;
  for (int dy = -H; dy <= H; ++dy)
    for (int dx = -H; dx <= H; ++dx) {
      int cost = 254;
      if (!lethal(dx, dy)) {
        double d2 = INFINITY;
        for (size_t e = 0; e < edge.size(); e += 2) {
          const double ex = (double)(dx - edge[e]), ey = (double)(dy - edge[e + 1]);
          d2 = std::fmin(d2, ex * ex + ey * ey);
        }
        const double d = std::sqrt(d2);
        if (d * res <= l->inscribed_radius + 1e-9)
          cost = 253;
        else if (d <= l->inflation_radius / res + 1e-9)
          cost = (int)std::floor(252.0 * std::exp(-l->cost_scaling_factor * (d * res - l->inscribed_radius)));
        else
          cost = 0;
      }
      grid[(size_t)(dy + H) * W + (dx + H)] = (uint8_t)cost;
      if (cost > 0) hw = std::max(hw, std::max(std::abs(dx), std::abs(dy)));
    }
  *half = hw;
  if (hw > kMaxHalf) return fail_arg("the local costmap stencil's half-width above 32");
  const int w = 2 * hw + 1;
  stencil->assign((size_t)w * w, 0);
  for (int r = 0; r < w; ++r)
    for (int c = 0; c < w; ++c) (*stencil)[(size_t)r * w + c] = grid[(size_t)(r + H - hw) * W + (c + H - hw)];
  return SMPC_OK;
}

extern "C" int smpc_local_costmap_stencil(const smpc_local_costmap* local, double resolution, uint8_t* out,
                                          int capacity, int* half_width) {
  if (!local || !half_width) return smpc_host_fail(SMPC_ERR_ARGUMENT, "local_costmap_stencil: NULL argument");
  std::vector<uint8_t> s;
  const int rc = smpc_local_costmap_build_stencil(local, resolution, &s, half_width, "local_costmap_stencil");
  if (rc != SMPC_OK) return rc;
  if (out) {
    if (capacity < (int)s.size()) return smpc_host_fail(SMPC_ERR_ARGUMENT, "local_costmap_stencil: capacity too small");
    std::copy(s.begin(), s.end(), out);
  }
  return SMPC_OK;
}
