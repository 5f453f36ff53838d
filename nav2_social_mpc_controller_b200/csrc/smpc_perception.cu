// smpc_perception.cu — sensor-limited perception of the closed-loop episodes (smpc_run_perceived_episodes): between the
// true scene state and the FOV filter, each robot's list of people (and, in shared scenes, other robots) is cut to what
// a range-limited sensor with line of sight, missed detections and noisy tracks reports. Laid out like the crowd
// kernels: one warp per robot, lanes over the list's rows (two slots per lane, L <= 64), the rows' true offsets from the
// robot in shared memory for the O(L^2) occlusion test, one lane per row for the ray walk over the costmap bytes, and
// an order-preserving compaction with __ballot_sync / __popc over the two slots.
// Random numbers are counter-based (Philox4x32-10 on (k, stream, agent id, draw)), so results do not depend on the
// launch configuration, the early-stop poll or the batch composition.
// Compiled with -fmad=false (Makefile): the visibility decision uses only IEEE-rounded + - * / sqrt, so
// tests/perception_ref.py reproduces it exactly.
#include <cuda_runtime.h>

#include <cmath>
#include <string>

#include "../../include/smpc.h"
#include "smpc_host_state.h"

namespace {

constexpr int kWarps = 4;
constexpr int kMaxRows = 64;     // two slots per lane
constexpr double kPersonal = 1.2;  // m, the personal zone of the person metrics

struct PerceptionSmem {  // per warp: the true offsets (p - robot) of the list's rows and their squared distances
  double dx[kMaxRows], dy[kMaxRows], d2[kMaxRows];
};

// Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3"; Random123's philox4x32 with 10 rounds)
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 key) {
  for (int r = 0; r < 10; ++r) {
    const unsigned lo0 = 0xD2511F53u * c.x, hi0 = __umulhi(0xD2511F53u, c.x);
    const unsigned lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi(0xCD9E8D57u, c.z);
    c = make_uint4(hi1 ^ c.y ^ key.x, lo1, hi0 ^ c.w ^ key.y, lo0);
    key.x += 0x9E3779B9u;
    key.y += 0xBB67AE85u;
  }
  return c;
}

// two words -> a uniform in (0, 1] with 53 random bits: 2^-53 .. 1
__device__ __forceinline__ double uniform53(unsigned a, unsigned b) {
  return (double)(((unsigned long long)a << 21) + (b >> 11) + 1ull) * 0x1p-53;
}

// two standard normals from one Philox block (Box-Muller)
__device__ __forceinline__ void normal2(uint4 w, double* n0, double* n1) {
  const double r = sqrt(-2.0 * log(uniform53(w.x, w.y)));
  double s, c;
  sincospi(2.0 * uniform53(w.z, w.w), &s, &c);  // cos, sin of 2 pi u2 without a large-argument reduction
  *n0 = r * c;
  *n1 = r * s;
}

// Amanatides-Woo walk in grid units from the robot's cell to the row's cell: true when a cell strictly between them lies
// in the costmap with cost >= occ. Steps x when tmx <= tmy (conservative at exact corners) and never past the end
// index on an axis, so the walk takes exactly |dix| + |diy| steps; cells outside the costmap do not block.
__device__ bool wall_between(const uint8_t* map, int size_x, int size_y, double gx0, double gy0, double gx1, double gy1,
                             int occ) {
  int cx = (int)floor(gx0), cy = (int)floor(gy0);
  const int ex = (int)floor(gx1), ey = (int)floor(gy1);
  int nx = abs(ex - cx), ny = abs(ey - cy);
  const int sx = ex > cx ? 1 : -1, sy = ey > cy ? 1 : -1;
  const double ax = fabs(gx1 - gx0), ay = fabs(gy1 - gy0);
  double tmx = INFINITY, tmy = INFINITY, tdx = INFINITY, tdy = INFINITY;
  if (nx > 0) {
    tmx = (sx > 0 ? (double)(cx + 1) - gx0 : gx0 - (double)cx) / ax;
    tdx = 1.0 / ax;
  }
  if (ny > 0) {
    tmy = (sy > 0 ? (double)(cy + 1) - gy0 : gy0 - (double)cy) / ay;
    tdy = 1.0 / ay;
  }
  for (int s = nx + ny - 1; s > 0; --s) {  // the last step lands on the row's own cell
    if (ny == 0 || (nx > 0 && tmx <= tmy)) {
      cx += sx;
      tmx += tdx;
      --nx;
    } else {
      cy += sy;
      tmy += tdy;
      --ny;
    }
    if ((unsigned)cx < (unsigned)size_x && (unsigned)cy < (unsigned)size_y && map[(size_t)cy * size_x + cx] >= occ)
      return true;
  }
  return false;
}

__global__ void __launch_bounds__(kWarps * 32) smpc_perception_kernel(smpc_perception_args a) {
  __shared__ PerceptionSmem smem[kWarps];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * kWarps + warp;
  if (b >= a.B) return;  // warp-uniform
  if (!a.active[b]) {
    if (lane == 0) a.n_seen[b] = 0;
    return;
  }
  PerceptionSmem& s = smem[warp];
  const int L = a.L;
  const int n = min(a.n_list[b], L);
  const double rx = a.pose[3 * b], ry = a.pose[3 * b + 1];
  const double* in = a.list + (size_t)b * L * 5;
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int j = lane + 32 * q;
    if (j >= n) continue;
    const double dx = in[5 * j] - rx, dy = in[5 * j + 1] - ry;
    s.dx[j] = dx;
    s.dy[j] = dy;
    s.d2[j] = dx * dx + dy * dy;
  }
  __syncwarp();

  const int me = b % a.R;
  const unsigned stream = a.stream_index ? (unsigned)a.stream_index[b] : (unsigned)b;
  const uint2 key = make_uint2((unsigned)a.seed, (unsigned)(a.seed >> 32));
  const int mi = a.map_index ? a.map_index[b] : b % a.n_costmaps;
  const uint8_t* map = a.maps + (size_t)mi * a.size_y * a.size_x;
  const double ox = a.map_org[2 * mi], oy = a.map_org[2 * mi + 1];
  bool vis[2] = {false, false}, miss = false;
  unsigned id[2] = {0u, 0u};
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int j = lane + 32 * q;
    if (j >= n) continue;
    // rows 0 .. R-2 of a shared scene's view are the other robots in index order; people keep their scene slot
    const int other = j < a.R - 1 ? (j < me ? j : j + 1) : -1;
    id[q] = other >= 0 ? (unsigned)(a.K + other) : (unsigned)(j - (a.R - 1));
    const double ex = s.dx[j], ey = s.dy[j], d2 = s.d2[j];
    const double dist = sqrt(d2);
    bool v = dist <= a.max_range;
    if (v && a.detect_prob < 1.0) {
      const uint4 w = philox4x32_10(make_uint4((unsigned)a.k, stream, id[q], 2u), key);
      v = uniform53(w.x, w.y) <= a.detect_prob;
    }
    if (v && a.occluder_r2 > 0.0)
      for (int i = 0; i < n; ++i) {
        if (!(s.d2[i] < d2)) continue;  // only a strictly closer row occludes
        const double fx = s.dx[i], fy = s.dy[i];
        const double t = (fx * ex + fy * ey) / d2;
        if (!(t > 0.0 && t < 1.0)) continue;
        const double gx = fx - t * ex, gy = fy - t * ey;
        if (gx * gx + gy * gy < a.occluder_r2) {
          v = false;
          break;
        }
      }
    if (v && a.occluding_cost > 0)
      v = !wall_between(map, a.size_x, a.size_y, (rx - ox) / a.resolution, (ry - oy) / a.resolution,
                        (in[5 * j] - ox) / a.resolution, (in[5 * j + 1] - oy) / a.resolution, a.occluding_cost);
    vis[q] = v;
    if (!v && other < 0 && dist < kPersonal) miss = true;
  }

  // order-preserving compaction: slot 0 rows (0 .. 31) come before slot 1 rows (32 .. 63)
  const unsigned m0 = __ballot_sync(0xffffffffu, vis[0]), m1 = __ballot_sync(0xffffffffu, vis[1]);
  const unsigned below = (1u << lane) - 1u;
  const int n0 = __popc(m0), n_out = n0 + __popc(m1);
  double* out = a.seen + (size_t)b * L * 5;
  double* log = a.seen_log ? a.seen_log + ((size_t)b * a.T + a.k) * L * 5 : nullptr;
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    if (!vis[q]) continue;
    const int j = lane + 32 * q;
    const int o = q == 0 ? __popc(m0 & below) : n0 + __popc(m1 & below);
    double row[5];
    for (int c = 0; c < 5; ++c) row[c] = in[5 * j + c];
    if (a.pos_noise > 0.0) {  // zero noise adds nothing, not even a signed zero
      double n0x, n0y;
      normal2(philox4x32_10(make_uint4((unsigned)a.k, stream, id[q], 0u), key), &n0x, &n0y);
      row[0] = row[0] + a.pos_noise * n0x;
      row[1] = row[1] + a.pos_noise * n0y;
    }
    if (a.vel_noise > 0.0) {
      double n1x, n1y;
      normal2(philox4x32_10(make_uint4((unsigned)a.k, stream, id[q], 1u), key), &n1x, &n1y);
      row[2] = row[2] + a.vel_noise * n1x;
      row[3] = row[3] + a.vel_noise * n1y;
    }
    for (int c = 0; c < 5; ++c) out[5 * o + c] = row[c];
    if (log)
      for (int c = 0; c < 5; ++c) log[5 * o + c] = row[c];
  }
  if (log)
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int o = lane + 32 * q;
      if (o >= n_out && o < L)
        for (int c = 0; c < 5; ++c) log[5 * o + c] = 0.0;
    }
  const bool any_miss = __any_sync(0xffffffffu, miss);
  if (lane == 0) {
    a.n_seen[b] = n_out;
    a.unseen[b] += any_miss;
    if (a.n_seen_log) a.n_seen_log[(size_t)b * a.T + a.k] = n_out;
  }
}

}  // namespace

int smpc_perception_enqueue(smpc_handle* h, const smpc_perception_args& a, cudaStream_t st) {
  if (a.B == 0) return SMPC_OK;
  smpc_perception_kernel<<<(unsigned)((a.B + kWarps - 1) / kWarps), kWarps * 32, 0, st>>>(a);
  SMPC_FLEET_CUDA(cudaGetLastError());
  smpc_handle_count_launch(h);
  return SMPC_OK;
}
