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
#include "smpc_perception.cuh"

namespace {

constexpr int kWarps = 4;
constexpr int kMaxRows = 64;     // two slots per lane
constexpr double kPersonal = 1.2;  // m, the personal zone of the person metrics

struct PerceptionSmem {  // per warp: the true offsets (p - robot) of the list's rows and their squared distances
  double dx[kMaxRows], dy[kMaxRows], d2[kMaxRows];
};

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
