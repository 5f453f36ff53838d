// smpc_tracker.cu — tracked perception of the closed-loop episodes (smpc_run_tracked_episodes): the perception stage of
// smpc_perception.cu followed by a per-robot people tracker. Detections are exactly those of smpc_perception_kernel
// (the same range, wall, occlusion and detection tests and the same Philox counters); the measurement is the noisy
// position only. Each agent id of a robot has one constant-velocity Kalman track, confirmed after confirm_hits
// detections, coasted through up to max_coast misses and published at its estimate; the FOV filter reads the list
// published latency ticks earlier from a ring of latency + 1 slots the host rotates.
// Laid out like smpc_perception_kernel: one warp per robot, lanes over the list's rows (two slots per lane, L <= 64),
// the true offsets in shared memory for the O(L^2) occlusion test, one lane per row for the ray walk and the filter
// step, and an order-preserving compaction with __ballot_sync / __popc into the ring slot.
// The filter step, per axis with the covariance (p_pp, p_pv, p_vv) both axes share, in this order (tests/tracker_ref.py
// follows it; -fmad=false in the Makefile keeps every product and sum IEEE-rounded):
//   q_pp = a2 * dt2 * dt2 / 4, q_pv = a2 * dt2 * dt / 2, q_vv = a2 * dt2   (a2 = accel_noise^2, dt2 = dt * dt)
//   predict: p = p + dt * v
//            p_pp = p_pp + 2 * dt * p_pv + dt2 * p_vv + q_pp;  p_pv = p_pv + dt * p_vv + q_pv;  p_vv = p_vv + q_vv
//   update:  S = p_pp + r2 (r2 = meas_noise^2), k0 = p_pp / S, k1 = p_pv / S, i = z - p
//            p = p + k0 * i;  v = v + k1 * i
//            p_vv = p_vv - k1 * p_pv;  p_pv = p_pv - k0 * p_pv;  p_pp = p_pp - k0 * p_pp
//   birth:   p = z, v = 0, p_pp = r2, p_pv = 0, p_vv = init_vel_std^2
#include <cuda_runtime.h>

#include <cmath>
#include <string>

#include "../../include/smpc.h"
#include "smpc_host_state.h"
#include "smpc_perception.cuh"

namespace {

constexpr int kWarps = 4;
constexpr int kMaxRows = 64;       // two slots per lane
constexpr int kMaxHits = 16;       // hits saturate here (confirm_hits <= 16)
constexpr double kPersonal = 1.2;  // m, the personal zone of the person metrics

struct TrackerSmem {  // per warp: the true offsets (p - robot) of the list's rows and their squared distances
  double dx[kMaxRows], dy[kMaxRows], d2[kMaxRows];
};

__global__ void __launch_bounds__(kWarps * 32) smpc_tracked_perception_kernel(smpc_tracker_args t) {
  __shared__ TrackerSmem smem[kWarps];
  const smpc_perception_args& a = t.p;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.x * kWarps + warp;
  if (b >= a.B) return;  // warp-uniform
  if (!a.active[b]) {    // a finished robot publishes nothing and its tracks freeze
    if (lane == 0) {
      t.pub_n[b] = 0;
      t.del_n[b] = 0;  // the next tick's slot: nothing reads it before the next launch overwrites it
    }
    return;
  }
  TrackerSmem& s = smem[warp];
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
  const double dt = t.dt, dt2 = dt * dt, a2 = t.accel_noise * t.accel_noise, r2 = t.meas_noise * t.meas_noise;
  const double q_pp = a2 * dt2 * dt2 / 4.0, q_pv = a2 * dt2 * dt / 2.0, q_vv = a2 * dt2;
  bool pub[2] = {false, false}, miss = false;
  unsigned id[2] = {0u, 0u};
  double est[2][4];
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int j = lane + 32 * q;
    if (j >= n) continue;
    // detection: smpc_perception_kernel's tests, in its order
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
        const double tt = (fx * ex + fy * ey) / d2;
        if (!(tt > 0.0 && tt < 1.0)) continue;
        const double gx = fx - tt * ex, gy = fy - tt * ey;
        if (gx * gx + gy * gy < a.occluder_r2) {
          v = false;
          break;
        }
      }
    if (v && a.occluding_cost > 0)
      v = !wall_between(map, a.size_x, a.size_y, (rx - ox) / a.resolution, (ry - oy) / a.resolution,
                        (in[5 * j] - ox) / a.resolution, (in[5 * j + 1] - oy) / a.resolution, a.occluding_cost);
    if (!v && other < 0 && dist < kPersonal) miss = true;

    // the track of this id
    const size_t ti = (size_t)b * t.M + id[q];
    int hits = t.hits[ti], misses = t.misses[ti];
    double px = 0.0, py = 0.0, vx = 0.0, vy = 0.0, pp = 0.0, pv = 0.0, vv = 0.0;
    if (hits > 0) {  // predict
      px = t.px[ti]; py = t.py[ti]; vx = t.vx[ti]; vy = t.vy[ti];
      pp = t.p_pp[ti]; pv = t.p_pv[ti]; vv = t.p_vv[ti];
      px = px + dt * vx;
      py = py + dt * vy;
      pp = pp + 2.0 * dt * pv + dt2 * vv + q_pp;
      pv = pv + dt * vv + q_pv;
      vv = vv + q_vv;
    }
    if (v) {
      double zx = in[5 * j], zy = in[5 * j + 1];
      if (a.pos_noise > 0.0) {  // the position draw of smpc_perception_kernel; zero noise adds nothing
        double n0x, n0y;
        normal2(philox4x32_10(make_uint4((unsigned)a.k, stream, id[q], 0u), key), &n0x, &n0y);
        zx = zx + a.pos_noise * n0x;
        zy = zy + a.pos_noise * n0y;
      }
      if (hits == 0) {  // birth
        px = zx; py = zy; vx = 0.0; vy = 0.0;
        pp = r2; pv = 0.0; vv = t.init_vel_std * t.init_vel_std;
        hits = 1;
      } else {  // update
        const double S = pp + r2, k0 = pp / S, k1 = pv / S;
        const double ix = zx - px, iy = zy - py;
        px = px + k0 * ix;
        py = py + k0 * iy;
        vx = vx + k1 * ix;
        vy = vy + k1 * iy;
        vv = vv - k1 * pv;
        pv = pv - k0 * pv;
        pp = pp - k0 * pp;
        hits = min(hits + 1, kMaxHits);
      }
      misses = 0;
    } else if (hits > 0 && ++misses > t.max_coast) {  // death
      hits = 0;
      misses = 0;
    }
    t.hits[ti] = hits;
    t.misses[ti] = misses;
    if (hits > 0) {
      t.px[ti] = px; t.py[ti] = py; t.vx[ti] = vx; t.vy[ti] = vy;
      t.p_pp[ti] = pp; t.p_pv[ti] = pv; t.p_vv[ti] = vv;
    }
    pub[q] = hits >= t.confirm_hits;  // confirm_hits >= 1: no track, nothing published
    est[q][0] = px; est[q][1] = py; est[q][2] = vx; est[q][3] = vy;
  }

  // order-preserving compaction of the published tracks into the ring slot of tick k
  const unsigned m0 = __ballot_sync(0xffffffffu, pub[0]), m1 = __ballot_sync(0xffffffffu, pub[1]);
  const unsigned below = (1u << lane) - 1u;
  const int n0 = __popc(m0), n_pub = n0 + __popc(m1);
  double* out = t.pub + (size_t)b * L * 5;
  int32_t* out_id = t.pub_id + (size_t)b * L;
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    if (!pub[q]) continue;
    const int o = q == 0 ? __popc(m0 & below) : n0 + __popc(m1 & below);
    for (int c = 0; c < 4; ++c) out[5 * o + c] = est[q][c];
    out[5 * o + 4] = 0.0;  // a position tracker estimates no turn rate
    out_id[o] = (int32_t)id[q];
  }
  if (lane == 0) t.pub_n[b] = n_pub;
  __syncwarp();  // with latency 0 the delayed slot is the one just written

  // what the FOV filter receives at tick k: the slot of tick k - latency, against the true list of tick k
  const int nd = t.del_n[b];
  const double* del = t.del + (size_t)b * L * 5;
  const int32_t* del_id = t.del_id + (size_t)b * L;
  double* log = a.seen_log ? a.seen_log + ((size_t)b * a.T + a.k) * L * 5 : nullptr;
  int32_t* id_log = t.id_log ? t.id_log + ((size_t)b * a.T + a.k) * L : nullptr;
  unsigned got_lo = 0u, got_hi = 0u;  // bit i: person i was delivered
  unsigned rows = 0u;
  double pe = 0.0, ve = 0.0;
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int o = lane + 32 * q;
    if (o < nd) {
      const int i = del_id[o];
      if (log)
        for (int c = 0; c < 5; ++c) log[5 * o + c] = del[5 * o + c];
      if (id_log) id_log[o] = i;
      if (i < a.K) {  // a person: its true row of tick k is row i + R - 1 of the list
        if (i < 32) got_lo |= 1u << i;
        else got_hi |= 1u << (i - 32);
        const double* tr = in + 5 * (i + a.R - 1);
        const double dx = del[5 * o] - tr[0], dy = del[5 * o + 1] - tr[1];
        const double dvx = del[5 * o + 2] - tr[2], dvy = del[5 * o + 3] - tr[3];
        rows += 1u;
        pe = pe + sqrt(dx * dx + dy * dy);
        ve = ve + sqrt(dvx * dvx + dvy * dvy);
      }
    } else if (o < L) {
      if (log)
        for (int c = 0; c < 5; ++c) log[5 * o + c] = 0.0;
      if (id_log) id_log[o] = -1;
    }
  }
  got_lo = __reduce_or_sync(0xffffffffu, got_lo);
  got_hi = __reduce_or_sync(0xffffffffu, got_hi);
  rows = __reduce_add_sync(0xffffffffu, rows);
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) {
    pe = pe + __shfl_xor_sync(0xffffffffu, pe, m);
    ve = ve + __shfl_xor_sync(0xffffffffu, ve, m);
  }
  bool untracked = false;
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int j = lane + 32 * q;
    if (j >= n || j < a.R - 1 || !(sqrt(s.d2[j]) < kPersonal)) continue;
    const int i = j - (a.R - 1);
    if (!(((i < 32 ? got_lo : got_hi) >> (i & 31)) & 1u)) untracked = true;
  }
  const bool any_miss = __any_sync(0xffffffffu, miss), any_untracked = __any_sync(0xffffffffu, untracked);
  if (lane == 0) {
    a.unseen[b] += any_miss;
    t.untracked[b] += any_untracked;
    t.track_rows[b] += (int32_t)rows;
    t.pos_err[b] += pe;
    t.vel_err[b] += ve;
    if (a.n_seen_log) a.n_seen_log[(size_t)b * a.T + a.k] = nd;
  }
}

}  // namespace

int smpc_tracked_perception_enqueue(smpc_handle* h, const smpc_tracker_args& a, cudaStream_t st) {
  if (a.p.B == 0) return SMPC_OK;
  smpc_tracked_perception_kernel<<<(unsigned)((a.p.B + kWarps - 1) / kWarps), kWarps * 32, 0, st>>>(a);
  SMPC_FLEET_CUDA(cudaGetLastError());
  smpc_handle_count_launch(h);
  return SMPC_OK;
}
