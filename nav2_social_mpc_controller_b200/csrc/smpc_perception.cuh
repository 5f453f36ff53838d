// smpc_perception.cuh — device functions of the perception stage that smpc_perception.cu and smpc_tracker.cu share:
// the counter-based random numbers and the wall test of the line of sight (include/smpc.h, smpc_perception).
// Both files compile with -fmad=false, so the wall test uses only IEEE-rounded arithmetic in either.
#pragma once

#include <cuda_runtime.h>

#include <cstdint>

namespace {

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

}  // namespace
