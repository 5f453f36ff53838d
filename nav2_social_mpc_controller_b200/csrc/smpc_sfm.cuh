// smpc_sfm.cuh — the lightsfm social force model (reference include/nav2_social_mpc_controller/sfm.hpp:239-281) and
// computeObstacle (src/optimizer.cpp:673-728) shared by the people projection of the controller (smpc_project.cu) and
// the reactive crowd of the closed-loop episodes (smpc_crowd.cu). Both kernels therefore move people with the same
// arithmetic.
#pragma once
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>

#include "smpc_math.cuh"

namespace smpc {

__device__ __forceinline__ double wrap_pi(double a) {
  while (a <= -M_PI) a += 2 * M_PI;
  while (a > M_PI) a -= 2 * M_PI;
  return a;
}

// lightsfm social force of one agent pair exactly as the reference writes it (sfm.hpp:239-281): d = other - me,
// w = my velocity - other's. Out of line: sfm_pair only comes here for degenerate geometry (coincident agents, zero
// interaction vector, |sin theta| < 1e-9 — e.g. two people standing still, where theta == 0 switches the lateral term
// off), where the two-atan2 form and its exact-zero tests decide the result.
static __device__ __noinline__ void sfm_pair_reference(double dx, double dy, double wx, double wy, double* fx, double* fy) {
  const double kSocial = 2.1, kLambda = 2.0, kGamma = 0.35, kN = 2.0, kNPrime = 3.0;
  const double z = dx * dx + dy * dy;
  const double dn = sqrt(z);
  double ex = dx, ey = dy;
  if (z > 0.0) {
    ex = dx / dn;
    ey = dy / dn;
  }
  const double Ix = kLambda * wx + ex, Iy = kLambda * wy + ey;
  const double il = sqrt(Ix * Ix + Iy * Iy);
  const double ix = Ix / il, iy = Iy / il;
  const double a1 = wrap_pi(atan2(iy, ix));
  const double a2 = wrap_pi(atan2(ey, ex));
  const double th = wrap_pi(a2 - a1);
  const double B = kGamma * il;
  const double fv = -exp(-dn / B - (kNPrime * B * th) * (kNPrime * B * th));
  double sgn = -1.0;
  if (th == 0) sgn = 0; else if (th > 0) sgn = 1;
  const double fa = -sgn * exp(-dn / B - (kN * B * th) * (kN * B * th));
  *fx = kSocial * (fv * ix + fa * (-iy));
  *fy = kSocial * (fv * iy + fa * ix);
}

// (sfx, sfy) plus the social force of the agent at d = other - me with w = my velocity - other's. The generic
// branch adds with an explicit FMA: written inline in the loop, `sfx += kSocial * (...)` contracted into one, and this
// keeps that rounding wherever the function is inlined.
// Generic geometry: unit vectors by reciprocal square roots, ONE atan2 of (cross, dot) for the angle from the
// interaction direction i to e, the kernel's own exp (smpc_math.cuh; each within ~1 ulp of the libm call it
// replaces — the projected trajectories move by ~1e-15). Degenerate geometry: the reference's formulation.
__device__ __forceinline__ double2 sfm_pair(double dx, double dy, double wx, double wy, double sfx, double sfy) {
  const double kSocial = 2.1, kLambda = 2.0, kGamma = 0.35, kN = 2.0, kNPrime = 3.0;
  const double z = dx * dx + dy * dy;
  const double inv_dn = rsqrt_pos(z);  // NaN for z == 0: caught by the test on `cross` below
  const double dn = z * inv_dn, ex = dx * inv_dn, ey = dy * inv_dn;
  const double Ix = kLambda * wx + ex, Iy = kLambda * wy + ey;
  const double L2 = Ix * Ix + Iy * Iy;
  const double inv_il = rsqrt_pos(L2);
  const double il = L2 * inv_il, ix = Ix * inv_il, iy = Iy * inv_il;
  const double cross = ey * ix - ex * iy, dot = ex * ix + ey * iy;
  if (fabs(cross) > 1e-9) {  // false for NaN
    const double th = atan2_unit(cross, dot);
    const double Bth = kGamma * il * th, base = -dn * inv_il * (1.0 / kGamma);
    const double fv = -exp_nonpos(base - (kNPrime * Bth) * (kNPrime * Bth));
    const double fa = -copysign(exp_nonpos(base - (kN * Bth) * (kN * Bth)), th);
    sfx = fma(fv * ix - fa * iy, kSocial, sfx);
    sfy = fma(fv * iy + fa * ix, kSocial, sfy);
  } else {
    double rx, ry;
    sfm_pair_reference(dx, dy, wx, wy, &rx, &ry);
    sfx += rx;
    sfy += ry;
  }
  return make_double2(sfx, sfy);
}

// computeObstacle: the vector the reference stores in obstacles1 (agent - nearest obstacle cell, SURVEY Q10) from an
// obstacle-distance grid of od_width x od_height cells of od_resolution m with origin (ox, oy). False beyond the
// grid's far edges (or for an index outside it). A point left of or below the origin is NOT reported: the conversion
// of a negative cell coordinate to unsigned saturates to 0 on the GPU, so it reads column / row 0, as the projection
// always has (its bits are pinned). A caller that needs "none outside the grid" tests x >= ox and y >= oy itself.
__device__ __forceinline__ bool nearest_obstacle(uint32_t od_width, uint32_t od_height, float od_resolution,
                                                 const uint32_t* idx, double ox, double oy, double x, double y,
                                                 double* out_x, double* out_y) {
  const unsigned int xc = (unsigned int)floor((x - ox) / od_resolution);
  const unsigned int yc = (unsigned int)floor((y - oy) / od_resolution);
  if (xc >= od_width || yc >= od_height) return false;
  const unsigned int ob = idx[xc + yc * od_width];
  if (ob >= od_width * od_height) return false;
  const unsigned int cy = ob / od_width, cx = ob % od_width;
  const float fx = cx * od_resolution + ox;  // float-rounded like the reference (:719-720)
  const float fy = cy * od_resolution + oy;
  *out_x = x - (double)fx;
  *out_y = y - (double)fy;
  return true;
}

}  // namespace smpc
