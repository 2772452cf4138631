// icp_step.cuh -- the update step of the reference loop (labels_segmentation/icp.py:5-53), coded
// once for every kernel that runs it: the SE(2) pose, the centred match sums, the closed-form 2D
// Kabsch increment, applying and composing that increment, and the per-pair result.
//
// These expressions define the result bits of the CTA, pair and scan-to-map kernels and of
// best_fit.  nvcc contracts a * b + c into one FMA where the source allows it, so the operation
// order of every expression below is part of the result: write a new caller through these helpers,
// not through an algebraically equal form (e.g. compose() is not se2_mul with a rotation built from
// (cs, -sn, sn, cs): that contracts differently).
#pragma once

#include <cuda_runtime.h>

#include <cstdint>

#include "b200icp.h"

// x -> R x + T, stored row-major as b200icp.h lays out a pose: r00 r01 r10 r11 tx ty
struct Se2 {
  double r00, r01, r10, r11, tx, ty;
};
__device__ __forceinline__ Se2 se2_identity() { return Se2{1.0, 0.0, 0.0, 1.0, 0.0, 0.0}; }
__device__ __forceinline__ Se2 se2_load(const double* p) { return Se2{p[0], p[1], p[2], p[3], p[4], p[5]}; }
__device__ __forceinline__ void se2_store(double* p, const Se2& a) {
  p[0] = a.r00; p[1] = a.r01; p[2] = a.r10; p[3] = a.r11; p[4] = a.tx; p[5] = a.ty;
}
// a o b : first b, then a  (x -> Ra (Rb x + tb) + ta)
__device__ __forceinline__ Se2 se2_mul(const Se2& a, const Se2& b) {
  Se2 c;
  c.r00 = a.r00 * b.r00 + a.r01 * b.r10; c.r01 = a.r00 * b.r01 + a.r01 * b.r11;
  c.r10 = a.r10 * b.r00 + a.r11 * b.r10; c.r11 = a.r10 * b.r01 + a.r11 * b.r11;
  c.tx = a.r00 * b.tx + a.r01 * b.ty + a.tx;
  c.ty = a.r10 * b.tx + a.r11 * b.ty + a.ty;
  return c;
}

// Pose p of an init_pose table ([pairs][6]), identity when there is none.
__device__ __forceinline__ Se2 load_init_pose(const double* init_pose, int64_t p) {
  return init_pose ? se2_load(init_pose + p * 6) : se2_identity();
}

__device__ __forceinline__ double2 apply(const Se2& a, double2 q) {
  return make_double2(a.r00 * q.x + a.r01 * q.y + a.tx, a.r10 * q.x + a.r11 * q.y + a.ty);
}

// One ICP increment: rotation by (cos, sin), then translation.
struct Increment {
  double cs, sn, tx, ty;
};

// The increment as a pose (the pose_last output).
__device__ __forceinline__ Se2 as_se2(const Increment& d) { return Se2{d.cs, -d.sn, d.sn, d.cs, d.tx, d.ty}; }

__device__ __forceinline__ double2 apply(const Increment& d, double2 q) {      // icp.py:45
  return make_double2(d.cs * q.x - d.sn * q.y + d.tx, d.sn * q.x + d.cs * q.y + d.ty);
}

// d o a: the cumulative pose after the increment d
__device__ __forceinline__ Se2 compose(const Increment& d, const Se2& a) {
  Se2 c;
  c.r00 = d.cs * a.r00 - d.sn * a.r10; c.r01 = d.cs * a.r01 - d.sn * a.r11;
  c.r10 = d.sn * a.r00 + d.cs * a.r10; c.r11 = d.sn * a.r01 + d.cs * a.r11;
  c.tx = d.cs * a.tx - d.sn * a.ty + d.tx; c.ty = d.sn * a.tx + d.cs * a.ty + d.ty;
  return c;
}

// One match (a, b) in the centred sums r[0..7]: a' = a - oa, b' = b - ob, then sum a', sum b' and
// sum a' b'^T.  Centring on a point near the clouds keeps the single-pass covariance
// H = sum a'b'^T - (sum a')(sum b')^T / n (icp.py:10-16) free of cancellation.
__device__ __forceinline__ void add_match(double* r, double ax, double ay, double qx, double qy) {
  r[0] += ax; r[1] += ay; r[2] += qx; r[3] += qy;
  r[4] = fma(ax, qx, r[4]); r[5] = fma(ax, qy, r[5]);
  r[6] = fma(ay, qx, r[6]); r[7] = fma(ay, qy, r[7]);
}

// best_fit_transform (icp.py:5-26) from the sums r[0..7] of add_match over the matches, inv = 1 /
// their count, (oax, oay) / (obx, oby) the origins the sources / targets were centred on: the
// closed-form proper rotation the SVD route (icp.py:17-23) returns, and t = cB - R cA (icp.py:25).
// A degenerate H (h2 == 0) gives the identity rotation.
__device__ __forceinline__ Increment kabsch_increment(const double* r, double inv, double oax, double oay,
                                                      double obx, double oby) {
  const double max_ = r[0] * inv, may_ = r[1] * inv;        // centroids rel. the origins (icp.py:10-11)
  const double mbx = r[2] * inv, mby = r[3] * inv;
  const double h00 = fma(-r[0], mbx, r[4]), h01 = fma(-r[0], mby, r[5]);
  const double h10 = fma(-r[1], mbx, r[6]), h11 = fma(-r[1], mby, r[7]);
  const double num = h01 - h10, den = h00 + h11;
  const double h2 = fma(num, num, den * den);
  Increment d{1.0, 0.0, 0.0, 0.0};
  if (h2 > 0.0) {
    const double rh = rsqrt(h2);
    d.cs = den * rh; d.sn = num * rh;
  }
  const double cax = oax + max_, cay = oay + may_;
  d.tx = (obx + mbx) - (d.cs * cax - d.sn * cay);
  d.ty = (oby + mby) - (d.sn * cax + d.cs * cay);
  return d;
}

// The per-pair scalars of b200icp_outputs (thread 0 of the pair); rmse = sqrt(mean_d2).
__device__ __forceinline__ void write_pair_result(const b200icp_outputs& out, int64_t p, const Se2& pose,
                                                  const Increment& last, double err, double mean_d2, int inl,
                                                  int iters) {
  se2_store(out.pose_total + p * 6, pose);
  if (out.pose_last) se2_store(out.pose_last + p * 6, as_se2(last));
  out.error[p] = err;
  if (out.rmse) out.rmse[p] = sqrt(mean_d2);
  if (out.inliers) out.inliers[p] = inl;
  out.iterations[p] = iters;
}
