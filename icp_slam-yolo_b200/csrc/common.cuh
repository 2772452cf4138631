// common.cuh -- what every CUDA source of the library shares: the point layout, the pair
// addressing of b200icp_problem, the float64 distance every exact decision uses, the error API
// behind b200icp_last_error(), and (icp_step.cuh) the update step of the ICP loop.
#pragma once

#include <cuda_runtime.h>
#include <math_constants.h>

#include <cstdint>

#include "b200icp.h"
#include "icp_step.cuh"

constexpr unsigned kFull = 0xffffffffu;   // all lanes of a warp
constexpr int kGroup = 8;          // targets per search group
constexpr int kMaxWarps = 8;       // CTA size limit of the per-pair kernels
constexpr int kMaxS = 4;           // source points per lane
constexpr int kMaxSrcPitch = kMaxS * kMaxWarps * 32;   // 1024
constexpr int kMaxTgtPitch = 4096;

// Records a printf-style message for b200icp_last_error() and returns `code`.
int set_error(int code, const char* fmt, ...) __attribute__((format(printf, 2, 3)));
// B200ICP_OK if no CUDA error is pending, else B200ICP_ERR_CUDA with the message
// "<what>: <CUDA error string>" (`what` is printf-style).
int check_launch(const char* what, ...) __attribute__((format(printf, 1, 2)));
// Lets `kern` use `bytes` of dynamic shared memory, more than the 48 KB default (bytes < 0: the most
// the device allows).  Set once per kernel and device; later calls return at once.
int opt_in_dynamic_smem(const void* kern, int bytes);
// Validates the problem description shared by the pair-batch entry points; `pitch_limit` = false skips
// the pitch limits of the fused kernels (entry points that stage no shared-memory tile).
int check_problem(const b200icp_problem* pr, int64_t n_pairs, bool pitch_limit = true);

struct KernelArgs {
  b200icp_problem prob;
  b200icp_options opt;
  b200icp_outputs out;
  int32_t* nn_idx;      // nn kernel only
  double* nn_dist2;     // nn kernel only
  int64_t n_pairs;
  int32_t mcap;         // tgt_pitch rounded up to kGroup
  int32_t ncap;         // warp kernel: src_pitch rounded up to 32 * SC
  int32_t use_gate;
  int32_t passes;       // warp kernels: ncap / (32 * sources per lane)
  int32_t reuse;        // fused warp kernel: skip the sweep of a pass while its sources provably keep their group
};

__device__ __forceinline__ int64_t tri_offset(int64_t i, int64_t rows) {
  return i * (2 * rows - i - 1) / 2;       // pairs (i', j) with i' < i
}

// Which rows does pair p use?  (b200icp_pairing in b200icp.h)
__device__ __forceinline__ void resolve_rows(const b200icp_problem& pr, int64_t p,
                                             int64_t& srow, int64_t& trow) {
  if (pr.pairing == B200ICP_PAIR_ROWWISE) {
    srow = p; trow = p;
  } else if (pr.pairing == B200ICP_PAIR_EXPLICIT) {
    srow = pr.src_row[p]; trow = pr.tgt_row[p];
  } else {
    const int64_t rows = pr.n_rows;
    const int64_t q = pr.first_pair + p;
    const double b = 2.0 * (double)rows - 1.0;
    int64_t i = (int64_t)floor((b - sqrt(fmax(b * b - 8.0 * (double)q, 0.0))) * 0.5);
    i = max((int64_t)0, min(i, rows - 2));
    while (i > 0 && tri_offset(i, rows) > q) --i;
    while (i < rows - 2 && tri_offset(i + 1, rows) <= q) ++i;
    trow = i;
    srow = q - tri_offset(i, rows) + i + 1;
  }
}

// Valid points of the two rows of a pair: the row length, capped at the pitch.
__device__ __forceinline__ void row_lengths(const b200icp_problem& pr, int64_t srow, int64_t trow, int& n, int& m) {
  n = pr.src_len ? min(pr.src_len[srow], pr.src_pitch) : pr.src_pitch;
  m = pr.tgt_len ? min(pr.tgt_len[trow], pr.tgt_pitch) : pr.tgt_pitch;
}

// "No neighbour" (index -1, d^2 = +inf) in the slots i0, i0 + stride, ... below pitch of an NN row.
__device__ __forceinline__ void nn_fill_none(int32_t* idx, double* d2, int i0, int pitch, int stride) {
  for (int i = i0; i < pitch; i += stride) {
    idx[i] = -1;
    if (d2) d2[i] = CUDART_INF;
  }
}

__device__ __forceinline__ double2 load_point(const void* base, int dtype, int64_t i) {
  if (dtype == B200ICP_F64) return __ldg(reinterpret_cast<const double2*>(base) + i);
  const float2 v = __ldg(reinterpret_cast<const float2*>(base) + i);
  return make_double2((double)v.x, (double)v.y);
}

// float64 squared distance with numpy's operation order (no contraction), so exact
// ties resolve as in a float64 brute-force argmin.
__device__ __forceinline__ double dist2_f64(double sx, double sy, double2 t) {
  const double dx = __dsub_rn(sx, t.x), dy = __dsub_rn(sy, t.y);
  return __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
}

// How far above the FP32 best another group's minimum may lie and still hide the true
// (float64) nearest neighbour.  u = 2^-24.  cs = max |centred source coordinate| (FP32).
//   direct  : sqrt(d32) is within 2.9*eta of the true distance, eta = (cs + tmax) * 2u
//             -> compare distances:  thr = (sqrt(best)(1 + 2^-20) + 4*eta)^2 (1 + 2^-22)
//   expanded: |e32 - e_exact| <= 6u*tmax*(cs + tmax) per value (tt rounding + two FMAs) and
//             the FP32-rounded points sit within rho = 2.83u*max(cs,tmax) of the true
//             ones -> margin = 2*8u*tmax*(cs+tmax) + 4*dB*rho + 2*rho^2 on (second - best),
//             dB an upper bound of the best distance.            (Derivations: DESIGN.md)
// Guard band of the expanded form in e-space, monotone in cs:  2*8u*tmax(cs+tmax) for the two
// FFMA roundings + 4*dB*rho + 2*rho^2 for the FP32 rounding of the points themselves, with the
// best distance bounded by dB <= sqrt(2)(cs+tmax) and rho = 2.83u*max(cs,tmax):
//   margin <= 2^-20 (cs+tmax)(tmax + 1.2 max(cs,tmax))
__device__ __forceinline__ float expanded_margin(float cs, float tmax) {
  return 9.5367432e-7f * (cs + tmax) * fmaf(1.2f, fmaxf(cs, tmax), tmax);
}
