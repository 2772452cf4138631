// b200icp.cu -- sm_100a kernels and C ABI of the 2D ICP scan-matching path.
//
// Reference behaviour being replaced (paths relative to the reference repo):
//   labels_segmentation/icp.py:28-53  icp()                 -> icp_align_kernel
//   labels_segmentation/icp.py:37-38  KDTree(B).query(src)   -> nn_candidates + nn_resolve
//   labels_segmentation/icp.py:5-26   best_fit_transform()   -> pose solve inside icp_align_kernel
//   duc/ICP_LIDAR/process.py:38-52    polar_to_cartesian_3d  -> polar_to_cartesian_kernel
//
// Kernel design (see DESIGN.md):
//   * one CTA per scan pair, the whole <=max_iterations loop on the device;
//   * target scan staged once per pair in shared memory: float64 (x,y) for exact
//     re-evaluation / gather, and negated float32 SoA copies for the candidate search;
//   * candidate search: each lane owns S source points in registers and sweeps the
//     targets in groups of 8 with packed FP32x2 math (FADD2/FMUL2/FFMA2) and FMNMX,
//     tracking per source the best group, its minimum and the runner-up group minimum;
//   * every decision is then re-made in float64: the best group is rescanned exactly
//     (ascending index, strict <, i.e. lowest index wins ties); if the runner-up group
//     lies inside the FP32 error guard band the whole warp rescans all targets for that
//     source in float64 and a shuffle argmin with (distance, index) ordering decides;
//   * all O(N) state (source points, centroid / covariance sums, pose, error) is float64,
//     reduced by warp shuffles + one shared-memory hop, every thread solving the 2x2
//     Kabsch problem in closed form redundantly (no broadcast step).
#include <cuda_runtime.h>
#include <math_constants.h>

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <set>
#include <utility>

#include "b200icp.h"

namespace {

constexpr int kGroup = 8;          // targets per search group
constexpr int kMaxWarps = 8;       // CTA size limit of the per-pair kernels
constexpr int kMaxS = 4;           // source points per lane
constexpr int kMaxSrcPitch = kMaxS * kMaxWarps * 32;   // 1024
constexpr int kMaxTgtPitch = 4096;
constexpr int64_t kAutoCtaPairs = 512;    // at or below: CTA-per-pair fused kernel (latency), above: W warps per pair (throughput)
constexpr int kRedStride = 8;      // doubles per warp slot in the staging reductions
constexpr int kRedStride2 = 12;    // doubles per warp slot in the per-iteration reduction
constexpr unsigned kFull = 0xffffffffu;
// CTAs of kMaxWarps warps that must fit one SM: caps registers per thread
// (65536 / (256 * kMinBlocks)); typical CTAs have 4 warps, so twice as many are resident.
#ifndef B200ICP_MIN_BLOCKS
#define B200ICP_MIN_BLOCKS 2
#endif

thread_local char g_last_error[512] = "";

void set_error(const char* fmt, const char* a = "", const char* b = "") {
  snprintf(g_last_error, sizeof(g_last_error), fmt, a, b);
}

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

// ------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------
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

__device__ __forceinline__ double2 load_point(const void* base, int dtype, int64_t i) {
  if (dtype == B200ICP_F64) return __ldg(reinterpret_cast<const double2*>(base) + i);
  const float2 v = __ldg(reinterpret_cast<const float2*>(base) + i);
  return make_double2((double)v.x, (double)v.y);
}

// Sum K doubles over the CTA.  Warp shuffle tree, one shared-memory hop, then every
// thread adds the per-warp partials in the same fixed order, so all threads hold the
// same bits and no broadcast is needed.  `scratch` must not be the buffer used by the
// previous call (callers alternate between two).
template <int K>
__device__ __forceinline__ void block_sum(double (&v)[K], double* scratch, int warp, int lane,
                                          int nwarps) {
  constexpr int kStride = K <= kRedStride ? kRedStride : kRedStride2;
#pragma unroll
  for (int k = 0; k < K; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(kFull, v[k], o);
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < K; ++k) scratch[warp * kStride + k] = v[k];
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < K; ++k) {
    double acc = scratch[k];
    for (int w = 1; w < nwarps; ++w) acc += scratch[w * kStride + k];
    v[k] = acc;
  }
}

// ------------------------------------------------------------------------------------
// shared-memory tile of one target scan
// ------------------------------------------------------------------------------------
struct TargetTile {
  double2* t64;    // [mcap] exact float64 points (sentinel = +inf beyond m)
  float* fx;       // [mcap] centred float32 x   (direct form stores the NEGATED value)
  float* fy;       // [mcap] centred float32 y
  float* ft;       // [mcap] |centred point|^2 rounded once (expanded form only)
  double* red;     // [2][kMaxWarps][kRedStride2] reduction scratch (double buffered)
  float* wmax;     // [kMaxWarps]
  double ox, oy;   // origin = target centroid; distances are translation invariant and
                   // small centred magnitudes keep the FP32 guard band narrow
  float tmax;      // max |centred target coordinate|
  int m, mcap, ngroups;
};

__host__ __device__ inline size_t tile_bytes(int mcap) {
  return (size_t)mcap * (sizeof(double2) + 3 * sizeof(float)) +
         2 * kMaxWarps * kRedStride2 * sizeof(double) + kMaxWarps * sizeof(float);
}

__device__ __forceinline__ void carve_tile(unsigned char* smem, int mcap, TargetTile& t) {
  t.t64 = reinterpret_cast<double2*>(smem);
  t.fx = reinterpret_cast<float*>(t.t64 + mcap);
  t.fy = t.fx + mcap;
  t.ft = t.fy + mcap;
  // mcap is a multiple of 8, so (16 + 12) * mcap keeps 8-byte alignment for the doubles
  t.red = reinterpret_cast<double*>(t.ft + mcap);
  t.wmax = reinterpret_cast<float*>(t.red + 2 * kMaxWarps * kRedStride2);
  t.mcap = mcap;
}

// Stage the target scan: float64 copy, centroid, centred float32 SoA copies (+ |t|^2), pad.
__device__ __forceinline__ void stage_targets(const void* tgt, int dtype, int64_t row_off, int m,
                                              TargetTile& t, int tid, int nthreads, int warp,
                                              int lane, int nwarps) {
  t.m = m;
  t.ngroups = (m + kGroup - 1) / kGroup;
  double sum[2] = {0.0, 0.0};
  for (int j = tid; j < t.mcap; j += nthreads) {
    double2 q = make_double2(CUDART_INF, CUDART_INF);      // sentinel: infinitely far
    if (j < m) {
      q = load_point(tgt, dtype, row_off + j);
      sum[0] += q.x; sum[1] += q.y;
    }
    t.t64[j] = q;
  }
  block_sum<2>(sum, t.red, warp, lane, nwarps);             // syncs: t64 is visible after this
  t.ox = sum[0] / (double)m;
  t.oy = sum[1] / (double)m;
  float amax = 0.f;
  for (int j = tid; j < t.mcap; j += nthreads) {
    if (j < m) {
      const double2 q = t.t64[j];
      const float cx = (float)(q.x - t.ox), cy = (float)(q.y - t.oy);
      amax = fmaxf(amax, fmaxf(fabsf(cx), fabsf(cy)));
      t.fx[j] = cx; t.fy[j] = cy;
      t.ft[j] = (float)((double)cx * (double)cx + (double)cy * (double)cy);
    } else {
      t.fx[j] = 0.f; t.fy[j] = 0.f; t.ft[j] = CUDART_INF_F;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(kFull, amax, o));
  if (lane == 0) t.wmax[warp] = amax;
  __syncthreads();
  float r = t.wmax[0];
  for (int w = 1; w < nwarps; ++w) r = fmaxf(r, t.wmax[w]);
  t.tmax = r;
}

// ------------------------------------------------------------------------------------
// candidate search (FP32): per source the best group of 8 targets, its minimum and the
// runner-up group minimum.  Two arithmetic forms of the same brute-force sweep:
//   EXPANDED: e_j = |t_j|^2 - 2 s.t_j  (= d^2 - |s|^2)    2 FFMA + 1 FMNMX per pair
//   direct  : d_j = (sx - tx_j)^2 + (sy - ty_j)^2            2 FADD + FMUL + FFMA + FMNMX
// The expanded form is ~1.6x cheaper in issue slots; its larger rounding error only widens
// the guard band of nn_resolve, never the result.
// ------------------------------------------------------------------------------------
template <int S>
struct Candidates {
  float best[S];
  float second[S];
  int group[S];
};

template <int S>
__device__ __forceinline__ void track(Candidates<S>& c, int k, float m, int g) {
  const float old = c.best[k];
  c.second[k] = fminf(c.second[k], fmaxf(old, m));
  c.group[k] = (m < old) ? g : c.group[k];
  c.best[k] = fminf(old, m);
}

template <int S>
__device__ __forceinline__ void nn_candidates(const TargetTile& t, const float (&sx)[S],
                                              const float (&sy)[S], Candidates<S>& c) {
  const float4* __restrict__ x4 = reinterpret_cast<const float4*>(t.fx);
  const float4* __restrict__ y4 = reinterpret_cast<const float4*>(t.fy);
  const float4* __restrict__ q4 = reinterpret_cast<const float4*>(t.ft);
  float a[S], b[S];
#pragma unroll
  for (int k = 0; k < S; ++k) {
    float vx = -2.0f * sx[k];
    float vy = -2.0f * sy[k];
    // opaque copies: stops ptxas from re-converting the float64 state inside the loop
    asm volatile("" : "+f"(vx), "+f"(vy));
    a[k] = vx; b[k] = vy;
    c.best[k] = CUDART_INF_F;
    c.second[k] = CUDART_INF_F;
    c.group[k] = 0;
  }
  const int ngroups = t.ngroups;
#pragma unroll 1
  for (int g = 0; g < ngroups; ++g) {
    const float4 xa = x4[2 * g], xb = x4[2 * g + 1];
    const float4 ya = y4[2 * g], yb = y4[2 * g + 1];
    const float4 qa = q4[2 * g], qb = q4[2 * g + 1];
#pragma unroll
    for (int k = 0; k < S; ++k) {
      // packed FP32x2: two targets per FFMA2 issue slot (the loop is issue/ALU bound,
      // not FMA-pipe bound: profiles/r1_ubench_issue_rates.txt)
      const float2 ak = make_float2(a[k], a[k]), bk = make_float2(b[k], b[k]);
      const float2 e01 = __ffma2_rn(ak, make_float2(xa.x, xa.y), __ffma2_rn(bk, make_float2(ya.x, ya.y), make_float2(qa.x, qa.y)));
      const float2 e23 = __ffma2_rn(ak, make_float2(xa.z, xa.w), __ffma2_rn(bk, make_float2(ya.z, ya.w), make_float2(qa.z, qa.w)));
      const float2 e45 = __ffma2_rn(ak, make_float2(xb.x, xb.y), __ffma2_rn(bk, make_float2(yb.x, yb.y), make_float2(qb.x, qb.y)));
      const float2 e67 = __ffma2_rn(ak, make_float2(xb.z, xb.w), __ffma2_rn(bk, make_float2(yb.z, yb.w), make_float2(qb.z, qb.w)));
      const float m = fminf(fminf(fminf(e01.x, e01.y), fminf(e23.x, e23.y)),
                            fminf(fminf(e45.x, e45.y), fminf(e67.x, e67.y)));
      track<S>(c, k, m, g);
    }
  }
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

__device__ __forceinline__ bool is_ambiguous(float best, float second, float scx, float scy, float tmax) {
  const float cs = fmaxf(fabsf(scx), fabsf(scy));
  return (second - best) <= expanded_margin(cs, tmax);   // near-equal floats subtract exactly
}

// sqrt of a float64 in [~1e-30, ~1e30]: FP32 rsqrt seed + two Newton steps on the residual
// (9 instructions instead of ~20 + a slow-path branch).  Faithfully rounded (<= 1 ulp), which is
// far inside the 1e-9 relative error budget of the mean-distance bookkeeping.
__device__ __forceinline__ double sqrt_f64_fast(double x) {
  const float xf = (float)x;
  if (!(xf > 1e-30f && xf < 1e30f)) return sqrt(x);          // zero, tiny, huge, NaN: library path
  const double y = (double)rsqrtf(xf);
  double g = x * y;
  const double h = 0.5 * y;
  g = fma(fma(-g, g, x), h, g);
  g = fma(fma(-g, g, x), h, g);
  return g;
}

// Re-decide every correspondence in float64.  Must be called by all lanes of the warp.
template <int S>
__device__ __forceinline__ void nn_resolve(const TargetTile& t, const Candidates<S>& c,
                                           const double (&sx)[S], const double (&sy)[S],
                                           const float (&fx)[S], const float (&fy)[S],
                                           const bool (&valid)[S], int lane, int (&idx)[S],
                                           double (&d2)[S]) {
  const double2* __restrict__ t64 = t.t64;
#pragma unroll
  for (int k = 0; k < S; ++k) {
    const bool ambiguous = valid[k] && is_ambiguous(c.best[k], c.second[k], fx[k], fy[k], t.tmax);
    // fast path: the winner is inside the best group; rescan its 8 targets exactly
    // (ascending index, strict <: lowest index wins exact ties)
    double bd = CUDART_INF;
    int bj = c.group[k] * kGroup;
    if (valid[k]) {
      const int j0 = c.group[k] * kGroup;
#pragma unroll
      for (int u = 0; u < kGroup; ++u) {
        const double d = dist2_f64(sx[k], sy[k], t64[j0 + u]);
        if (d < bd) { bd = d; bj = j0 + u; }
      }
    }
    // slow path (rare): warp-cooperative exact scan of all targets for that source
    unsigned pending = __ballot_sync(kFull, ambiguous);
    while (pending) {
      const int owner = __ffs(pending) - 1;
      pending &= pending - 1;
      const double qx = __shfl_sync(kFull, sx[k], owner);
      const double qy = __shfl_sync(kFull, sy[k], owner);
      double ld = CUDART_INF;
      int lj = 0x7fffffff;
      for (int j = lane; j < t.m; j += 32) {
        const double d = dist2_f64(qx, qy, t64[j]);
        if (d < ld) { ld = d; lj = j; }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const double od = __shfl_xor_sync(kFull, ld, o);
        const int oj = __shfl_xor_sync(kFull, lj, o);
        if (od < ld || (od == ld && oj < lj)) { ld = od; lj = oj; }
      }
      if (lane == owner) { bd = ld; bj = lj; }
    }
    idx[k] = bj;
    d2[k] = bd;
  }
}

// One full search for the S source points a lane owns (float64 in, exact answer out).
template <int S>
__device__ __forceinline__ void nn_search(const TargetTile& t, const double (&sx)[S],
                                          const double (&sy)[S], const bool (&valid)[S], int lane,
                                          int (&idx)[S], double (&d2)[S]) {
  float fx[S], fy[S];
#pragma unroll
  for (int k = 0; k < S; ++k) {
    fx[k] = (float)(sx[k] - t.ox);
    fy[k] = (float)(sy[k] - t.oy);
  }
  Candidates<S> c;
  nn_candidates<S>(t, fx, fy, c);
  nn_resolve<S>(t, c, sx, sy, fx, fy, valid, lane, idx, d2);
}

// ------------------------------------------------------------------------------------
// kernel: nearest-neighbour search only (icp.py:37-38)
// ------------------------------------------------------------------------------------
template <int S>
__global__ void __launch_bounds__(kMaxWarps * 32, B200ICP_MIN_BLOCKS) nn_pair_kernel(const KernelArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  TargetTile t;
  carve_tile(smem_raw, a.mcap, t);

  const int tid = threadIdx.x, nthreads = blockDim.x;
  const int warp = tid >> 5, lane = tid & 31, nwarps = nthreads >> 5;
  const int64_t p = blockIdx.x;
  const b200icp_problem& pr = a.prob;

  int64_t srow, trow;
  resolve_rows(pr, p, srow, trow);
  const int n = pr.src_len ? min(pr.src_len[srow], pr.src_pitch) : pr.src_pitch;
  const int m = pr.tgt_len ? min(pr.tgt_len[trow], pr.tgt_pitch) : pr.tgt_pitch;
  int32_t* idx_out = a.nn_idx + p * pr.src_pitch;
  double* d2_out = a.nn_dist2 ? a.nn_dist2 + p * pr.src_pitch : nullptr;

  if (n <= 0 || m <= 0) {
    for (int i = tid; i < pr.src_pitch; i += nthreads) {
      idx_out[i] = -1;
      if (d2_out) d2_out[i] = CUDART_INF;
    }
    return;
  }
  stage_targets(pr.tgt_points, pr.dtype, trow * pr.tgt_pitch, m, t, tid, nthreads, warp,
                          lane, nwarps);
  double sx[S], sy[S];
  bool valid[S];
#pragma unroll
  for (int k = 0; k < S; ++k) {
    const int i = tid + k * nthreads;
    valid[k] = i < n;
    double2 q = make_double2(t.ox, t.oy);
    if (valid[k]) q = load_point(pr.src_points, pr.dtype, srow * pr.src_pitch + i);
    sx[k] = q.x; sy[k] = q.y;
  }
  int idx[S];
  double d2[S];
  nn_search<S>(t, sx, sy, valid, lane, idx, d2);
#pragma unroll
  for (int k = 0; k < S; ++k) {
    const int i = tid + k * nthreads;
    if (i < pr.src_pitch) {
      idx_out[i] = valid[k] ? idx[k] : -1;
      if (d2_out) d2_out[i] = valid[k] ? d2[k] : CUDART_INF;
    }
  }
}

// ------------------------------------------------------------------------------------
// kernel: the whole ICP loop for one pair (icp.py:28-53)
// ------------------------------------------------------------------------------------
template <int S>
__global__ void __launch_bounds__(kMaxWarps * 32, B200ICP_MIN_BLOCKS) icp_align_kernel(const KernelArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  TargetTile t;
  carve_tile(smem_raw, a.mcap, t);
  double* red = t.red;

  const int tid = threadIdx.x, nthreads = blockDim.x;
  const int warp = tid >> 5, lane = tid & 31, nwarps = nthreads >> 5;
  const int64_t p = blockIdx.x;
  const b200icp_problem& pr = a.prob;
  const b200icp_options& op = a.opt;
  const b200icp_outputs& out = a.out;

  int64_t srow, trow;
  resolve_rows(pr, p, srow, trow);
  const int n = pr.src_len ? min(pr.src_len[srow], pr.src_pitch) : pr.src_pitch;
  const int m = pr.tgt_len ? min(pr.tgt_len[trow], pr.tgt_pitch) : pr.tgt_pitch;

  // cumulative pose (src = Rt * A + tt) starts at the initial pose (gicp_lidar.py:32 shape)
  double R00 = 1.0, R01 = 0.0, R10 = 0.0, R11 = 1.0, T0 = 0.0, T1 = 0.0;
  if (op.init_pose) {
    const double* ip = op.init_pose + p * 6;
    R00 = ip[0]; R01 = ip[1]; R10 = ip[2]; R11 = ip[3]; T0 = ip[4]; T1 = ip[5];
  }
  double c_last = 1.0, s_last = 0.0, t0_last = 0.0, t1_last = 0.0;   // last increment
  double err = CUDART_INF, mean_d2 = CUDART_INF;
  int iters = 0, inl = 0;

  double sx[S], sy[S];
  bool valid[S];
  int idx[S];
#pragma unroll
  for (int k = 0; k < S; ++k) { sx[k] = 0.0; sy[k] = 0.0; valid[k] = false; idx[k] = -1; }

  const bool ran = n > 0 && m > 0 && op.max_iterations > 0;
  if (ran) {
    stage_targets(pr.tgt_points, pr.dtype, trow * pr.tgt_pitch, m, t, tid, nthreads,
                            warp, lane, nwarps);
#pragma unroll
    for (int k = 0; k < S; ++k) {
      const int i = tid + k * nthreads;
      valid[k] = i < n;
      if (valid[k]) {
        const double2 q = load_point(pr.src_points, pr.dtype, srow * pr.src_pitch + i);
        if (op.init_pose) {
          sx[k] = R00 * q.x + R01 * q.y + T0;
          sy[k] = R10 * q.x + R11 * q.y + T1;
        } else {
          sx[k] = q.x; sy[k] = q.y;          // icp.py:32  src = copy(A)
        }
      }
    }
    const double gate = op.max_corr_dist;
    const bool use_gate = a.use_gate != 0;
    const double inv_n = 1.0 / (double)n;
    double prev_error = 0.0;                                   // icp.py:33

    for (int it = 0; it < op.max_iterations; ++it) {           // icp.py:35
      // ---- correspondence search (icp.py:37-38)
      double d2[S];
      nn_search<S>(t, sx, sy, valid, lane, idx, d2);
      // ---- gather matches (icp.py:39), gate, ONE reduction of centred sums.
      // Coordinates are taken relative to the tile origin (the target centroid), so the
      // single-pass covariance  H = sum a'b'^T - (sum a')(sum b')^T / n  (icp.py:10-16) loses
      // nothing to cancellation: |centroid offsets| << point spread.
      double r[11] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
      for (int k = 0; k < S; ++k) {
        if (valid[k]) {
          const double dist = sqrt(d2[k]);
          if (!use_gate || dist < gate) {
            const double2 b = t.t64[idx[k]];
            const double ax = sx[k] - t.ox, ay = sy[k] - t.oy;
            const double qx = b.x - t.ox, qy = b.y - t.oy;
            r[0] += ax; r[1] += ay; r[2] += qx; r[3] += qy;
            r[4] = fma(ax, qx, r[4]); r[5] = fma(ax, qy, r[5]);
            r[6] = fma(ay, qx, r[6]); r[7] = fma(ay, qy, r[7]);
            r[8] += dist; r[9] += d2[k]; r[10] += 1.0;
          }
        }
      }
      block_sum<11>(r, red + (it & 1) * kMaxWarps * kRedStride2, warp, lane, nwarps);
      const double cnt = r[10];
      if (cnt < 0.5) {            // every correspondence gated out: stop, search not counted
        err = CUDART_INF; mean_d2 = CUDART_INF; inl = 0;
        break;
      }
      if (out.index_history) {
        int32_t* h = out.index_history + (p * op.max_iterations + it) * (int64_t)pr.src_pitch;
#pragma unroll
        for (int k = 0; k < S; ++k) {
          const int i = tid + k * nthreads;
          if (i < pr.src_pitch) h[i] = valid[k] ? idx[k] : -1;
        }
      }
      const double inv = use_gate ? 1.0 / cnt : inv_n;
      const double max_ = r[0] * inv, may_ = r[1] * inv;        // centroids rel. origin (icp.py:10-11)
      const double mbx = r[2] * inv, mby = r[3] * inv;
      const double mean_error = r[8] * inv;                     // icp.py:48
      // ---- closed-form 2D Kabsch: the proper rotation the SVD route (icp.py:17-23) returns
      const double h00 = fma(-r[0], mbx, r[4]), h01 = fma(-r[0], mby, r[5]);
      const double h10 = fma(-r[1], mbx, r[6]), h11 = fma(-r[1], mby, r[7]);
      const double num = h01 - h10, den = h00 + h11;
      const double h2 = fma(num, num, den * den);
      double cs = 1.0, sn = 0.0;
      if (h2 > 0.0) {
        const double rh = rsqrt(h2);
        cs = den * rh; sn = num * rh;
      }
      const double cax = t.ox + max_, cay = t.oy + may_;
      const double tx = (t.ox + mbx) - (cs * cax - sn * cay);   // icp.py:25
      const double ty = (t.oy + mby) - (sn * cax + cs * cay);
      // ---- apply (icp.py:45) and compose the cumulative pose
#pragma unroll
      for (int k = 0; k < S; ++k) {
        if (valid[k]) {
          const double x = sx[k], y = sy[k];
          sx[k] = cs * x - sn * y + tx;
          sy[k] = sn * x + cs * y + ty;
        }
      }
      {
        const double n00 = cs * R00 - sn * R10, n01 = cs * R01 - sn * R11;
        const double n10 = sn * R00 + cs * R10, n11 = sn * R01 + cs * R11;
        const double nt0 = cs * T0 - sn * T1 + tx, nt1 = sn * T0 + cs * T1 + ty;
        R00 = n00; R01 = n01; R10 = n10; R11 = n11; T0 = nt0; T1 = nt1;
      }
      c_last = cs; s_last = sn; t0_last = tx; t1_last = ty;
      err = mean_error; mean_d2 = r[9] * inv; inl = (int)(cnt + 0.5);
      iters = it + 1;
      // ---- convergence (icp.py:49-51); identical in every thread
      if (fabs(prev_error - mean_error) < op.tolerance) break;
      prev_error = mean_error;
    }
  }

  if (tid == 0) {
    double* pt = out.pose_total + p * 6;
    pt[0] = R00; pt[1] = R01; pt[2] = R10; pt[3] = R11; pt[4] = T0; pt[5] = T1;
    if (out.pose_last) {
      double* pl = out.pose_last + p * 6;
      pl[0] = c_last; pl[1] = -s_last; pl[2] = s_last; pl[3] = c_last;
      pl[4] = t0_last; pl[5] = t1_last;
    }
    out.error[p] = err;
    if (out.rmse) out.rmse[p] = sqrt(mean_d2);
    if (out.inliers) out.inliers[p] = inl;
    out.iterations[p] = iters;
  }
  if (out.indices || out.src_final) {
#pragma unroll
    for (int k = 0; k < S; ++k) {
      const int i = tid + k * nthreads;
      if (i < pr.src_pitch) {
        if (out.indices) out.indices[p * pr.src_pitch + i] = (i < n && iters > 0) ? idx[k] : -1;
        if (out.src_final) {
          double2 v = make_double2(0.0, 0.0);
          if (i < n) {
            if (ran) {
              v = make_double2(sx[k], sy[k]);
            } else {     // nothing ran: report the (pre-transformed) input
              const double2 q = load_point(pr.src_points, pr.dtype, srow * pr.src_pitch + i);
              v = make_double2(R00 * q.x + R01 * q.y + T0, R10 * q.x + R11 * q.y + T1);
            }
          }
          reinterpret_cast<double2*>(out.src_final)[p * pr.src_pitch + i] = v;
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------
// kernel: the whole ICP loop, ONE WARP PER PAIR (icp.py:28-53)
//
// The per-iteration work outside the candidate sweep (exact re-decision, distance, sums,
// pose solve) is what limits the block-per-pair kernel above: with 4 warps per pair every
// warp repeats the pose solve, the reductions cross shared memory and two barriers, and the
// float64 rescans run at FP64-pipe rate.  Here a single warp owns the pair:
//   * no block barrier anywhere; reductions are warp shuffles only; the pose is solved once;
//   * each lane sweeps SC source points per pass (all 360 points of a scan in one pass at
//     SC = 12), so one set of target LDS feeds 8*SC pair-evals;
//   * shared memory per warp holds only the centred float32 SoA target tile and the float64
//     source state; the float64 targets stay in global memory (L1/L2) and are touched once
//     per source per iteration (the matched point), because the in-group decision is made in
//     FP32 direct-difference form first (error ~1e-3 mm) and only near-ties fall back to the
//     warp-cooperative float64 scan.
// ------------------------------------------------------------------------------------
struct WarpTile {
  const void* tgt;      // global target table
  int64_t row_off;      // first point of this pair's target row
  int dtype;
  float* tile;          // [mcap/8][24]: per group of 8 targets x[8], y[8], |t|^2[8] (centred float32),
                        // 96 contiguous bytes = six LDS.128 off one address
  double2* src;         // [ncap] float64 source state
  float* gcx;           // [mcap/8] bounding circle of each group of 8 targets (pruned sweep)
  float* gcy;
  float* grad;
  unsigned char* grp;   // [src_pitch] group of every source's nearest neighbour at its last full sweep
                        // (one byte when the targets form <= 256 groups, else two)
  float* tpass;         // [passes] sweep-reuse thresholds (see WarpCtx::cum_move)
  bool grp16;
  double ox, oy;
  float tmax;
  int m, mcap, ngroups;
};

constexpr int kCtxBytes = 128;        // PairCtx slot in shared memory

// Sweep state of the throughput kernel: per source the THREE smallest group minima, each with its
// group number packed into the low mantissa bits (`keep` = ~((1 << bits) - 1), bits = log2 of the
// group count).  The keys stay floats -- a few low mantissa bits changed -- so fmin / fmax order
// them and no select is needed for the group numbers: six ALU operations per group and source.
// Tracking two groups instead of one is what lets a source keep its candidate set for many
// iterations: the nearest neighbour of a point near the seam of two groups of 8 flips between
// them after millimetres of motion, but stays inside their UNION until the point has moved half
// the gap to the third group.  The perturbation of the keys (relative 2^(bits-23), see key_eps)
// only widens guard bands: the two candidate groups are re-decided exactly afterwards.
template <int S>
struct Cand3 {
  float kb[S], ks[S], kt[S];
};

template <int S>
__device__ __forceinline__ void track3(Cand3<S>& c, int k, float m, unsigned g, unsigned keep) {
  const float key = __uint_as_float((__float_as_uint(m) & keep) | g);
  const float b = c.kb[k], s = c.ks[k];
  c.kt[k] = fminf(c.kt[k], fmaxf(s, key));
  c.ks[k] = fminf(s, fmaxf(b, key));
  c.kb[k] = fminf(b, key);
}

// Absolute error of a packed key: |e| <= 2 (cs + tmax)^2 for the expanded form, relative 2^(bits-23).
__device__ __forceinline__ float key_eps(float cs, float tmax, unsigned keep) {
  const float rel = (float)(~keep + 1u) * 1.1920929e-7f;          // 2^bits * 2^-23
  const float s = cs + tmax;
  return rel * 2.02f * s * s;
}

// Candidate sweep over the warp tile (expanded form, packed FFMA2), every group.
template <int S>
__device__ __forceinline__ void warp_candidates(const WarpTile& t, const float (&sx)[S],
                                                const float (&sy)[S], Cand3<S>& c, unsigned keep) {
  const float4* __restrict__ g4 = reinterpret_cast<const float4*>(t.tile);
  float a[S], b[S];
#pragma unroll
  for (int k = 0; k < S; ++k) {
    float vx = -2.0f * sx[k], vy = -2.0f * sy[k];
    asm volatile("" : "+f"(vx), "+f"(vy));
    a[k] = vx; b[k] = vy;
    c.kb[k] = CUDART_INF_F; c.ks[k] = CUDART_INF_F; c.kt[k] = CUDART_INF_F;
  }
  const int ngroups = t.ngroups;
#pragma unroll 1
  for (int g = 0; g < ngroups; ++g) {
    const float4 xa = g4[6 * g], xb = g4[6 * g + 1];
    const float4 ya = g4[6 * g + 2], yb = g4[6 * g + 3];
    const float4 qa = g4[6 * g + 4], qb = g4[6 * g + 5];
#pragma unroll
    for (int k = 0; k < S; ++k) {
      const float2 ak = make_float2(a[k], a[k]), bk = make_float2(b[k], b[k]);
      const float2 e01 = __ffma2_rn(ak, make_float2(xa.x, xa.y), __ffma2_rn(bk, make_float2(ya.x, ya.y), make_float2(qa.x, qa.y)));
      const float2 e23 = __ffma2_rn(ak, make_float2(xa.z, xa.w), __ffma2_rn(bk, make_float2(ya.z, ya.w), make_float2(qa.z, qa.w)));
      const float2 e45 = __ffma2_rn(ak, make_float2(xb.x, xb.y), __ffma2_rn(bk, make_float2(yb.x, yb.y), make_float2(qb.x, qb.y)));
      const float2 e67 = __ffma2_rn(ak, make_float2(xb.z, xb.w), __ffma2_rn(bk, make_float2(yb.z, yb.w), make_float2(qb.z, qb.w)));
      const float m = fminf(fminf(fminf(e01.x, e01.y), fminf(e23.x, e23.y)),
                            fminf(fminf(e45.x, e45.y), fminf(e67.x, e67.y)));
      track3<S>(c, k, m, (unsigned)g, keep);
    }
  }
}

// One group of 8 targets against the S sources of a lane (expanded form, packed FFMA2),
// split into the shared-memory loads and the arithmetic so the candidate loop can fetch the
// next group while the current one is being evaluated.
struct GroupRegs {
  float4 xa, xb, ya, yb, qa, qb;
};

__device__ __forceinline__ GroupRegs load_group(const WarpTile& t, int g) {
  const float4* __restrict__ g4 = reinterpret_cast<const float4*>(t.tile) + 6 * g;
  GroupRegs r;
  r.xa = g4[0]; r.xb = g4[1];
  r.ya = g4[2]; r.yb = g4[3];
  r.qa = g4[4]; r.qb = g4[5];
  return r;
}

template <int S>
__device__ __forceinline__ void eval_group(const GroupRegs& r, int g, const float (&a)[S],
                                           const float (&b)[S], Cand3<S>& c, unsigned keep) {
#pragma unroll
  for (int k = 0; k < S; ++k) {
    const float2 ak = make_float2(a[k], a[k]), bk = make_float2(b[k], b[k]);
    const float2 e01 = __ffma2_rn(ak, make_float2(r.xa.x, r.xa.y), __ffma2_rn(bk, make_float2(r.ya.x, r.ya.y), make_float2(r.qa.x, r.qa.y)));
    const float2 e23 = __ffma2_rn(ak, make_float2(r.xa.z, r.xa.w), __ffma2_rn(bk, make_float2(r.ya.z, r.ya.w), make_float2(r.qa.z, r.qa.w)));
    const float2 e45 = __ffma2_rn(ak, make_float2(r.xb.x, r.xb.y), __ffma2_rn(bk, make_float2(r.yb.x, r.yb.y), make_float2(r.qb.x, r.qb.y)));
    const float2 e67 = __ffma2_rn(ak, make_float2(r.xb.z, r.xb.w), __ffma2_rn(bk, make_float2(r.yb.z, r.yb.w), make_float2(r.qb.z, r.qb.w)));
    const float m = fminf(fminf(fminf(e01.x, e01.y), fminf(e23.x, e23.y)),
                          fminf(fminf(e45.x, e45.y), fminf(e67.x, e67.y)));
    track3<S>(c, k, m, (unsigned)g, keep);
  }
}

// Evaluate every group whose bit is set in `mask` (groups base_g + bit).
template <int S>
__device__ __forceinline__ void eval_mask(const WarpTile& t, unsigned mask, int base_g,
                                          const float (&a)[S], const float (&b)[S],
                                          Cand3<S>& c, unsigned keep) {
  while (mask) {
    const int g = base_g + __ffs(mask) - 1;
    mask &= mask - 1;
    const GroupRegs r = load_group(t, g);
    eval_group<S>(r, g, a, b, c, keep);
  }
}

// Warp-wide min / max of a float through the integer REDUX unit (one instruction instead of a
// five-step shuffle tree): floats are mapped to order-preserving unsigned keys first.
__device__ __forceinline__ unsigned f32_ordered(float f) {
  const unsigned u = __float_as_uint(f);
  return u ^ ((unsigned)((int)u >> 31) | 0x80000000u);
}
__device__ __forceinline__ float f32_unordered(unsigned k) {
  return __uint_as_float(k ^ (((k >> 31) - 1u) | 0x80000000u));
}
__device__ __forceinline__ float warp_min_f32(float f) {
  return f32_unordered(__reduce_min_sync(kFull, f32_ordered(f)));
}
__device__ __forceinline__ float warp_max_f32(float f) {
  return f32_unordered(__reduce_max_sync(kFull, f32_ordered(f)));
}

// squared distance from a point to an axis-aligned box (0 inside)
__device__ __forceinline__ float box_dist2(float px, float py, float x0, float x1, float y0, float y1) {
  const float dx = fmaxf(fmaxf(x0 - px, px - x1), 0.f);
  const float dy = fmaxf(fmaxf(y0 - py, py - y1), 0.f);
  return fmaf(dx, dx, dy * dy);
}

// Pruned candidate sweep.  The 32*S sources of a pass are consecutive scan points, i.e. a short
// piece of wall; their bounding box is compared with the bounding circle of every group of
// 8 targets.  Stage A evaluates the groups whose circles touch the sources' box; that
// yields, per source, an upper bound of its nearest-neighbour distance.  Stage B evaluates
// every remaining group whose circle could still hold a point within (that bound + the
// ambiguity margin) of any source.  Every skipped group is PROVEN farther than best + margin
// for every source of the pass, so the tracked best / runner-up / group are exactly what the
// full sweep would have produced for the purposes of nn-resolution (DESIGN.md 4.1); on
// unordered inputs every group overlaps and this degenerates to the full sweep.
template <int S>
__device__ __forceinline__ int warp_candidates_pruned(const WarpTile& t, const float (&sx)[S],
                                                      const float (&sy)[S], const bool (&valid)[S],
                                                      Cand3<S>& c, unsigned keep, float reach_scale,
                                                      float& reach_out) {
  int evaluated = 0;            // groups swept in this pass (diagnostics)
  float a[S], b[S], ss[S];
  float x0 = CUDART_INF_F, x1 = -CUDART_INF_F, y0 = CUDART_INF_F, y1 = -CUDART_INF_F;
#pragma unroll
  for (int k = 0; k < S; ++k) {
    a[k] = -2.0f * sx[k]; b[k] = -2.0f * sy[k];
    ss[k] = fmaf(sx[k], sx[k], sy[k] * sy[k]);
    c.kb[k] = CUDART_INF_F; c.ks[k] = CUDART_INF_F; c.kt[k] = CUDART_INF_F;
    if (valid[k]) {
      x0 = fminf(x0, sx[k]); x1 = fmaxf(x1, sx[k]);
      y0 = fminf(y0, sy[k]); y1 = fmaxf(y1, sy[k]);
    }
  }
  // bounding box of the pass's sources
  x0 = warp_min_f32(x0); x1 = warp_max_f32(x1);
  y0 = warp_min_f32(y0); y1 = warp_max_f32(y1);
  const float csk = fmaxf(fmaxf(fabsf(x0), fabsf(x1)), fmaxf(fabsf(y0), fabsf(y1)));
  // absolute slack for every FP32 rounding in the bound arithmetic: ~(csk + tmax) * 2^-20
  const float slack = (csk + t.tmax) * 9.5367432e-7f;
  const int ngroups = t.ngroups;
  const int words = (ngroups + 31) >> 5;
  const int lane = threadIdx.x & 31;
  // A group can hold a point within distance R of some source only if its circle (centre c,
  // radius rho) comes within R of the sources' box:  box_dist(c) <= R + rho (+ slack).
  // ---- stage A: R = 0, the groups whose circle touches the box
  float d2w0 = CUDART_INF_F, d2w1 = CUDART_INF_F, rw0 = 0.f, rw1 = 0.f;   // words 0/1 cached
  for (int w = 0; w < words; ++w) {
    const int g = (w << 5) + lane;
    float d2 = CUDART_INF_F, rr = 0.f;
    if (g < ngroups) {
      d2 = box_dist2(t.gcx[g], t.gcy[g], x0, x1, y0, y1) * 0.999996f;
      rr = t.grad[g] + slack;
    }
    if (w == 0) { d2w0 = d2; rw0 = rr; }
    if (w == 1) { d2w1 = d2; rw1 = rr; }
    const unsigned mask = __ballot_sync(kFull, d2 <= rr * rr);
    evaluated += __popc(mask);
    eval_mask<S>(t, mask, w << 5, a, b, c, keep);
  }
  // ---- upper bound of any source's NN distance^2 (the packed key may sit below the value by
  // key_eps), widened by the ambiguity margin
  float ub2 = 0.f;
#pragma unroll
  for (int k = 0; k < S; ++k)
    if (valid[k]) ub2 = fmaxf(ub2, c.kb[k] + ss[k]);
  ub2 = warp_max_f32(ub2) + key_eps(csk, t.tmax, keep);
  // slot-level margin >= every lane's is_ambiguous margin (monotone in cs); + the FP32 rounding
  // of |s|^2 itself (<= 4u * csk^2).  +inf if stage A hit nothing.
  const float margin = expanded_margin(csk, t.tmax);
  // reach_scale > 1 (sweep reuse): groups a little beyond the strict need are swept too, so that
  // every source learns a lower bound (reach) of its distance to all the groups NOT swept
  const float reach = sqrtf(fmaxf(ub2, 0.f) + 3.f * margin + csk * csk * 4.8e-7f) * 1.000004f * reach_scale;
  reach_out = reach;
  // ---- stage B: the remaining groups that can still matter
  for (int w = 0; w < words; ++w) {
    float d2, rr;
    if (w == 0) { d2 = d2w0; rr = rw0; }
    else if (w == 1) { d2 = d2w1; rr = rw1; }
    else {
      const int g = (w << 5) + lane;
      d2 = CUDART_INF_F; rr = 0.f;
      if (g < ngroups) {
        d2 = box_dist2(t.gcx[g], t.gcy[g], x0, x1, y0, y1) * 0.999996f;
        rr = t.grad[g] + slack;
      }
    }
    const float far = rr + reach;                          // +inf when stage A hit nothing
    const unsigned mask = __ballot_sync(kFull, (w << 5) + lane < ngroups && d2 > rr * rr && d2 <= far * far);
    evaluated += __popc(mask);
    eval_mask<S>(t, mask, w << 5, a, b, c, keep);
  }
  return evaluated;
}

// ------------------------------------------------------------------------------------
// kernel: the whole ICP loop, W WARPS PER PAIR, two phases per iteration (icp.py:28-53)
//
// Round-2 throughput kernel.  What bounded icp_align_warp_kernel was latency at 16 resident warps
// per SM (122 registers, 11.5 KB of shared memory per warp) and ~60 % of its instructions lying
// outside the candidate sweep.  This kernel
//   * gives a pair W warps that share ONE target tile (shared memory per warp drops by ~W/2) and is
//     compiled for 24 resident warps per SM (<= 80 registers): the search phase and the float64
//     phase no longer overlap in the register file --
//       phase 1 (search): per pass of 32*SC sources -> nearest target index, stored as uint16 in
//                shared memory; FP32 only (plus the rare float64 rescans);
//       phase 2 (update): every source: gather of its matched target, exact float64 distance,
//                the 11 centred sums; then warp shuffle + one shared-memory hop across the W warps,
//                closed-form pose, apply;
//   * extends the movement bound of the sweep reuse from "the group of 8 that holds the nearest
//     neighbour" to the nearest neighbour itself: a pass whose sources have all moved less than half
//     the gap between their nearest and their second-nearest target (lower bound of the in-group
//     runner-up and of everything outside the group) skips phase 1 ENTIRELY -- no set-up, no
//     culling, no in-group argmin -- and the iteration is gather + distance + sums only.
// Three levels per pass, decided from the running sum of the per-iteration maximum displacement
// (`cum_move`): cum_move <= tnn[pass]  -> indices kept;  <= tgrp[pass] -> in-group re-decision;
// else full (pruned or dense) sweep.  Every level yields the exact float64 nearest neighbour
// (lowest index on ties), so index histories are identical to the sweep-everything kernel.
// ------------------------------------------------------------------------------------
// Warp sums of ten per-lane doubles.  The xor butterfly (16, 8, 4, 2, 1) over all ten values costs
// 50 shuffle+add pairs; here every step lets a lane KEEP half of its values and SEND the other half
// to its partner, so the value count halves with the lane distance: 5 + 3 + 2 + 1 + 1 = 12 pairs.
// Each surviving partial is formed by exactly the additions the butterfly performs for that value
// (own + partner's, partner distances in the same order), so the sums carry the same bits.
// On return the lanes with fold10_owner(lane) = q >= 0 hold the warp sum of r[q].
__device__ __forceinline__ double warp_fold10(const double (&r)[11], int lane) {
  const bool s16 = lane & 16, s8 = lane & 8, s4 = lane & 4, s2 = lane & 2;
  double a[5], b[3], c[2];
#pragma unroll
  for (int q = 0; q < 5; ++q) {
    const double keep = s16 ? r[q + 5] : r[q], send = s16 ? r[q] : r[q + 5];
    a[q] = keep + __shfl_xor_sync(kFull, send, 16);
  }
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const double keep = s8 ? a[q + 3] : a[q], send = s8 ? a[q] : a[q + 3];
    b[q] = keep + __shfl_xor_sync(kFull, send, 8);
  }
  b[2] = a[2] + __shfl_xor_sync(kFull, a[2], 8);          // valid in the lanes that kept a[0..2]
  {
    const double keep = s4 ? b[2] : b[0], send = s4 ? b[0] : b[2];
    c[0] = keep + __shfl_xor_sync(kFull, send, 4);
  }
  c[1] = b[1] + __shfl_xor_sync(kFull, b[1], 4);          // valid in the lanes that kept b[0..1]
  const double keep = s2 ? c[1] : c[0], send = s2 ? c[0] : c[1];
  double d = keep + __shfl_xor_sync(kFull, send, 2);
  d += __shfl_xor_sync(kFull, d, 1);
  return d;
}
__device__ __forceinline__ int fold10_owner(int lane) {
  const int b4 = (lane >> 4) & 1, b3 = (lane >> 3) & 1, b2 = (lane >> 2) & 1, b1 = (lane >> 1) & 1;
  const bool valid = !(lane & 1) && !(b3 & b2) && !(b2 & b1);
  return valid ? 5 * b4 + 3 * b3 + 2 * b2 + b1 : -1;
}

struct PairCtx {            // shared memory; touched by thread 0 only until the final barrier
  double R[4], T[2];        // cumulative pose, src = R A + T
  double last[4];           // last increment: cos, sin, tx, ty
  double err, mean_d2;
  int iters, inl;
  unsigned long long evals; // pair evaluations executed by the sweeps of all warps
};
static_assert(sizeof(PairCtx) <= kCtxBytes, "PairCtx outgrew its shared-memory slot");

constexpr int kPairRedStride = 12;   // doubles per warp slot of the cross-warp reduction

constexpr int kPairMaxPasses = 16;    // 1,024 sources / 64: the threshold arrays have a fixed size

// Shared-memory layout of a pair: everything of fixed size first (PairCtx, reduction slots, the
// per-pass thresholds), so that with W a template parameter their addresses are immediates; then the
// source state, the target tile, the group circles and the per-source indices.
__host__ __device__ inline size_t pair_tile_bytes(int mcap, int ncap, int passes, int warps) {
  (void)passes;
  size_t b = kCtxBytes + (size_t)2 * warps * kPairRedStride * sizeof(double) +
             (size_t)2 * kPairMaxPasses * sizeof(float) + (size_t)ncap * sizeof(double2) +
             (size_t)mcap * 3 * sizeof(float) + (size_t)(mcap / kGroup) * 3 * sizeof(float) +
             (size_t)ncap * 2 * sizeof(unsigned short);
  return (b + 15) & ~(size_t)15;
}

struct PairTile : WarpTile {
  unsigned short* nnidx;    // [ncap] nearest target of every source at its last search
  unsigned short* grp2;     // [ncap] the OTHER group of the source's candidate pair (= its own group if alone)
  unsigned keep;            // mantissa bits a packed sweep key keeps: ~((1 << log2ceil(groups)) - 1)
  float* tgrp;              // [passes] cum_move up to which the sources of a pass keep their GROUP
  float* tnn;               // [passes] ... keep their nearest neighbour
  double* red;              // [2][W][kPairRedStride]
};

__device__ __forceinline__ void carve_pair_tile(unsigned char* smem, const KernelArgs& a, int warps,
                                                PairTile& t, PairCtx*& ctx) {
  t.mcap = a.mcap;
  ctx = reinterpret_cast<PairCtx*>(smem);
  t.red = reinterpret_cast<double*>(smem + kCtxBytes);
  t.tgrp = reinterpret_cast<float*>(t.red + 2 * warps * kPairRedStride);
  t.tnn = t.tgrp + kPairMaxPasses;
  t.src = reinterpret_cast<double2*>(t.tnn + kPairMaxPasses);
  t.tile = reinterpret_cast<float*>(t.src + a.ncap);
  t.gcx = t.tile + 3 * a.mcap;
  t.gcy = t.gcx + a.mcap / kGroup;
  t.grad = t.gcy + a.mcap / kGroup;
  t.nnidx = reinterpret_cast<unsigned short*>(t.grad + a.mcap / kGroup);
  t.grp2 = t.nnidx + a.ncap;
  unsigned bits = 1;
  while ((1u << bits) < (unsigned)(a.mcap / kGroup)) ++bits;
  t.keep = ~((1u << bits) - 1u);
  t.grp = nullptr; t.tpass = nullptr; t.grp16 = false;
}

// CTA-cooperative version of warp_stage_targets (same tile contents for a given origin).
template <int W>
__device__ __forceinline__ void pair_stage_targets(PairTile& t, int tid, int lane, int warp) {
  constexpr int NT = 32 * W;
  double sx = 0.0, sy = 0.0;
  for (int j = tid; j < t.m; j += NT) {
    const double2 q = load_point(t.tgt, t.dtype, t.row_off + j);
    sx += q.x; sy += q.y;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sx += __shfl_xor_sync(kFull, sx, o);
    sy += __shfl_xor_sync(kFull, sy, o);
  }
  if (W > 1) {
    if (lane == 0) { t.red[warp * kPairRedStride] = sx; t.red[warp * kPairRedStride + 1] = sy; }
    __syncthreads();
    sx = t.red[0]; sy = t.red[1];
#pragma unroll
    for (int w = 1; w < W; ++w) { sx += t.red[w * kPairRedStride]; sy += t.red[w * kPairRedStride + 1]; }
  }
  t.ox = sx / (double)t.m;
  t.oy = sy / (double)t.m;
  float amax = 0.f;
  for (int j = tid; j < t.mcap; j += NT) {
    float cx = 1e18f, cy = 1e18f, tt = CUDART_INF_F;        // sentinels: see warp_stage_targets
    if (j < t.m) {
      const double2 q = load_point(t.tgt, t.dtype, t.row_off + j);
      cx = (float)(q.x - t.ox); cy = (float)(q.y - t.oy);
      tt = (float)((double)cx * (double)cx + (double)cy * (double)cy);
      amax = fmaxf(amax, fmaxf(fabsf(cx), fabsf(cy)));
    }
    float* gq = t.tile + (j >> 3) * 24 + (j & 7);
    gq[0] = cx; gq[8] = cy; gq[16] = tt;
  }
  amax = warp_max_f32(amax);
  if (W > 1) {
    // second buffer of the reduction scratch: the first may still be read by a slower warp
    float* fm = reinterpret_cast<float*>(t.red + W * kPairRedStride);
    if (lane == 0) fm[warp] = amax;
    __syncthreads();                                         // also publishes the tile
    amax = fm[0];
#pragma unroll
    for (int w = 1; w < W; ++w) amax = fmaxf(amax, fm[w]);
  } else {
    __syncwarp();
  }
  t.tmax = amax;
  for (int g = tid; g < t.ngroups; g += NT) {                // bounding circle of every group
    float x0 = CUDART_INF_F, x1 = -CUDART_INF_F, y0 = CUDART_INF_F, y1 = -CUDART_INF_F;
    for (int u = 0; u < kGroup; ++u) {
      if (g * kGroup + u < t.m) {
        const float px = t.tile[g * 24 + u], py = t.tile[g * 24 + 8 + u];
        x0 = fminf(x0, px); x1 = fmaxf(x1, px);
        y0 = fminf(y0, py); y1 = fmaxf(y1, py);
      }
    }
    const float cx = 0.5f * (x0 + x1), cy = 0.5f * (y0 + y1);
    float r2 = 0.f;
    for (int u = 0; u < kGroup; ++u) {
      if (g * kGroup + u < t.m) {
        const float dx = t.tile[g * 24 + u] - cx, dy = t.tile[g * 24 + 8 + u] - cy;
        r2 = fmaxf(r2, fmaf(dx, dx, dy * dy));
      }
    }
    t.gcx[g] = cx; t.gcy[g] = cy;
    t.grad[g] = sqrtf(r2) * 1.000004f + 1e-30f;
  }
}

// The exact decision inside the (up to) two candidate groups of a source: FP32 direct-difference
// distances of their 16 targets, the slot number packed into the low mantissa byte (relative
// perturbation <= 2^-15, covered by kUpD), so the argmin and the runner-up are plain min/max
// chains.  Returns the winning slot (0..7: group ga, 8..15: group gb), whether a runner-up lies
// inside the FP32 guard band (-> float64 rescan), `ubd` >= the exact distance from the source to
// the winner and `los` <= the exact distance to every other target of the two groups.
// (smallest, second smallest) of two such pairs: three operations (min, max, 3-input min).
__device__ __forceinline__ void merge_two_smallest(unsigned& lo, unsigned& hi, unsigned lo2, unsigned hi2) {
  const unsigned m = max(lo, lo2);
  lo = min(lo, lo2);
  hi = min(min(hi, hi2), m);
}

__device__ __forceinline__ int in_group_decide(const WarpTile& t, int ga, int gb, bool two, float fx, float fy,
                                               bool& near_tie, float& ubd, float& los) {
  const float2 ny = make_float2(-fy, -fy);
  unsigned best = 0x7f800000u, second = 0x7f800000u;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    // no second group: its targets are evaluated from 1e18 away (d ~ 1e36, finite also for the
    // sentinels at +1e18): they never win and never come near the winner
    const float hx = (h == 1 && !two) ? 1e18f : -fx;
    const float2 nx = make_float2(hx, hx);
    const float4* __restrict__ g4 = reinterpret_cast<const float4*>(t.tile) + 6 * (h ? gb : ga);
    const float4 xa = g4[0], xb = g4[1];
    const float4 ya = g4[2], yb = g4[3];
    const float2 u0 = __fadd2_rn(make_float2(xa.x, xa.y), nx), v0 = __fadd2_rn(make_float2(ya.x, ya.y), ny);
    const float2 u1 = __fadd2_rn(make_float2(xa.z, xa.w), nx), v1 = __fadd2_rn(make_float2(ya.z, ya.w), ny);
    const float2 u2 = __fadd2_rn(make_float2(xb.x, xb.y), nx), v2 = __fadd2_rn(make_float2(yb.x, yb.y), ny);
    const float2 u3 = __fadd2_rn(make_float2(xb.z, xb.w), nx), v3 = __fadd2_rn(make_float2(yb.z, yb.w), ny);
    const float2 d01 = __ffma2_rn(v0, v0, __fmul2_rn(u0, u0)), d23 = __ffma2_rn(v1, v1, __fmul2_rn(u1, u1));
    const float2 d45 = __ffma2_rn(v2, v2, __fmul2_rn(u2, u2)), d67 = __ffma2_rn(v3, v3, __fmul2_rn(u3, u3));
    const float ds[8] = {d01.x, d01.y, d23.x, d23.y, d45.x, d45.y, d67.x, d67.y};   // sentinels: ~2e36
    unsigned key[8];
    // one PRMT per key: the slot number replaces the low mantissa BYTE (two registers hold the eight
    // slot bytes; the group bit is or-ed into the two survivors of the group's tournament).  d >= 0:
    // the bit patterns are ordered like the values
    const unsigned slots_lo = 0x03020100u, slots_hi = 0x07060504u;
#pragma unroll
    for (int u = 0; u < kGroup; ++u)
      key[u] = __byte_perm(__float_as_uint(ds[u]), u < 4 ? slots_lo : slots_hi, 0x3214u + (unsigned)(u & 3));
    // tournament instead of a 16-long dependent min/max chain: 17 operations per group, depth 4
    unsigned lo[4], hi[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) { lo[u] = min(key[2 * u], key[2 * u + 1]); hi[u] = max(key[2 * u], key[2 * u + 1]); }
    merge_two_smallest(lo[0], hi[0], lo[1], hi[1]);
    merge_two_smallest(lo[2], hi[2], lo[3], hi[3]);
    merge_two_smallest(lo[0], hi[0], lo[2], hi[2]);
    if (h == 1) { lo[0] |= 8u; hi[0] |= 8u; }
    merge_two_smallest(best, second, lo[0], hi[0]);
  }
  // the keys lost their low mantissa byte: d^2 is known to 2^-15, d to 2^-16 (1.53e-5) relative
  const float bd = __uint_as_float(best & ~255u), sd = __uint_as_float(second & ~255u);
  constexpr float kUpD = 1.00002f;
  const float cs = fmaxf(fabsf(fx), fabsf(fy));
  const float guard = (cs + t.tmax) * 4.76837158e-7f;                // 2^-21 (cs + tmax)
  ubd = sqrtf(bd) * kUpD + guard;
  near_tie = sd <= ubd * ubd * 1.000001f;
  los = sqrtf(sd) * 0.999996f - guard;
  return (int)(best & 15u);
}

// Phase 1 for one pass: the exact nearest target of the SC sources (base + k*32 + lane) of every
// lane -> t.nnidx, and the other group of its candidate pair -> t.grp2.  `reuse_grp`: no sweep,
// re-decide inside the two stored groups.  bud_grp / bud_nn (identical in every lane on return):
// how far the sources of this pass may move before the nearest neighbour of one of them can leave
// its two groups / change at all; <= 0 means "no bound".
template <int SC, bool PRUNE>
__device__ __forceinline__ long long pair_search_pass(const PairTile& t, int base, int n, int m, int lane,
                                                      bool reuse_grp, bool track, float& bud_grp,
                                                      float& bud_nn) {
  long long evals = 0;
  float fx[SC], fy[SC], lbg[SC];
  int ga[SC], gb[SC];
  bool two[SC], amb3[SC];
#pragma unroll
  for (int k = 0; k < SC; ++k) {
    const double2 s = t.src[base + k * 32 + lane];
    fx[k] = (float)(s.x - t.ox); fy[k] = (float)(s.y - t.oy);
    lbg[k] = -1.f;
    amb3[k] = false;
  }
  if (reuse_grp) {
#pragma unroll
    for (int k = 0; k < SC; ++k) {
      const int i = base + k * 32 + lane;
      ga[k] = i < n ? (int)(t.nnidx[i] >> 3) : 0;
      gb[k] = i < n ? (int)t.grp2[i] : 0;
      two[k] = gb[k] != ga[k];                           // a lone group is stored twice
    }
  } else {
    Cand3<SC> c;
    const unsigned keep = t.keep;
    if (PRUNE) {
      bool vld[SC];
#pragma unroll
      for (int k = 0; k < SC; ++k) vld[k] = base + k * 32 + lane < n;
      float reach;
      const int groups = warp_candidates_pruned<SC>(t, fx, fy, vld, c, keep, track ? 2.0f : 1.0f, reach);
      evals += (long long)groups * kGroup * min(32 * SC, n - base);
      if (track) {
#pragma unroll
        for (int k = 0; k < SC; ++k) lbg[k] = reach * 0.999996f;
      }
    } else {
      warp_candidates<SC>(t, fx, fy, c, keep);
      evals += (long long)t.ngroups * kGroup * min(32 * SC, n - base);
      if (track) {
#pragma unroll
        for (int k = 0; k < SC; ++k) lbg[k] = CUDART_INF_F;
      }
    }
#pragma unroll
    for (int k = 0; k < SC; ++k) {
      const float cs = fmaxf(fabsf(fx[k]), fabsf(fy[k]));
      const float ek = key_eps(cs, t.tmax, keep);
      const float margin = expanded_margin(cs, t.tmax);
      ga[k] = (int)(__float_as_uint(c.kb[k]) & ~keep);
      two[k] = c.ks[k] < CUDART_INF_F;
      gb[k] = two[k] ? (int)(__float_as_uint(c.ks[k]) & ~keep) : ga[k];
      // a THIRD group inside the error band of the best: the nearest neighbour may lie outside the
      // two candidates -> float64 rescan of all targets (near-equal floats subtract exactly)
      amb3[k] = (c.kt[k] - c.kb[k]) <= margin + 2.f * ek;
      if (track) {
        // every group but the two candidates: d^2 >= third + |s|^2 - (FP32 error of the expanded
        // form, of |s|^2 and of the packed key)
        const float ss = fmaf(fx[k], fx[k], fy[k] * fy[k]);
        const float lo2 = (c.kt[k] + ss) - (2.f * margin + cs * cs * 4.8e-7f + ek);
        lbg[k] = fminf(lbg[k], sqrtf(fmaxf(lo2, 0.f)) * 0.999996f);
      }
    }
  }
  int j[SC], other[SC];
  bool amb[SC];
  bool any_amb = false;
  float bg = CUDART_INF_F, bn = CUDART_INF_F;
#pragma unroll
  for (int k = 0; k < SC; ++k) {
    bool tie_in;
    float ubd, los;
    const int slot = in_group_decide(t, ga[k], gb[k], two[k], fx[k], fy[k], tie_in, ubd, los);
    j[k] = (slot < 8 ? ga[k] : gb[k]) * kGroup + (slot & 7);
    other[k] = slot < 8 ? gb[k] : ga[k];
    const bool valid = base + k * 32 + lane < n;
    amb[k] = valid && (tie_in || amb3[k]);
    any_amb |= amb[k];
    if (valid) {
      // an ambiguous source is re-decided in float64 below: no FP32 bound describes that decision
      bn = fminf(bn, amb[k] ? -1.f : 0.5f * (los - ubd));
      bg = fminf(bg, amb[k] ? -1.f : 0.5f * (lbg[k] - ubd));
    }
  }
  if (__any_sync(kFull, any_amb)) {      // rare: warp-cooperative float64 scan of all targets
#pragma unroll
    for (int k = 0; k < SC; ++k) {
      unsigned pending = __ballot_sync(kFull, amb[k]);
      if (!pending) continue;
      const double2 s = t.src[base + k * 32 + lane];
      int jk = j[k];
      while (pending) {
        const int owner = __ffs(pending) - 1;
        pending &= pending - 1;
        const double qx = __shfl_sync(kFull, s.x, owner), qy = __shfl_sync(kFull, s.y, owner);
        double ld = CUDART_INF;
        int lj = 0x7fffffff;
        for (int jj = lane; jj < m; jj += 32) {
          const double d = dist2_f64(qx, qy, load_point(t.tgt, t.dtype, t.row_off + jj));
          if (d < ld) { ld = d; lj = jj; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const double od = __shfl_xor_sync(kFull, ld, o);
          const int oj = __shfl_xor_sync(kFull, lj, o);
          if (od < ld || (od == ld && oj < lj)) { ld = od; lj = oj; }
        }
        if (lane == owner) jk = lj;
      }
      if (amb[k]) {                                      // keep (winner's group, one of the old candidates)
        const int gj = jk >> 3;
        other[k] = gj == ga[k] ? gb[k] : ga[k];
      }
      j[k] = jk;
    }
  }
#pragma unroll
  for (int k = 0; k < SC; ++k) {
    const int i = base + k * 32 + lane;
    if (i < n) { t.nnidx[i] = (unsigned short)j[k]; t.grp2[i] = (unsigned short)other[k]; }
  }
  bud_nn = warp_min_f32(bn);
  bud_grp = (track && !reuse_grp) ? warp_min_f32(bg) : -1.f;
  return evals;
}

#ifndef B200ICP_PAIR_RESIDENT_WARPS
#define B200ICP_PAIR_RESIDENT_WARPS 24      // resident warps per SM the kernel is compiled for (register cap)
#endif
// LEAN: float32 tables, no gate, no per-point index outputs (the throughput configuration): the
// float64 phase is compiled without the corresponding tests and without the inlier count.
template <int SC, bool PRUNE, int W, bool LEAN>
__global__ void __launch_bounds__(32 * W, (PRUNE ? B200ICP_PAIR_RESIDENT_WARPS : 16) / W)
icp_align_pair_kernel(const KernelArgs a) {      // (the dense sweep holds 6 sources per lane: 128 registers, 16 warps)
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int NT = 32 * W;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t p = blockIdx.x;
  const b200icp_problem& pr = a.prob;
  const b200icp_options& op = a.opt;
  const b200icp_outputs& out = a.out;

  int64_t srow, trow;
  resolve_rows(pr, p, srow, trow);
  const int n = pr.src_len ? min(pr.src_len[srow], pr.src_pitch) : pr.src_pitch;
  const int m = pr.tgt_len ? min(pr.tgt_len[trow], pr.tgt_pitch) : pr.tgt_pitch;

  PairTile t;
  PairCtx* ctx;
  carve_pair_tile(smem_raw, a, W, t, ctx);
  t.tgt = pr.tgt_points; t.row_off = trow * pr.tgt_pitch; t.dtype = LEAN ? (int)B200ICP_F32 : pr.dtype;
  t.m = m; t.ngroups = (m + kGroup - 1) / kGroup;

  const bool ran = n > 0 && m > 0 && op.max_iterations > 0;
  if (tid == 0) {
    double R00 = 1.0, R01 = 0.0, R10 = 0.0, R11 = 1.0, T0 = 0.0, T1 = 0.0;
    if (op.init_pose) {
      const double* ip = op.init_pose + p * 6;
      R00 = ip[0]; R01 = ip[1]; R10 = ip[2]; R11 = ip[3]; T0 = ip[4]; T1 = ip[5];
    }
    ctx->R[0] = R00; ctx->R[1] = R01; ctx->R[2] = R10; ctx->R[3] = R11;
    ctx->T[0] = T0; ctx->T[1] = T1;
    ctx->last[0] = 1.0; ctx->last[1] = 0.0; ctx->last[2] = 0.0; ctx->last[3] = 0.0;
    ctx->err = CUDART_INF; ctx->mean_d2 = CUDART_INF;
    ctx->iters = 0; ctx->inl = 0; ctx->evals = 0ull;
  }
  for (int q = tid; q < a.passes; q += NT) { t.tgrp[q] = -CUDART_INF_F; t.tnn[q] = -CUDART_INF_F; }
  if (W > 1) __syncthreads(); else __syncwarp();
  int32_t* idx_out = (!LEAN && out.indices) ? out.indices + p * pr.src_pitch : nullptr;
  long long evals = 0;

  if (ran) {
    pair_stage_targets<W>(t, tid, lane, warp);
    float smax = 0.f;          // bound of |s - c| over the source points, c = target centroid
    for (int i = tid; i < a.ncap; i += NT) {
      double2 v = make_double2(t.ox, t.oy);                // padding slots: benign, never used
      if (i < n) {
        const double2 q = load_point(pr.src_points, t.dtype, srow * pr.src_pitch + i);
        v = q;                                             // icp.py:32  src = copy(A)
        if (op.init_pose)
          v = make_double2(ctx->R[0] * q.x + ctx->R[1] * q.y + ctx->T[0],
                           ctx->R[2] * q.x + ctx->R[3] * q.y + ctx->T[1]);
        smax = fmaxf(smax, fmaxf(__double2float_ru(fabs(v.x - t.ox)), __double2float_ru(fabs(v.y - t.oy))));
      }
      t.src[i] = v;
    }
    smax = warp_max_f32(smax);
    if (W > 1) {
      float* fm = reinterpret_cast<float*>(t.red);        // first buffer: free again after the staging barriers
      if (lane == 0) fm[warp] = smax;
      __syncthreads();                                     // also publishes src and the group circles
      smax = fm[0];
#pragma unroll
      for (int w = 1; w < W; ++w) smax = fmaxf(smax, fm[w]);
      __syncthreads();                                     // fm is reduction scratch from now on
    } else {
      __syncwarp();
    }
    smax *= 1.4142137f;
    float mv_prev = CUDART_INF_F;      // displacement bound of the previous update
    double prev_error = 0.0;           // icp.py:33
    double cum_move = 0.0;             // sum of the per-iteration displacement bounds
    const bool use_gate = !LEAN && a.use_gate != 0;
    const double inv_n = 1.0 / (double)n;

    for (int it = 0; it < op.max_iterations; ++it) {       // icp.py:35
      // ---- phase 1: correspondence search (icp.py:37-38), only where the movement bound demands it
      // every sweep also yields the bounds of the reuse (the two-group budget usually survives even
      // the large moves of the first iterations)
      const bool track = a.reuse != 0;
      // which of this warp's passes need a search: one threshold per lane, one ballot (a pass is
      // searched and its thresholds are written by the same warp in every iteration)
      const float cm = __double2float_ru(cum_move);
      unsigned need;
      {
        const bool own = lane < a.passes && lane % W == warp && lane * (32 * SC) < n;
        need = __ballot_sync(kFull, own && !(track && cm <= t.tnn[own ? lane : 0]));
      }
      while (need) {
        const int pass = __ffs(need) - 1;
        need &= need - 1;
        const int base = pass * 32 * SC;
        const bool reuse_grp = track && cm <= t.tgrp[pass];
        float bud_grp, bud_nn;
        evals += pair_search_pass<SC, PRUNE>(t, base, n, m, lane, reuse_grp, track, bud_grp, bud_nn);
        if (track && lane == 0) {
          if (!reuse_grp)
            t.tgrp[pass] = bud_grp > 0.f ? __double2float_rd(cum_move + 0.999 * (double)bud_grp) : -CUDART_INF_F;
          t.tnn[pass] = bud_nn > 0.f ? fminf(t.tgrp[pass], __double2float_rd(cum_move + 0.999 * (double)bud_nn))
                                     : -CUDART_INF_F;
        }
      }
      __syncwarp();
      // ---- phase 2: gather (icp.py:39), exact distances, ONE set of centred sums
      int32_t* hist = (!LEAN && out.index_history)
          ? out.index_history + (p * op.max_iterations + it) * (int64_t)pr.src_pitch : nullptr;
      double r[11] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
      // Sources are summed in blocks of 64 dealt round-robin to the warps, whatever the pass width of
      // the search: the float64 sums -- and with them every bit of the result -- do not depend on
      // SC / PRUNE (the dense and the pruned kernels are interchangeable bit for bit).
      if (SC != 2 && W > 1) __syncthreads();               // indices written by another warp's pass
      for (int base = warp * 64; base < n; base += W * 64) {
        {
          constexpr int k0 = 0;
          if (LEAN && base + (k0 + 2) * 32 <= n) {
            // both 32-source slots are full (warp-uniform test): straight-line code, no per-lane tests
            int jj[2];
            double2 bm[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              jj[u] = (int)t.nnidx[base + (k0 + u) * 32 + lane];
              bm[u] = load_point(t.tgt, B200ICP_F32, t.row_off + jj[u]);
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              const double2 s = t.src[base + (k0 + u) * 32 + lane];
              const double2 b = bm[u];
              const double d2 = dist2_f64(s.x, s.y, b);
              const double dist = sqrt_f64_fast(d2);
              const double ax = s.x - t.ox, ay = s.y - t.oy;
              const double qx = b.x - t.ox, qy = b.y - t.oy;
              r[0] += ax; r[1] += ay; r[2] += qx; r[3] += qy;
              r[4] = fma(ax, qx, r[4]); r[5] = fma(ax, qy, r[5]);
              r[6] = fma(ay, qx, r[6]); r[7] = fma(ay, qy, r[7]);
              r[8] += dist; r[9] += d2;
            }
            continue;
          }
          int jj[2];
          double2 bm[2];
#pragma unroll
          for (int u = 0; u < 2; ++u) {                    // both loads in flight before the first use
            const int i = base + (k0 + u) * 32 + lane;
            jj[u] = i < n ? (int)t.nnidx[i] : 0;
            bm[u] = load_point(t.tgt, t.dtype, t.row_off + jj[u]);
          }
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int i = base + (k0 + u) * 32 + lane;
            if (i < n) {
              const double2 s = t.src[i];
              const double2 b = bm[u];
              const double d2 = dist2_f64(s.x, s.y, b);
              const double dist = sqrt_f64_fast(d2);
              if (!use_gate || dist < op.max_corr_dist) {
                const double ax = s.x - t.ox, ay = s.y - t.oy;
                const double qx = b.x - t.ox, qy = b.y - t.oy;
                r[0] += ax; r[1] += ay; r[2] += qx; r[3] += qy;
                r[4] = fma(ax, qx, r[4]); r[5] = fma(ax, qy, r[5]);
                r[6] = fma(ay, qx, r[6]); r[7] = fma(ay, qy, r[7]);
                r[8] += dist; r[9] += d2;
                if (!LEAN) r[10] += 1.0;
              }
              if (idx_out) idx_out[i] = jj[u];
              if (hist) hist[i] = jj[u];
            }
          }
        }
      }
      constexpr int NR = LEAN ? 10 : 11;                   // LEAN: no gate, the inlier count is n
      {         // warp sums, then one hop across the warps; every thread adds the partials in warp order
        const double mine = warp_fold10(r, lane);
        if (!LEAN) {
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) r[10] += __shfl_xor_sync(kFull, r[10], o);
        }
        double* slot = t.red + ((it & 1) * W + warp) * kPairRedStride;
        const int q = fold10_owner(lane);
        if (q >= 0) slot[q] = mine;
        if (!LEAN && lane == 0) slot[10] = r[10];
        if (W > 1) __syncthreads(); else __syncwarp();
        const double2* part = reinterpret_cast<const double2*>(t.red + (it & 1) * W * kPairRedStride);
#pragma unroll
        for (int q2 = 0; q2 < (NR + 1) / 2; ++q2) {
          double2 acc = part[q2];
#pragma unroll
          for (int w = 1; w < W; ++w) {
            const double2 o = part[w * (kPairRedStride / 2) + q2];
            acc.x += o.x; acc.y += o.y;
          }
          r[2 * q2] = acc.x;
          if (2 * q2 + 1 < 11) r[2 * q2 + 1] = acc.y;
        }
      }
      const double cnt = LEAN ? (double)n : r[10];
      if (cnt < 0.5) {            // every correspondence gated out: stop, search not counted
        if (tid == 0) { ctx->err = CUDART_INF; ctx->mean_d2 = CUDART_INF; ctx->inl = 0; }
        if (hist) for (int i = tid; i < n; i += NT) hist[i] = -1;
        break;
      }
      const double inv = use_gate ? 1.0 / cnt : inv_n;
      const double max_ = r[0] * inv, may_ = r[1] * inv;       // centroids rel. origin (icp.py:10-11)
      const double mbx = r[2] * inv, mby = r[3] * inv;
      const double mean_error = r[8] * inv;                    // icp.py:48
      // closed-form 2D Kabsch: the proper rotation the SVD route (icp.py:17-23) returns
      const double h00 = fma(-r[0], mbx, r[4]), h01 = fma(-r[0], mby, r[5]);
      const double h10 = fma(-r[1], mbx, r[6]), h11 = fma(-r[1], mby, r[7]);
      const double num = h01 - h10, den = h00 + h11;
      const double h2 = fma(num, num, den * den);
      double cs = 1.0, sn = 0.0;
      if (h2 > 0.0) {
        const double rh = rsqrt(h2);
        cs = den * rh; sn = num * rh;
      }
      const double cax = t.ox + max_, cay = t.oy + may_;
      const double tx = (t.ox + mbx) - (cs * cax - sn * cay);  // icp.py:25
      const double ty = (t.oy + mby) - (sn * cax + cs * cay);
      for (int base = warp * 64; base < n; base += W * 64) {   // apply (icp.py:45), the blocks this warp summed
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const int i = base + k * 32 + lane;
          if (i < n) {
            const double2 s = t.src[i];
            t.src[i] = make_double2(cs * s.x - sn * s.y + tx, sn * s.x + cs * s.y + ty);
          }
        }
      }
      if (SC != 2 && W > 1) __syncthreads();               // the next search reads points another warp moved
      // Upper bound of every point's displacement in this update: with c the target centroid,
      // s' - s = (R - I)(s - c) + [(R - I) c + t], so |s' - s| <= |R - I| smax + |(R - I) c + t| with
      // |R - I| = sqrt((cos - 1)^2 + sin^2) and smax >= |s - c| for every point (initial maximum, grown
      // by every bound since).  The two small vectors are formed in float64 (cancellation), their
      // norms in float32 and inflated by 1e-5 (a bound need not be tight), plus the rounding of
      // the update itself (a few float64 ulp of the coordinates).  Identical in every thread.
      float mv = 0.f;
      if (a.reuse) {
        const double c1 = cs - 1.0;
        const float c1f = (float)c1, snf = (float)sn;
        const float ddx = (float)(fma(c1, t.ox, -sn * t.oy) + tx), ddy = (float)(fma(sn, t.ox, c1 * t.oy) + ty);
        const float rho = sqrtf(fmaf(c1f, c1f, snf * snf)), dd = sqrtf(fmaf(ddx, ddx, ddy * ddy));
        const float ulp = 1.0e-15f * (fabsf((float)t.ox) + fabsf((float)t.oy) + smax + fabsf((float)tx) + fabsf((float)ty));
        mv = fmaf(rho, smax, dd) * 1.00001f + ulp + 1e-30f;
        smax = __fadd_ru(smax, mv);
        mv_prev = mv;
        cum_move += (double)mv * 1.000001;
      }
      const bool converged = fabs(prev_error - mean_error) < op.tolerance;   // icp.py:49-50
      prev_error = mean_error;                                               // icp.py:51
      if (tid == 0) {            // compose the cumulative pose, record the increment
        const double R00 = ctx->R[0], R01 = ctx->R[1], R10 = ctx->R[2], R11 = ctx->R[3];
        const double T0 = ctx->T[0], T1 = ctx->T[1];
        ctx->R[0] = cs * R00 - sn * R10; ctx->R[1] = cs * R01 - sn * R11;
        ctx->R[2] = sn * R00 + cs * R10; ctx->R[3] = sn * R01 + cs * R11;
        ctx->T[0] = cs * T0 - sn * T1 + tx; ctx->T[1] = sn * T0 + cs * T1 + ty;
        ctx->last[0] = cs; ctx->last[1] = sn; ctx->last[2] = tx; ctx->last[3] = ty;
        ctx->err = mean_error; ctx->mean_d2 = r[9] * inv; ctx->inl = (int)(cnt + 0.5);
        ctx->iters = it + 1;
      }
      __syncwarp();
      if (converged) break;
    }
  }

  if (out.evaluated_pairs && lane == 0 && evals) atomicAdd(&ctx->evals, (unsigned long long)evals);
  if (W > 1) __syncthreads(); else __syncwarp();
  const int iters = ctx->iters;
  if (tid == 0) {
    double* pt = out.pose_total + p * 6;
    pt[0] = ctx->R[0]; pt[1] = ctx->R[1]; pt[2] = ctx->R[2]; pt[3] = ctx->R[3];
    pt[4] = ctx->T[0]; pt[5] = ctx->T[1];
    if (out.pose_last) {
      double* pl = out.pose_last + p * 6;
      pl[0] = ctx->last[0]; pl[1] = -ctx->last[1]; pl[2] = ctx->last[1]; pl[3] = ctx->last[0];
      pl[4] = ctx->last[2]; pl[5] = ctx->last[3];
    }
    out.error[p] = ctx->err;
    if (out.rmse) out.rmse[p] = sqrt(ctx->mean_d2);
    if (out.inliers) out.inliers[p] = ctx->inl;
    out.iterations[p] = iters;
    if (out.evaluated_pairs) out.evaluated_pairs[p] = (int64_t)ctx->evals;
  }
  if (idx_out) {
    for (int i = tid; i < pr.src_pitch; i += NT)
      if (i >= n || iters == 0) idx_out[i] = -1;
  }
  if (out.src_final) {
    double2* dst = reinterpret_cast<double2*>(out.src_final) + p * pr.src_pitch;
    for (int i = tid; i < pr.src_pitch; i += NT) {
      double2 v = make_double2(0.0, 0.0);
      if (i < n) {
        if (ran) {
          v = t.src[i];
        } else {         // nothing ran: report the (pre-transformed) input
          const double2 q = load_point(pr.src_points, pr.dtype, srow * pr.src_pitch + i);
          v = make_double2(ctx->R[0] * q.x + ctx->R[1] * q.y + ctx->T[0],
                           ctx->R[2] * q.x + ctx->R[3] * q.y + ctx->T[1]);
        }
      }
      dst[i] = v;
    }
  }
}

// ------------------------------------------------------------------------------------
// kernel: correspondence search only, one warp per pair (icp.py:37-38): the tile, sweep and exact
// re-decision of the fused loop (phase 1), one search, outputs idx and the exact float64 d^2.
// ------------------------------------------------------------------------------------
template <int SC, bool PRUNE>
__global__ void __launch_bounds__(32, B200ICP_PAIR_RESIDENT_WARPS) nn_warp_kernel(const KernelArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int lane = threadIdx.x;
  const int64_t p = blockIdx.x;
  const b200icp_problem& pr = a.prob;
  int64_t srow, trow;
  resolve_rows(pr, p, srow, trow);
  const int n = pr.src_len ? min(pr.src_len[srow], pr.src_pitch) : pr.src_pitch;
  const int m = pr.tgt_len ? min(pr.tgt_len[trow], pr.tgt_pitch) : pr.tgt_pitch;
  int32_t* idx_out = a.nn_idx + p * pr.src_pitch;
  double* d2_out = a.nn_dist2 ? a.nn_dist2 + p * pr.src_pitch : nullptr;
  if (n <= 0 || m <= 0) {
    for (int i = lane; i < pr.src_pitch; i += 32) {
      idx_out[i] = -1;
      if (d2_out) d2_out[i] = CUDART_INF;
    }
    return;
  }
  PairTile t;
  PairCtx* ctx;
  carve_pair_tile(smem_raw, a, 1, t, ctx);
  t.tgt = pr.tgt_points; t.row_off = trow * pr.tgt_pitch; t.dtype = pr.dtype;
  t.m = m; t.ngroups = (m + kGroup - 1) / kGroup;
  pair_stage_targets<1>(t, lane, lane, 0);
  for (int i = lane; i < a.ncap; i += 32)
    t.src[i] = i < n ? load_point(pr.src_points, pr.dtype, srow * pr.src_pitch + i) : make_double2(t.ox, t.oy);
  __syncwarp();
  for (int base = 0; base < n; base += 32 * SC) {
    float bud_grp, bud_nn;
    pair_search_pass<SC, PRUNE>(t, base, n, m, lane, false, false, bud_grp, bud_nn);
    __syncwarp();
#pragma unroll
    for (int k = 0; k < SC; ++k) {
      const int i = base + k * 32 + lane;
      if (i < n) {
        const int j = (int)t.nnidx[i];
        idx_out[i] = j;
        if (d2_out) {
          const double2 s = t.src[i];
          d2_out[i] = dist2_f64(s.x, s.y, load_point(t.tgt, t.dtype, t.row_off + j));
        }
      }
    }
  }
  for (int i = n + lane; i < pr.src_pitch; i += 32) {
    idx_out[i] = -1;
    if (d2_out) d2_out[i] = CUDART_INF;
  }
}

// ------------------------------------------------------------------------------------
// kernel: best_fit_transform(A, B) for matched rows (icp.py:5-26), one warp per pair:
// centroids, centred 2x2 cross-covariance (single pass, each cloud relative to its first point),
// closed-form proper rotation, t = cB - R cA.
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) best_fit_warp_kernel(const KernelArgs a) {
  const int lane = threadIdx.x;
  const int64_t p = blockIdx.x;
  const b200icp_problem& pr = a.prob;
  int64_t srow, trow;
  resolve_rows(pr, p, srow, trow);
  const int ns = pr.src_len ? min(pr.src_len[srow], pr.src_pitch) : pr.src_pitch;
  const int nt = pr.tgt_len ? min(pr.tgt_len[trow], pr.tgt_pitch) : pr.tgt_pitch;
  const int n = min(ns, nt);
  double* pose = a.out.pose_total + p * 6;
  if (n <= 0) {
    if (lane == 0) { pose[0] = 1; pose[1] = 0; pose[2] = 0; pose[3] = 1; pose[4] = 0; pose[5] = 0; }
    return;
  }
  // each cloud relative to its own first point: the single-pass sums then cancel only as much as
  // the spread of the cloud, however far apart the two clouds are
  const double2 oa = load_point(pr.src_points, pr.dtype, srow * pr.src_pitch);
  const double2 o = load_point(pr.tgt_points, pr.dtype, trow * pr.tgt_pitch);
  double r[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int i = lane; i < n; i += 32) {
    const double2 s = load_point(pr.src_points, pr.dtype, srow * pr.src_pitch + i);
    const double2 b = load_point(pr.tgt_points, pr.dtype, trow * pr.tgt_pitch + i);
    const double ax = s.x - oa.x, ay = s.y - oa.y, qx = b.x - o.x, qy = b.y - o.y;
    r[0] += ax; r[1] += ay; r[2] += qx; r[3] += qy;
    r[4] = fma(ax, qx, r[4]); r[5] = fma(ax, qy, r[5]);
    r[6] = fma(ay, qx, r[6]); r[7] = fma(ay, qy, r[7]);
  }
#pragma unroll
  for (int q = 0; q < 8; ++q) {
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) r[q] += __shfl_xor_sync(kFull, r[q], s);
  }
  if (lane == 0) {
    const double inv = 1.0 / (double)n;
    const double max_ = r[0] * inv, may_ = r[1] * inv, mbx = r[2] * inv, mby = r[3] * inv;
    const double h00 = fma(-r[0], mbx, r[4]), h01 = fma(-r[0], mby, r[5]);
    const double h10 = fma(-r[1], mbx, r[6]), h11 = fma(-r[1], mby, r[7]);
    const double num = h01 - h10, den = h00 + h11;
    const double h2 = fma(num, num, den * den);
    double cs = 1.0, sn = 0.0;
    if (h2 > 0.0) { const double rh = rsqrt(h2); cs = den * rh; sn = num * rh; }
    const double cax = oa.x + max_, cay = oa.y + may_;
    pose[0] = cs; pose[1] = -sn; pose[2] = sn; pose[3] = cs;
    pose[4] = (o.x + mbx) - (cs * cax - sn * cay);          // icp.py:25
    pose[5] = (o.y + mby) - (sn * cax + cs * cay);
  }
}

// ------------------------------------------------------------------------------------
// kernel: scan preparation (process.py:38-52), one CTA per scan, order-preserving
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) polar_to_cartesian_kernel(
    const double* __restrict__ raw, const int32_t* __restrict__ raw_len, int raw_pitch,
    const b200icp_polar_filter f, double* __restrict__ xy_out, int32_t* __restrict__ len_out, int out_pitch) {
  __shared__ int warp_counts[8];
  __shared__ int base_shared;
  const int scan = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nwarps = blockDim.x >> 5;
  const int rows = min(raw_len ? raw_len[scan] : raw_pitch, raw_pitch);
  const double* src = raw + (int64_t)scan * raw_pitch * 3;
  double2* dst = reinterpret_cast<double2*>(xy_out) + (int64_t)scan * out_pitch;
  if (tid == 0) base_shared = 0;
  __syncthreads();
  for (int r0 = 0; r0 < rows; r0 += blockDim.x) {
    const int r = r0 + tid;
    bool keep = false;
    double x = 0.0, y = 0.0;
    if (r < rows) {
      const double quality = src[r * 3 + 0], angle = src[r * 3 + 1], dist = src[r * 3 + 2];
      const bool front = !f.use_arc || (angle <= f.arc_lo) || (angle >= f.arc_hi);   // process.py:45
      keep = dist > f.min_dist && dist < f.max_dist && quality > f.min_quality && front;   // process.py:46
      if (keep) {
        const double rad = angle * (3.14159265358979323846 / 180.0);       // math.radians
        double sn, cs;
        sincos(rad, &sn, &cs);
        x = dist * cs;                                                      // process.py:48
        y = f.y_sign < 0 ? -dist * sn : dist * sn;                          // process.py:49 (realtime_1.py:167: +)
      }
    }
    const unsigned ballot = __ballot_sync(kFull, keep);
    if (lane == 0) warp_counts[warp] = __popc(ballot);
    __syncthreads();
    int offset = base_shared;
    for (int w = 0; w < warp; ++w) offset += warp_counts[w];
    offset += __popc(ballot & ((1u << lane) - 1u));
    if (keep && offset < out_pitch) dst[offset] = make_double2(x, y);
    __syncthreads();
    if (tid == 0) {
      int total = 0;
      for (int w = 0; w < nwarps; ++w) total += warp_counts[w];
      base_shared += total;
    }
    __syncthreads();
  }
  if (tid == 0) len_out[scan] = min(base_shared, out_pitch);
  const int kept = min(base_shared, out_pitch);
  for (int i = kept + tid; i < out_pitch; i += blockDim.x) dst[i] = make_double2(0.0, 0.0);
}

// ------------------------------------------------------------------------------------
// kernels: order-preserving point selection (the steps either side of registration in the
// SLAM loop: local-map radius crop, duc/ICP_LIDAR/mainn.py:300-303; dynamic-point removal by
// NN distance, duc/ICP_LIDAR/process.py:75-84).  count -> exclusive scan -> scatter.
// ------------------------------------------------------------------------------------
constexpr int kSelBlock = 1024;      // points per CTA (256 threads x 4)

__device__ __forceinline__ bool select_keep(const void* points, int dtype, int64_t i, int mode,
                                            const double* key, double cx, double cy, double thr) {
  if (mode == 0) return key[i] < thr;
  // mainn.py:302  distances_sq < R^2, rounded as NumPy rounds it (a contracted FMA decides points
  // within an ulp of the circle differently)
  return dist2_f64(cx, cy, load_point(points, dtype, i)) < thr;
}

__global__ void __launch_bounds__(256) select_count_kernel(const void* points, int dtype, int64_t n,
                                                           int mode, const double* key, double cx,
                                                           double cy, double thr, int64_t* block_counts) {
  __shared__ int wc[8];
  const int64_t base = (int64_t)blockIdx.x * kSelBlock;
  int c = 0;
  for (int k = 0; k < 4; ++k) {
    const int64_t i = base + k * 256 + threadIdx.x;
    if (i < n && select_keep(points, dtype, i, mode, key, cx, cy, thr)) ++c;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(kFull, c, o);
  if ((threadIdx.x & 31) == 0) wc[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int w = 0; w < 8; ++w) t += wc[w];
    block_counts[blockIdx.x] = t;
  }
}

// exclusive scan of the per-block counts in place (one CTA: every thread owns a contiguous
// segment, warp-shuffle scan of the segment sums); total -> counts[n_blocks] and *count_out
__global__ void __launch_bounds__(1024) select_scan_kernel(int64_t* counts, int64_t n_blocks, int64_t* count_out) {
  __shared__ long long wsum[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t per = (n_blocks + 1023) / 1024;
  const int64_t b = min(n_blocks, tid * per), e = min(n_blocks, b + per);
  long long s = 0;
  for (int64_t k = b; k < e; ++k) s += counts[k];
  long long inc = s;                                   // inclusive scan inside the warp
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long v = __shfl_up_sync(kFull, inc, o);
    if (lane >= o) inc += v;
  }
  if (lane == 31) wsum[warp] = inc;
  __syncthreads();
  if (warp == 0) {                                     // exclusive scan of the 32 warp totals
    const long long w = wsum[lane];
    long long winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const long long v = __shfl_up_sync(kFull, winc, o);
      if (lane >= o) winc += v;
    }
    wsum[lane] = winc - w;
  }
  __syncthreads();
  long long run = wsum[warp] + inc - s;
  for (int64_t k = b; k < e; ++k) { const long long c = counts[k]; counts[k] = run; run += c; }
  if (tid == 1023) { counts[n_blocks] = run; *count_out = run; }
}

__global__ void __launch_bounds__(256) select_scatter_kernel(const void* points, int dtype, int64_t n,
                                                             int mode, const double* key, double cx,
                                                             double cy, double thr,
                                                             const int64_t* block_offsets, void* out) {
  __shared__ int wc[4][8];
  const int64_t base = (int64_t)blockIdx.x * kSelBlock;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  bool keep[4];
  unsigned ballots[4];
  for (int k = 0; k < 4; ++k) {                         // point order: k-major, then thread
    const int64_t i = base + k * 256 + threadIdx.x;
    keep[k] = i < n && select_keep(points, dtype, i, mode, key, cx, cy, thr);
    ballots[k] = __ballot_sync(kFull, keep[k]);
    if (lane == 0) wc[k][warp] = __popc(ballots[k]);
  }
  __syncthreads();
  int64_t off = block_offsets[blockIdx.x];
  for (int k = 0; k < 4; ++k) {
    int before = 0;
    for (int w = 0; w < warp; ++w) before += wc[k][w];
    if (keep[k]) {
      const int64_t dst = off + before + __popc(ballots[k] & ((1u << lane) - 1u));
      const int64_t i = base + k * 256 + threadIdx.x;
      if (dtype == B200ICP_F64) reinterpret_cast<double2*>(out)[dst] = reinterpret_cast<const double2*>(points)[i];
      else reinterpret_cast<float2*>(out)[dst] = reinterpret_cast<const float2*>(points)[i];
    }
    int row = 0;
    for (int w = 0; w < 8; ++w) row += wc[k][w];
    off += row;
  }
}

// ------------------------------------------------------------------------------------
// kernel: prefix composition of pairwise poses into global poses (sequence odometry:
// T_{0,k+1} = T_{0,k} o T_k; the reference's SLAM loops carry the pose frame to frame,
// duc/ICP_LIDAR/slam_offline.py:382-392).  One CTA, three phases: every thread composes a
// contiguous segment, thread 0 scans the 1,024 segment totals, every thread rewrites its
// segment with its prefix.  out[0] = identity, out[k+1] = out[k] o pose[k].
// ------------------------------------------------------------------------------------
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

__global__ void __launch_bounds__(1024) chain_poses_kernel(const double* __restrict__ poses, int64_t n,
                                                           double* __restrict__ out) {
  __shared__ double seg[1024][6];
  const int tid = threadIdx.x;
  const int64_t per = (n + 1023) / 1024;
  const int64_t b = min(n, tid * per), e = min(n, b + per);
  Se2 acc = se2_identity();
  for (int64_t k = b; k < e; ++k) acc = se2_mul(acc, se2_load(poses + 6 * k));
  // exclusive scan of the 1,024 segment totals: composition is associative, so a shuffle scan
  // inside every warp and one over the 32 warp totals replace the serial loop (order of the
  // factors preserved: earlier segments on the left)
  const int lane = tid & 31, warp = tid >> 5;
  Se2 inc = acc;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    Se2 v;
    v.r00 = __shfl_up_sync(kFull, inc.r00, o); v.r01 = __shfl_up_sync(kFull, inc.r01, o);
    v.r10 = __shfl_up_sync(kFull, inc.r10, o); v.r11 = __shfl_up_sync(kFull, inc.r11, o);
    v.tx = __shfl_up_sync(kFull, inc.tx, o); v.ty = __shfl_up_sync(kFull, inc.ty, o);
    if (lane >= o) inc = se2_mul(v, inc);
  }
  Se2 excl = inc;                        // exclusive within the warp: the neighbour's inclusive value
  excl.r00 = __shfl_up_sync(kFull, inc.r00, 1); excl.r01 = __shfl_up_sync(kFull, inc.r01, 1);
  excl.r10 = __shfl_up_sync(kFull, inc.r10, 1); excl.r11 = __shfl_up_sync(kFull, inc.r11, 1);
  excl.tx = __shfl_up_sync(kFull, inc.tx, 1); excl.ty = __shfl_up_sync(kFull, inc.ty, 1);
  if (lane == 0) excl = se2_identity();
  if (lane == 31) se2_store(seg[warp], inc);           // warp totals in seg[0..31]
  __syncthreads();
  if (warp == 0) {
    const Se2 w = se2_load(seg[lane]);
    Se2 winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      Se2 v;
      v.r00 = __shfl_up_sync(kFull, winc.r00, o); v.r01 = __shfl_up_sync(kFull, winc.r01, o);
      v.r10 = __shfl_up_sync(kFull, winc.r10, o); v.r11 = __shfl_up_sync(kFull, winc.r11, o);
      v.tx = __shfl_up_sync(kFull, winc.tx, o); v.ty = __shfl_up_sync(kFull, winc.ty, o);
      if (lane >= o) winc = se2_mul(v, winc);
    }
    Se2 wex;
    wex.r00 = __shfl_up_sync(kFull, winc.r00, 1); wex.r01 = __shfl_up_sync(kFull, winc.r01, 1);
    wex.r10 = __shfl_up_sync(kFull, winc.r10, 1); wex.r11 = __shfl_up_sync(kFull, winc.r11, 1);
    wex.tx = __shfl_up_sync(kFull, winc.tx, 1); wex.ty = __shfl_up_sync(kFull, winc.ty, 1);
    if (lane == 0) wex = se2_identity();
    se2_store(seg[32 + lane], wex);                    // exclusive warp prefixes in seg[32..63]
  }
  if (tid == 0) se2_store(out, se2_identity());
  __syncthreads();
  acc = se2_mul(se2_load(seg[32 + warp]), excl);
  for (int64_t k = b; k < e; ++k) {
    acc = se2_mul(acc, se2_load(poses + 6 * k));
    se2_store(out + 6 * (k + 1), acc);
  }
}

// ------------------------------------------------------------------------------------
// kernel: FP32 FFMA throughput probe (roofline denominator of the NN phase)
// ------------------------------------------------------------------------------------
constexpr int kProbeChains = 16;
__global__ void __launch_bounds__(256) ffma_probe_kernel(float* sink, int inner_iters) {
  float acc[kProbeChains];
  const float a = 1.0f + 1e-7f * (float)threadIdx.x, b = 1e-9f * (float)(blockIdx.x + 1);
#pragma unroll
  for (int i = 0; i < kProbeChains; ++i) acc[i] = (float)i;
  for (int it = 0; it < inner_iters; ++it) {
#pragma unroll
    for (int i = 0; i < kProbeChains; ++i) acc[i] = fmaf(acc[i], a, b);
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < kProbeChains; ++i) s += acc[i];
  if (s == 123.456f) sink[0] = s;     // never true in practice; keeps the chain live
}

// ------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------
struct LaunchShape {
  int S;           // CTA-per-pair kernels: source points per lane
  int warps;
  size_t smem;
  int mcap;
};

bool pick_shape(const b200icp_problem* pr, LaunchShape& ls) {
  const int pitch = pr->src_pitch;
  int S = (pitch + 127) / 128;               // aim at <= 4 warps until S saturates
  if (S < 1) S = 1;
  if (S > kMaxS) S = kMaxS;
  int warps = (pitch + 32 * S - 1) / (32 * S);
  if (warps < 1) warps = 1;
  if (warps > kMaxWarps) return false;
  ls.S = S;
  ls.warps = warps;
  ls.mcap = (pr->tgt_pitch + kGroup - 1) / kGroup * kGroup;
  ls.smem = tile_bytes(ls.mcap);
  return true;
}

int check_problem(const b200icp_problem* pr, int64_t n_pairs) {
  if (!pr) { set_error("problem is NULL"); return B200ICP_ERR_INVALID_ARGUMENT; }
  if (n_pairs < 0) { set_error("n_pairs < 0"); return B200ICP_ERR_INVALID_ARGUMENT; }
  if (!pr->src_points || !pr->tgt_points) {
    set_error("src_points / tgt_points is NULL");
    return B200ICP_ERR_INVALID_ARGUMENT;
  }
  if (pr->src_pitch < 1 || pr->tgt_pitch < 1) {
    set_error("pitch must be >= 1");
    return B200ICP_ERR_INVALID_ARGUMENT;
  }
  if (pr->dtype != B200ICP_F32 && pr->dtype != B200ICP_F64) {
    set_error("dtype must be B200ICP_F32 or B200ICP_F64");
    return B200ICP_ERR_INVALID_ARGUMENT;
  }
  if (pr->pairing < B200ICP_PAIR_ROWWISE || pr->pairing > B200ICP_PAIR_TRIANGLE) {
    set_error("unknown pairing");
    return B200ICP_ERR_INVALID_ARGUMENT;
  }
  if (pr->pairing == B200ICP_PAIR_EXPLICIT && (!pr->src_row || !pr->tgt_row)) {
    set_error("EXPLICIT pairing needs src_row and tgt_row");
    return B200ICP_ERR_INVALID_ARGUMENT;
  }
  if (pr->pairing == B200ICP_PAIR_TRIANGLE) {
    const int64_t rows = pr->n_rows;
    if (rows < 2 || pr->first_pair < 0 || pr->first_pair + n_pairs > rows * (rows - 1) / 2) {
      set_error("TRIANGLE pairing: pair range outside n_rows*(n_rows-1)/2");
      return B200ICP_ERR_INVALID_ARGUMENT;
    }
  }
  if (pr->src_pitch > kMaxSrcPitch || pr->tgt_pitch > kMaxTgtPitch) {
    set_error("pitch beyond the fused per-pair kernel (src <= 1024, tgt <= 4096)");
    return B200ICP_ERR_UNSUPPORTED_SHAPE;
  }
  if (n_pairs > 0x7fffffffLL) { set_error("n_pairs > 2^31-1 per call"); return B200ICP_ERR_INVALID_ARGUMENT; }
  return B200ICP_OK;
}

int cuda_fail(cudaError_t e, const char* what) {
  set_error("%s: %s", what, cudaGetErrorString(e));
  return B200ICP_ERR_CUDA;
}

// One launch per call.  The opt-in to more than 48 KB of dynamic shared memory is made once per
// kernel and device (the largest size the device allows), not on every launch.
template <typename Kern>
int launch_pairs(Kern kern, const LaunchShape& ls, const KernelArgs& args, cudaStream_t st) {
  if (ls.smem > 48 * 1024) {
    // (all kernels share the function-pointer type, so the memo is keyed by pointer and device)
    static std::mutex mu;
    static std::set<std::pair<const void*, int>> opted_in;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lock(mu);
    const std::pair<const void*, int> key(reinterpret_cast<const void*>(kern), dev);
    if (!opted_in.count(key)) {
      int max_optin = 0;
      cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin);
      if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(max dynamic smem)");
      opted_in.insert(key);
    }
  }
  kern<<<(unsigned)args.n_pairs, ls.warps * 32, ls.smem, st>>>(args);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "kernel launch");
  return B200ICP_OK;
}

// W-warps-per-pair fused kernel: passes of 64 sources (pruned sweep) or 192 sources (dense sweep),
// dealt round-robin to W <= 4 warps.  W = the warp count in 2..4 that leaves the fewest idle
// warp-rounds, the smallest on ties: measured on B200 (profiles/r2_kernel_tuning.md) two warps beat
// one (shared tile: 24 instead of 18 resident warps per SM) and three or four (the redundant pose
// solve and the wait at the cross-warp sum grow with W): 360 points = 6 blocks of 64 on 2 warps.
constexpr int kPairS = 2, kPairDenseS = 6, kPairMaxWarps = 4;

int pair_warps_for(int passes, int forced) {
  if (passes < 1) passes = 1;
  if (forced >= 1 && forced <= kPairMaxWarps) return forced < passes ? forced : passes;
  if (passes == 1) return 1;
  int best = 2, best_idle = 1 << 30;
  for (int w = 2; w <= kPairMaxWarps && w <= passes; ++w) {
    const int idle = (passes + w - 1) / w * w - passes;
    if (idle < best_idle) { best = w; best_idle = idle; }
  }
  return best;
}

int launch_pair_kernel(const b200icp_problem* prob, const LaunchShape& ls, KernelArgs& args, bool dense,
                       int forced_warps, cudaStream_t st) {
  const int S = dense ? kPairDenseS : kPairS;
  args.ncap = (prob->src_pitch + 32 * S - 1) / (32 * S) * (32 * S);
  args.passes = args.ncap / (32 * S);
  if (args.passes > kPairMaxPasses) {
    set_error("source pitch exceeds the pair kernel's pass table");
    return B200ICP_ERR_UNSUPPORTED_SHAPE;
  }
  LaunchShape ps = ls;
  // W follows the 64-source blocks of the float64 phase, not the pass width of the search, so that
  // the dense and the pruned kernel add the sums in the same order (bit-identical results)
  ps.warps = pair_warps_for((prob->src_pitch + 63) / 64, forced_warps);
  ps.smem = pair_tile_bytes(ls.mcap, args.ncap, args.passes, ps.warps);
  // LEAN: the throughput configuration (float32 tables, no gate, no per-point index outputs)
  const bool lean = prob->dtype == B200ICP_F32 && !args.use_gate && !args.out.indices && !args.out.index_history;
#define B200ICP_PAIR_CASE(W)                                                                            \
  case W:                                                                                               \
    if (lean)                                                                                           \
      return dense ? launch_pairs(icp_align_pair_kernel<kPairDenseS, false, W, true>, ps, args, st)     \
                   : launch_pairs(icp_align_pair_kernel<kPairS, true, W, true>, ps, args, st);          \
    return dense ? launch_pairs(icp_align_pair_kernel<kPairDenseS, false, W, false>, ps, args, st)      \
                 : launch_pairs(icp_align_pair_kernel<kPairS, true, W, false>, ps, args, st);
  switch (ps.warps) {
    B200ICP_PAIR_CASE(1)
    B200ICP_PAIR_CASE(2)
    B200ICP_PAIR_CASE(3)
    default:
    B200ICP_PAIR_CASE(4)
  }
#undef B200ICP_PAIR_CASE
}

int launch_nn_warp_kernel(const b200icp_problem* prob, const LaunchShape& ls, KernelArgs& args, bool dense,
                          cudaStream_t st) {
  const int S = dense ? kPairDenseS : kPairS;
  args.ncap = (prob->src_pitch + 32 * S - 1) / (32 * S) * (32 * S);
  args.passes = args.ncap / (32 * S);
  if (args.passes > kPairMaxPasses) {
    set_error("source pitch exceeds the pair kernel's pass table");
    return B200ICP_ERR_UNSUPPORTED_SHAPE;
  }
  LaunchShape ps = ls;
  ps.warps = 1;
  ps.smem = pair_tile_bytes(ls.mcap, args.ncap, args.passes, 1);
  return dense ? launch_pairs(nn_warp_kernel<kPairDenseS, false>, ps, args, st)
               : launch_pairs(nn_warp_kernel<kPairS, true>, ps, args, st);
}

// Which kernel family for a batch?  b200icp.h: B200ICP_FLAG_WARP_KERNEL / _CTA_KERNEL, else by size.
bool use_cta_kernel(int64_t n_pairs, int flags, bool wants_stats) {
  if (flags & B200ICP_FLAG_WARP_KERNEL) return false;
  if (flags & B200ICP_FLAG_CTA_KERNEL) return true;
  return n_pairs <= kAutoCtaPairs && !(flags & B200ICP_FLAG_DENSE_SWEEP) && !wants_stats;
}

#define B200ICP_DISPATCH_CTA(KERNEL)                                         \
  switch (ls.S) {                                                            \
    case 1: return launch_pairs(KERNEL<1>, ls, args, st);                    \
    case 2: return launch_pairs(KERNEL<2>, ls, args, st);                    \
    case 3: return launch_pairs(KERNEL<3>, ls, args, st);                    \
    default: return launch_pairs(KERNEL<4>, ls, args, st);                   \
  }

}  // namespace

// shared with scan2map.cu (C++ linkage: not part of the C ABI)
void b200icp_set_error_str(const char* msg) { set_error("%s", msg); }

extern "C" {

int b200icp_version(void) { return B200ICP_VERSION_MAJOR * 1000 + B200ICP_VERSION_MINOR; }

const char* b200icp_last_error(void) { return g_last_error; }

int b200icp_max_src_pitch(void) { return kMaxSrcPitch; }
int b200icp_max_tgt_pitch(void) { return kMaxTgtPitch; }

int b200icp_nn_batch(const b200icp_problem* prob, int64_t n_pairs, int32_t* idx_out,
                     double* dist2_out, int32_t flags, void* stream) {
  int rc = check_problem(prob, n_pairs);
  if (rc != B200ICP_OK) return rc;
  if (!idx_out) { set_error("idx_out is NULL"); return B200ICP_ERR_INVALID_ARGUMENT; }
  if (n_pairs == 0) return B200ICP_OK;
  LaunchShape ls;
  if (!pick_shape(prob, ls)) { set_error("unsupported src_pitch"); return B200ICP_ERR_UNSUPPORTED_SHAPE; }
  KernelArgs args;
  memset(&args, 0, sizeof(args));
  args.prob = *prob;
  args.nn_idx = idx_out;
  args.nn_dist2 = dist2_out;
  args.n_pairs = n_pairs;
  args.mcap = ls.mcap;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // same rule as the fused loop: CTA per pair below the batch size that fills the GPU with one-warp CTAs
  if (!use_cta_kernel(n_pairs, flags, false))
    return launch_nn_warp_kernel(prob, ls, args, (flags & B200ICP_FLAG_DENSE_SWEEP) != 0, st);
  B200ICP_DISPATCH_CTA(nn_pair_kernel)
}

int b200icp_align_batch(const b200icp_problem* prob, int64_t n_pairs, const b200icp_options* opt,
                        const b200icp_outputs* out, void* stream) {
  int rc = check_problem(prob, n_pairs);
  if (rc != B200ICP_OK) return rc;
  if (!opt || !out) { set_error("options / outputs is NULL"); return B200ICP_ERR_INVALID_ARGUMENT; }
  if (!out->pose_total || !out->error || !out->iterations) {
    set_error("outputs.pose_total, .error and .iterations are required");
    return B200ICP_ERR_INVALID_ARGUMENT;
  }
  if (opt->max_iterations < 0) { set_error("max_iterations < 0"); return B200ICP_ERR_INVALID_ARGUMENT; }
  if (n_pairs == 0) return B200ICP_OK;
  LaunchShape ls;
  if (!pick_shape(prob, ls)) { set_error("unsupported src_pitch"); return B200ICP_ERR_UNSUPPORTED_SHAPE; }
  KernelArgs args;
  memset(&args, 0, sizeof(args));
  args.prob = *prob;
  args.opt = *opt;
  args.out = *out;
  args.n_pairs = n_pairs;
  args.mcap = ls.mcap;
  args.use_gate = (opt->max_corr_dist > 0.0 && std::isfinite(opt->max_corr_dist)) ? 1 : 0;
  args.reuse = (opt->flags & B200ICP_FLAG_NO_SWEEP_REUSE) ? 0 : 1;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // Which fused kernel?  W warps per pair sharing one tile has the best throughput once the pairs
  // fill the GPU (148 SMs x 12 CTAs); below that a pair's latency is what counts and the CTA-per-pair
  // kernel (up to 8 warps on one pair) is ~2x faster: 0.14 vs 0.23 ms for one 160 x 1,000
  // scan-to-local-map registration, crossover near 500 pairs of 360 x 360 (tools/latency_single.py).
  if (!use_cta_kernel(n_pairs, opt->flags, out->evaluated_pairs != nullptr))
    return launch_pair_kernel(prob, ls, args, (opt->flags & B200ICP_FLAG_DENSE_SWEEP) != 0,
                              (opt->flags >> B200ICP_FLAG_PAIR_WARPS_SHIFT) & 7, st);
  B200ICP_DISPATCH_CTA(icp_align_kernel)
}

int b200icp_best_fit_batch(const b200icp_problem* prob, int64_t n_pairs, double* pose_out, void* stream) {
  int rc = check_problem(prob, n_pairs);
  if (rc == B200ICP_ERR_UNSUPPORTED_SHAPE) rc = B200ICP_OK;      // no shared-memory tile: any pitch
  if (rc != B200ICP_OK) return rc;
  if (!pose_out) { set_error("pose_out is NULL"); return B200ICP_ERR_INVALID_ARGUMENT; }
  if (n_pairs == 0) return B200ICP_OK;
  KernelArgs args;
  memset(&args, 0, sizeof(args));
  args.prob = *prob;
  args.out.pose_total = pose_out;
  args.n_pairs = n_pairs;
  best_fit_warp_kernel<<<(unsigned)n_pairs, 32, 0, reinterpret_cast<cudaStream_t>(stream)>>>(args);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "best_fit_warp_kernel");
  return B200ICP_OK;
}

int b200icp_polar_to_cartesian(const double* raw, const int32_t* raw_len, int32_t n_scans,
                               int32_t raw_pitch, const b200icp_polar_filter* filter, double* xy_out,
                               int32_t* len_out, int32_t out_pitch, void* stream) {
  if (!raw || !xy_out || !len_out) { set_error("NULL pointer"); return B200ICP_ERR_INVALID_ARGUMENT; }
  if (n_scans < 0 || raw_pitch < 1 || out_pitch < 1) { set_error("bad size"); return B200ICP_ERR_INVALID_ARGUMENT; }
  if (n_scans == 0) return B200ICP_OK;
  b200icp_polar_filter f;                        // process.py:45-46,49 (canonical)
  f.min_dist = 1000.0; f.max_dist = 9000.0; f.min_quality = 10.0; f.arc_lo = 135.0; f.arc_hi = 225.0;
  f.use_arc = 1; f.y_sign = -1;
  if (filter) f = *filter;
  if (f.y_sign != 1 && f.y_sign != -1) { set_error("polar filter: y_sign must be +1 or -1"); return B200ICP_ERR_INVALID_ARGUMENT; }
  polar_to_cartesian_kernel<<<n_scans, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      raw, raw_len, raw_pitch, f, xy_out, len_out, out_pitch);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "polar_to_cartesian launch");
  return B200ICP_OK;
}

int b200icp_select_points(const void* points, int32_t dtype, int64_t n, int32_t mode, const double* key,
                          double cx, double cy, double threshold, void* out_points,
                          int64_t* count_out, int64_t* scratch, void* stream) {
  // an empty set may come with NULL points / out_points / key (an empty tensor has no storage)
  if ((n > 0 && (!points || !out_points)) || !count_out || !scratch || n < 0) { set_error("select_points: bad arguments"); return B200ICP_ERR_INVALID_ARGUMENT; }
  if (dtype != B200ICP_F32 && dtype != B200ICP_F64) { set_error("select_points: bad dtype"); return B200ICP_ERR_INVALID_ARGUMENT; }
  if (mode != 0 && mode != 1) { set_error("select_points: mode must be 0 (key) or 1 (radius)"); return B200ICP_ERR_INVALID_ARGUMENT; }
  if (mode == 0 && !key && n > 0) { set_error("select_points: mode 0 needs key"); return B200ICP_ERR_INVALID_ARGUMENT; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int64_t blocks = (n + kSelBlock - 1) / kSelBlock;
  if (blocks > 0) {
    select_count_kernel<<<(unsigned)blocks, 256, 0, st>>>(points, dtype, n, mode, key, cx, cy, threshold, scratch);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "select_count_kernel");
  }
  select_scan_kernel<<<1, 1024, 0, st>>>(scratch, blocks, count_out);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "select_scan_kernel");
  if (blocks > 0) {
    select_scatter_kernel<<<(unsigned)blocks, 256, 0, st>>>(points, dtype, n, mode, key, cx, cy, threshold, scratch, out_points);
    e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "select_scatter_kernel");
  }
  return B200ICP_OK;
}

int b200icp_chain_poses(const double* poses, int64_t n, double* out, void* stream) {
  if ((n > 0 && !poses) || !out || n < 0) { set_error("chain_poses: bad arguments"); return B200ICP_ERR_INVALID_ARGUMENT; }
  chain_poses_kernel<<<1, 1024, 0, reinterpret_cast<cudaStream_t>(stream)>>>(poses, n, out);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "chain_poses_kernel");
  return B200ICP_OK;
}

int b200icp_ffma_probe(float* sink, int32_t inner_iters, int64_t* flop_out, void* stream) {
  if (!sink || inner_iters < 1) { set_error("bad probe arguments"); return B200ICP_ERR_INVALID_ARGUMENT; }
  int dev = 0, sms = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return cuda_fail(e, "cudaGetDevice");
  e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (e != cudaSuccess) return cuda_fail(e, "cudaDeviceGetAttribute");
  const int blocks = sms * 8, threads = 256;
  ffma_probe_kernel<<<blocks, threads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(sink, inner_iters);
  e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "ffma probe launch");
  if (flop_out) *flop_out = (int64_t)blocks * threads * (int64_t)inner_iters * kProbeChains * 2;
  return B200ICP_OK;
}

}  // extern "C"
