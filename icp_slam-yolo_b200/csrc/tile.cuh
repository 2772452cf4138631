// tile.cuh -- the shared-memory target tile and the exact nearest-neighbour search of the
// CTA-per-pair kernels (align_cta.cu) and of GICP (gicp.cu).
#pragma once

#include <math_constants.h>

#include "common.cuh"

constexpr int kRedStride = 8;      // doubles per warp slot in the staging reductions
constexpr int kRedStride2 = 12;    // doubles per warp slot in the per-iteration reduction

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

__device__ __forceinline__ bool is_ambiguous(float best, float second, float scx, float scy, float tmax) {
  const float cs = fmaxf(fabsf(scx), fabsf(scy));
  return (second - best) <= expanded_margin(cs, tmax);   // near-equal floats subtract exactly
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
