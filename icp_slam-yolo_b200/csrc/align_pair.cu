// align_pair.cu -- the throughput kernels: the fused ICP loop with W warps per pair sharing one
// target tile (icp_align_pair_kernel), and the one-warp-per-pair nearest-neighbour search
// (nn_warp_kernel) built from its search phase.  DESIGN.md has the measurements.
#include <cuda_runtime.h>
#include <math_constants.h>

#include <cstdint>

#include "launch.cuh"

namespace {

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

// ------------------------------------------------------------------------------------
// Shared-memory state of one pair.  The candidate sweep reads the centred float32 targets from
// shared memory; the float64 targets stay in global memory (L1/L2) and are touched once per
// source per iteration (the matched point), because the in-group decision is made in FP32
// direct-difference form first (error ~1e-3 mm) and only near-ties fall back to the
// warp-cooperative float64 scan.
// ------------------------------------------------------------------------------------
struct PairTile {
  const void* tgt;      // global target table
  int64_t row_off;      // first point of this pair's target row
  int dtype;
  float* tile;          // [mcap/8][24]: per group of 8 targets x[8], y[8], |t|^2[8] (centred float32),
                        // 96 contiguous bytes = six LDS.128 off one address
  double2* src;         // [ncap] float64 source state
  float* gcx;           // [mcap/8] bounding circle of each group of 8 targets (pruned sweep)
  float* gcy;
  float* grad;
  double ox, oy;
  float tmax;
  int m, mcap, ngroups;
  unsigned short* nnidx;    // [ncap] nearest target of every source at its last search
  unsigned short* grp2;     // [ncap] the OTHER group of the source's candidate pair (= its own group if alone)
  unsigned keep;            // mantissa bits a packed sweep key keeps: ~((1 << log2ceil(groups)) - 1)
  float* tgrp;              // [passes] cum_move up to which the sources of a pass keep their GROUP
  float* tnn;               // [passes] ... keep their nearest neighbour
  double* red;              // [2][W][kPairRedStride]
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
__device__ __forceinline__ void warp_candidates(const PairTile& t, const float (&sx)[S],
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

__device__ __forceinline__ GroupRegs load_group(const PairTile& t, int g) {
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
__device__ __forceinline__ void eval_mask(const PairTile& t, unsigned mask, int base_g,
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
__device__ __forceinline__ int warp_candidates_pruned(const PairTile& t, const float (&sx)[S],
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
// W warps of a pair share ONE target tile, and the kernel is compiled for 24 resident warps per SM
// (<= 80 registers).  One warp per pair with a tile of its own is latency-bound at 16 resident warps
// per SM (122 registers, 11.5 KB of shared memory per warp), with ~60 % of its instructions outside
// the candidate sweep; sharing the tile cuts shared memory per warp by ~W/2.  Two phases per
// iteration, so that search and float64 state do not overlap in the register file:
//   phase 1 (search): per pass of 32*SC sources -> nearest target index, stored as uint16 in
//            shared memory; FP32 only (plus the rare float64 rescans);
//   phase 2 (update): every source: gather of its matched target, exact float64 distance,
//            the 11 centred sums; then warp shuffle + one shared-memory hop across the W warps,
//            closed-form pose, apply.
// The sweep reuse bounds the movement not only to "the group of 8 that holds the nearest neighbour"
// but to the nearest neighbour itself: a pass whose sources have all moved less than half the gap
// between their nearest and their second-nearest target (lower bound of the in-group runner-up and
// of everything outside the group) skips phase 1 ENTIRELY -- no set-up, no culling, no in-group
// argmin -- and the iteration is gather + distance + sums only.
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
__host__ __device__ inline size_t pair_tile_bytes(int mcap, int ncap, int warps) {
  size_t b = kCtxBytes + (size_t)2 * warps * kPairRedStride * sizeof(double) +
             (size_t)2 * kPairMaxPasses * sizeof(float) + (size_t)ncap * sizeof(double2) +
             (size_t)mcap * 3 * sizeof(float) + (size_t)(mcap / kGroup) * 3 * sizeof(float) +
             (size_t)ncap * 2 * sizeof(unsigned short);
  return (b + 15) & ~(size_t)15;
}

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
}

// Stage the target tile, all warps of the CTA together: the target centroid (the origin), per group
// of 8 the centred float32 x, y and |t|^2, and the bounding circle of every group.
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
    // sentinels: |t|^2 = +inf makes the expanded form +inf (no inf - inf: the coordinates stay
    // finite), and 1e18 makes the direct-difference form ~2e36, finite and never the minimum
    float cx = 1e18f, cy = 1e18f, tt = CUDART_INF_F;
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

__device__ __forceinline__ int in_group_decide(const PairTile& t, int ga, int gb, bool two, float fx, float fy,
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

}  // namespace

int launch_pair_kernel(const b200icp_problem* prob, const LaunchShape& ls, KernelArgs& args, bool dense,
                       int forced_warps, cudaStream_t st) {
  const int S = dense ? kPairDenseS : kPairS;
  args.ncap = (prob->src_pitch + 32 * S - 1) / (32 * S) * (32 * S);
  args.passes = args.ncap / (32 * S);
  if (args.passes > kPairMaxPasses)
    return set_error(B200ICP_ERR_UNSUPPORTED_SHAPE, "source pitch exceeds the pair kernel's pass table");
  LaunchShape ps = ls;
  // W follows the 64-source blocks of the float64 phase, not the pass width of the search, so that
  // the dense and the pruned kernel add the sums in the same order (bit-identical results)
  ps.warps = pair_warps_for((prob->src_pitch + 63) / 64, forced_warps);
  ps.smem = pair_tile_bytes(ls.mcap, args.ncap, ps.warps);
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
  if (args.passes > kPairMaxPasses)
    return set_error(B200ICP_ERR_UNSUPPORTED_SHAPE, "source pitch exceeds the pair kernel's pass table");
  LaunchShape ps = ls;
  ps.warps = 1;
  ps.smem = pair_tile_bytes(ls.mcap, args.ncap, 1);
  return dense ? launch_pairs(nn_warp_kernel<kPairDenseS, false>, ps, args, st)
               : launch_pairs(nn_warp_kernel<kPairS, true>, ps, args, st);
}
