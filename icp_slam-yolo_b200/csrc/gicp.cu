// gicp.cu -- 2D Generalized ICP: per-point regularised covariances and the fused GICP loop, one CTA
// per pair, built on the target tile and exact search of the CTA-per-pair kernels (tile.cuh).
//
// Reference behaviour being replaced (paths relative to the reference repo):
//   duc/ICP_LIDAR/gicp_lidar.py:12-36 gicp() (Open3D GICP)    -> covariance_kernel + gicp_align_kernel (2D)
#include <cuda_runtime.h>
#include <math_constants.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>

#include "launch.cuh"
#include "tile.cuh"

namespace {

// ------------------------------------------------------------------------------------
// 2D Generalized ICP (line-to-line; DESIGN.md §4.8): the registration objective of the reference's
// gicp() (duc/ICP_LIDAR/gicp_lidar.py:12-36), one CTA per pair.  Targets beyond one shared-memory
// tile are searched tile by tile (kGicpTile points each, ascending); every tile search is the exact
// one of nn_search and the per-tile winners merge by strict < on the absolute float64 d^2, so the
// result is the global float64 argmin with the lowest index on ties.
// ------------------------------------------------------------------------------------
constexpr int kGicpTile = kMaxTgtPitch;          // targets per shared-memory tile
constexpr int kGicpMaxTgtPitch = 65536;          // = 16 tiles
constexpr int kGicpMaxK = 32;                    // covariance neighbours: one per lane

struct GicpArgs {
  b200icp_problem prob;
  b200icp_gicp_options opt;
  b200icp_outputs out;
  const double* src_cov;    // [src rows][src_pitch][3]
  const double* tgt_cov;    // [tgt rows][tgt_pitch][3]
  int64_t n_pairs;
  int32_t mcap;             // tile capacity: min(tgt_pitch rounded up to kGroup, kGicpTile)
  int32_t use_gate;
};

// R p + t, rounded as the oracle rounds it (no contraction), so that the pivot and a source point at
// the centroid stay bit-identical.
__device__ __forceinline__ double2 apply_pose(const Se2& a, double x, double y) {
  return make_double2(__dadd_rn(__dadd_rn(__dmul_rn(a.r00, x), __dmul_rn(a.r01, y)), a.tx),
                      __dadd_rn(__dadd_rn(__dmul_rn(a.r10, x), __dmul_rn(a.r11, y)), a.ty));
}

template <int S>
// one CTA per SM at map sizes (a 4,096-point tile is 116 KB), so the register cap is that of one CTA
__global__ void __launch_bounds__(kMaxWarps * 32, 1) gicp_align_kernel(const GicpArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  TargetTile t;
  carve_tile(smem_raw, a.mcap, t);
  double* red = t.red;

  const int tid = threadIdx.x, nthreads = blockDim.x;
  const int warp = tid >> 5, lane = tid & 31, nwarps = nthreads >> 5;
  const int64_t p = blockIdx.x;
  const b200icp_problem& pr = a.prob;
  const b200icp_gicp_options& op = a.opt;
  const b200icp_outputs& out = a.out;

  int64_t srow, trow;
  resolve_rows(pr, p, srow, trow);
  int n, m;
  row_lengths(pr, srow, trow, n, m);
  const int64_t soff = srow * pr.src_pitch, toff = trow * pr.tgt_pitch;

  Se2 P = load_init_pose(op.init_pose, p);
  Increment last{1.0, 0.0, 0.0, 0.0};
  double err = CUDART_INF, mean_d2 = CUDART_INF;
  int iters = 0, inl = 0;

  double sx[S], sy[S], ca[S][3];
  bool valid[S];
  int idx[S];
#pragma unroll
  for (int k = 0; k < S; ++k) {
    const int i = tid + k * nthreads;
    valid[k] = i < n;
    sx[k] = 0.0; sy[k] = 0.0; idx[k] = -1;
    ca[k][0] = 1.0; ca[k][1] = 0.0; ca[k][2] = 1.0;
    if (valid[k]) {
      const double2 q = load_point(pr.src_points, pr.dtype, soff + i);
      sx[k] = q.x; sy[k] = q.y;
      const double* c = a.src_cov + (soff + i) * 3;
      ca[k][0] = c[0]; ca[k][1] = c[1]; ca[k][2] = c[2];
    }
  }

  if (n > 0 && m > 0) {
    const bool tiled = m > kGicpTile;
    if (!tiled) stage_targets(pr.tgt_points, pr.dtype, toff, m, t, tid, nthreads, warp, lane, nwarps);
    // pivot: the centroid of the original source (red[1]: stage_targets used red[0])
    double cen[2] = {0.0, 0.0};
#pragma unroll
    for (int k = 0; k < S; ++k) { cen[0] += sx[k]; cen[1] += sy[k]; }
    block_sum<2>(cen, red + kMaxWarps * kRedStride2, warp, lane, nwarps);
    const double cax = cen[0] / (double)n, cay = cen[1] / (double)n;
#pragma unroll
    for (int k = 0; k < S; ++k) {
      if (valid[k]) {
        const double2 v = apply_pose(P, sx[k], sy[k]);
        sx[k] = v.x; sy[k] = v.y;
      }
    }
    const double gate = op.max_corr_dist;
    const bool use_gate = a.use_gate != 0;
    const double inv_n = 1.0 / (double)n;
    double fit_prev = 0.0, rmse_prev = 0.0;
    int rb = 0;                                              // reduction buffer of the next block_sum
    for (int e = 0;; ++e) {
      // ---- evaluation: exact NN over all tiles
      double bd[S];
#pragma unroll
      for (int k = 0; k < S; ++k) { bd[k] = CUDART_INF; idx[k] = 0; }
      for (int base = 0; base < m; base += kGicpTile) {
        if (tiled) {
          __syncthreads();                                   // the previous tile and reductions are read
          stage_targets(pr.tgt_points, pr.dtype, toff + base, min(kGicpTile, m - base), t, tid, nthreads,
                        warp, lane, nwarps);
        }
        int li[S];
        double ld[S];
        nn_search<S>(t, sx, sy, valid, lane, li, ld);
#pragma unroll
        for (int k = 0; k < S; ++k) {
          if (ld[k] < bd[k]) { bd[k] = ld[k]; idx[k] = base + li[k]; }
        }
      }
      // ---- gate, evaluation sums and the Gauss-Newton system at this pose, one reduction:
      // r[0..5] = H (00 01 02 11 12 22), r[6..8] = g, r[9] = inliers, r[10] = sum d^2, r[11] = sum d
      const double2 c = apply_pose(P, cax, cay);
      double r[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
      for (int k = 0; k < S; ++k) {
        if (valid[k]) {
          const double dist = sqrt(bd[k]);
          if (!use_gate || dist < gate) {
            const int64_t j = toff + idx[k];
            const double2 b = load_point(pr.tgt_points, pr.dtype, j);
            const double* cb = a.tgt_cov + j * 3;
            // S = C_B + R C_A R^T, M = S^-1 (closed form)
            const double u00 = P.r00 * ca[k][0] + P.r01 * ca[k][1], u01 = P.r00 * ca[k][1] + P.r01 * ca[k][2];
            const double u10 = P.r10 * ca[k][0] + P.r11 * ca[k][1], u11 = P.r10 * ca[k][1] + P.r11 * ca[k][2];
            const double sa = __ldg(cb) + (u00 * P.r00 + u01 * P.r01);
            const double sb = __ldg(cb + 1) + (u00 * P.r10 + u01 * P.r11);
            const double sd = __ldg(cb + 2) + (u10 * P.r10 + u11 * P.r11);
            const double inv = 1.0 / (sa * sd - sb * sb);
            const double m00 = sd * inv, m01 = -sb * inv, m11 = sa * inv;
            const double rx = sx[k] - c.x, ry = sy[k] - c.y;
            const double e0 = b.x - sx[k], e1 = b.y - sy[k];
            const double w0 = m01 * rx - m00 * ry, w1 = m11 * rx - m01 * ry;
            const double v0 = m00 * e0 + m01 * e1, v1 = m01 * e0 + m11 * e1;
            r[0] += rx * w1 - ry * w0; r[1] += w0; r[2] += w1;
            r[3] += m00; r[4] += m01; r[5] += m11;
            r[6] += rx * v1 - ry * v0; r[7] += v0; r[8] += v1;
            r[9] += 1.0; r[10] += bd[k]; r[11] += dist;
          }
        }
      }
      block_sum<12>(r, red + rb * kMaxWarps * kRedStride2, warp, lane, nwarps);
      rb ^= 1;
      const double cnt = r[9];
      if (cnt < 0.5) {                                       // nothing inside the gate: stop
        err = CUDART_INF; mean_d2 = CUDART_INF; inl = 0;
        break;
      }
      mean_d2 = r[10] / cnt;
      const double fit = cnt * inv_n, rm = sqrt(mean_d2);
      err = r[11] / cnt; inl = (int)(cnt + 0.5);
      if (e > 0 && fabs(fit - fit_prev) < op.relative_fitness && fabs(rm - rmse_prev) < op.relative_rmse) break;
      if (iters >= op.max_iterations) break;
      fit_prev = fit; rmse_prev = rm;
      // ---- 3x3 Cholesky solve of H x = g (identical in every thread)
      const double H00 = r[0], H01 = r[1], H02 = r[2], H11 = r[3], H12 = r[4], H22 = r[5];
      if (!(H00 > 0.0) || !isfinite(H00)) break;
      const double L00 = sqrt(H00);
      const double L10 = H01 / L00, L20 = H02 / L00;
      const double p1 = H11 - L10 * L10;
      if (!(p1 > 0.0) || !isfinite(p1)) break;
      const double L11 = sqrt(p1);
      const double L21 = (H12 - L20 * L10) / L11;
      const double p2 = H22 - L20 * L20 - L21 * L21;
      if (!(p2 > 0.0) || !isfinite(p2)) break;
      const double L22 = sqrt(p2);
      const double y0 = r[6] / L00;
      const double y1 = (r[7] - L10 * y0) / L11;
      const double y2 = (r[8] - L20 * y0 - L21 * y1) / L22;
      const double dy = y2 / L22;
      const double dx = (y1 - L21 * dy) / L11;
      const double dth = (y0 - L10 * dx - L20 * dy) / L00;
      if (out.index_history) {
        int32_t* h = out.index_history + (p * op.max_iterations + iters) * (int64_t)pr.src_pitch;
#pragma unroll
        for (int k = 0; k < S; ++k) {
          const int i = tid + k * nthreads;
          if (i < pr.src_pitch) h[i] = valid[k] ? idx[k] : -1;
        }
      }
      // ---- apply s <- R(dth)(s - c) + c + d and compose T <- dT o T, each as an increment
      // s + ((R(dth) - I)(s - c) + d) with cos(dth) - 1 = -2 sin^2(dth / 2): a zero step leaves points
      // and pose bit for bit as they were, and a small one is not rounded through (s - c) + c
      double sh, ch;
      sincos(0.5 * dth, &sh, &ch);
      const double sn = __dmul_rn(__dmul_rn(2.0, sh), ch), cm1 = __dmul_rn(__dmul_rn(-2.0, sh), sh);
#pragma unroll
      for (int k = 0; k < S; ++k) {
        if (valid[k]) {
          const double ex = __dsub_rn(sx[k], c.x), ey = __dsub_rn(sy[k], c.y);
          sx[k] = __dadd_rn(sx[k], __dadd_rn(__dsub_rn(__dmul_rn(cm1, ex), __dmul_rn(sn, ey)), dx));
          sy[k] = __dadd_rn(sy[k], __dadd_rn(__dadd_rn(__dmul_rn(sn, ex), __dmul_rn(cm1, ey)), dy));
        }
      }
      {
        const double tx = P.tx - c.x, ty = P.ty - c.y;
        P = Se2{P.r00 + (cm1 * P.r00 - sn * P.r10), P.r01 + (cm1 * P.r01 - sn * P.r11),
                P.r10 + (sn * P.r00 + cm1 * P.r10), P.r11 + (sn * P.r01 + cm1 * P.r11),
                P.tx + ((cm1 * tx - sn * ty) + dx), P.ty + ((sn * tx + cm1 * ty) + dy)};
      }
      last = Increment{1.0 + cm1, sn, dx - (cm1 * c.x - sn * c.y), dy - (sn * c.x + cm1 * c.y)};
      ++iters;
    }
  }

  if (tid == 0) write_pair_result(out, p, P, last, err, mean_d2, inl, iters);
  if (out.indices || out.src_final) {
    const bool ran = n > 0 && m > 0;
#pragma unroll
    for (int k = 0; k < S; ++k) {
      const int i = tid + k * nthreads;
      if (i < pr.src_pitch) {
        if (out.indices) out.indices[p * pr.src_pitch + i] = (valid[k] && ran) ? idx[k] : -1;
        if (out.src_final) {
          double2 v = make_double2(0.0, 0.0);
          if (valid[k]) v = ran ? make_double2(sx[k], sy[k]) : apply_pose(P, sx[k], sy[k]);
          reinterpret_cast<double2*>(out.src_final)[p * pr.src_pitch + i] = v;
        }
      }
    }
  }
}

// Per-point regularised covariance (b200icp_estimate_covariances), one warp per point: an exact
// float64 k-NN over the point's row kept as a warp-distributed sorted list (lane l holds the l-th
// best (d^2, index)), then the mean and covariance summed sequentially in that order without
// contraction, so the sums equal the oracle's bit for bit.
__global__ void __launch_bounds__(256) covariance_kernel(const void* __restrict__ pts, const int32_t* __restrict__ len,
                                                         int32_t rows, int32_t pitch, int32_t dtype, int32_t k,
                                                         double eps, double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t total = (int64_t)rows * pitch;
  const int64_t wstride = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t q = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); q < total; q += wstride) {
    const int64_t r = q / pitch;
    const int i = (int)(q - r * pitch);
    const int n = len ? min(max(len[r], 0), pitch) : pitch;
    double* o = out + q * 3;
    if (i >= n) {
      if (lane < 3) o[lane] = 0.0;
      continue;
    }
    const int64_t off = r * pitch;
    const double2 qp = load_point(pts, dtype, off + i);
    const int kk = min(k, n);
    double kd = CUDART_INF;
    int ki = -1;
    for (int base = 0; base < n; base += 32) {
      const int j = base + lane;
      double d = CUDART_INF;
      if (j < n) d = dist2_f64(qp.x, qp.y, load_point(pts, dtype, off + j));
      unsigned cand = __ballot_sync(kFull, d < __shfl_sync(kFull, kd, kk - 1));
      while (cand) {                                 // ascending index: equal d^2 ranks after the list
        const int src = __ffs(cand) - 1;
        cand &= cand - 1;
        const double cd = __shfl_sync(kFull, d, src);
        if (!(cd < __shfl_sync(kFull, kd, kk - 1))) continue;
        const int pos = __popc(__ballot_sync(kFull, lane < kk && kd <= cd));
        const double ud = __shfl_up_sync(kFull, kd, 1);
        const int ui = __shfl_up_sync(kFull, ki, 1);
        if (lane < kk) {
          if (lane > pos) { kd = ud; ki = ui; }
          else if (lane == pos) { kd = cd; ki = base + src; }
        }
      }
    }
    const double2 nb = lane < kk ? load_point(pts, dtype, off + ki) : make_double2(0.0, 0.0);
    double mx = 0.0, my = 0.0;
    for (int l = 0; l < kk; ++l) {
      mx = __dadd_rn(mx, __shfl_sync(kFull, nb.x, l));
      my = __dadd_rn(my, __shfl_sync(kFull, nb.y, l));
    }
    mx = __ddiv_rn(mx, (double)kk);
    my = __ddiv_rn(my, (double)kk);
    double cxx = 0.0, cxy = 0.0, cyy = 0.0;
    for (int l = 0; l < kk; ++l) {
      const double dx = __dsub_rn(__shfl_sync(kFull, nb.x, l), mx);
      const double dy = __dsub_rn(__shfl_sync(kFull, nb.y, l), my);
      cxx = __dadd_rn(cxx, __dmul_rn(dx, dx));
      cxy = __dadd_rn(cxy, __dmul_rn(dx, dy));
      cyy = __dadd_rn(cyy, __dmul_rn(dy, dy));
    }
    cxx = __ddiv_rn(cxx, (double)kk);
    cxy = __ddiv_rn(cxy, (double)kk);
    cyy = __ddiv_rn(cyy, (double)kk);
    double rxx = 1.0, rxy = 0.0, ryy = 1.0;
    if (kk >= 3 && __dadd_rn(cxx, cyy) != 0.0) {
      const double phi = 0.5 * atan2(__dmul_rn(2.0, cxy), __dsub_rn(cxx, cyy));
      double s, c;
      sincos(phi, &s, &c);
      rxx = __dadd_rn(__dmul_rn(c, c), __dmul_rn(eps, __dmul_rn(s, s)));
      rxy = __dmul_rn(__dsub_rn(1.0, eps), __dmul_rn(c, s));
      ryy = __dadd_rn(__dmul_rn(s, s), __dmul_rn(eps, __dmul_rn(c, c)));
    }
    if (lane == 0) { o[0] = rxx; o[1] = rxy; o[2] = ryy; }
  }
}

}  // namespace

extern "C" {

int b200icp_estimate_covariances(const void* points, const int32_t* len, int32_t rows, int32_t pitch,
                                 int32_t dtype, int32_t k, double epsilon, double* cov_out, void* stream) {
  if (!points || !cov_out) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "estimate_covariances: points / cov_out is NULL");
  if (rows < 0 || pitch < 1) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "estimate_covariances: rows < 0 or pitch < 1");
  if (dtype != B200ICP_F32 && dtype != B200ICP_F64) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "estimate_covariances: bad dtype");
  if (k < 3 || k > kGicpMaxK) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "estimate_covariances: k must be in 3..32");
  if (!(epsilon > 0.0) || !std::isfinite(epsilon)) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "estimate_covariances: epsilon must be finite and > 0");
  if (pitch > kGicpMaxTgtPitch) return set_error(B200ICP_ERR_UNSUPPORTED_SHAPE, "estimate_covariances: pitch > 65536");
  if (rows == 0) return B200ICP_OK;
  const int64_t warps = (int64_t)rows * pitch;
  const int64_t blocks = std::min<int64_t>((warps + 7) / 8, 148LL * 64);
  covariance_kernel<<<(unsigned)blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      points, len, rows, pitch, dtype, k, epsilon, cov_out);
  return check_launch("covariance_kernel");
}

int b200icp_gicp_batch(const b200icp_problem* prob, int64_t n_pairs, const b200icp_gicp_options* opt,
                       const double* src_cov, const double* tgt_cov, const b200icp_outputs* out, void* stream) {
  int rc = check_problem(prob, n_pairs);
  if (rc == B200ICP_ERR_UNSUPPORTED_SHAPE) {          // targets are tiled: tgt_pitch up to 65536
    if (prob->src_pitch > kMaxSrcPitch || prob->tgt_pitch > kGicpMaxTgtPitch)
      return set_error(B200ICP_ERR_UNSUPPORTED_SHAPE, "gicp_batch: pitch beyond the GICP kernel (src <= 1024, tgt <= 65536)");
    if (n_pairs > 0x7fffffffLL) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "n_pairs > 2^31-1 per call");
    rc = B200ICP_OK;
  }
  if (rc != B200ICP_OK) return rc;
  if (!opt || !out || !src_cov || !tgt_cov)
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "gicp_batch: options / outputs / src_cov / tgt_cov is NULL");
  if (!out->pose_total || !out->error || !out->iterations)
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "outputs.pose_total, .error and .iterations are required");
  if (opt->max_iterations < 0) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "max_iterations < 0");
  if (n_pairs == 0) return B200ICP_OK;
  LaunchShape ls;
  if (!pick_shape(prob, ls)) return set_error(B200ICP_ERR_UNSUPPORTED_SHAPE, "unsupported src_pitch");
  ls.mcap = std::min(ls.mcap, kGicpTile);
  ls.smem = tile_bytes(ls.mcap);
  GicpArgs args;
  memset(&args, 0, sizeof(args));
  args.prob = *prob;
  args.opt = *opt;
  args.out = *out;
  args.src_cov = src_cov;
  args.tgt_cov = tgt_cov;
  args.n_pairs = n_pairs;
  args.mcap = ls.mcap;
  args.use_gate = (opt->max_corr_dist > 0.0 && std::isfinite(opt->max_corr_dist)) ? 1 : 0;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  B200ICP_DISPATCH_CTA(gicp_align_kernel)
}

}  // extern "C"
