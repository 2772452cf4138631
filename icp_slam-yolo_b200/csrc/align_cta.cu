// align_cta.cu -- the CTA-per-pair kernels: nearest-neighbour search and the fused ICP loop, one
// CTA per scan pair (the latency configuration of b200icp_nn_batch / b200icp_align_batch).
//
// Reference behaviour being replaced (paths relative to the reference repo):
//   labels_segmentation/icp.py:28-53  icp()                 -> icp_align_kernel
//   labels_segmentation/icp.py:37-38  KDTree(B).query(src)   -> nn_candidates + nn_resolve
//   labels_segmentation/icp.py:5-26   best_fit_transform()   -> pose solve inside icp_align_kernel
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

#include <cstdint>

#include "launch.cuh"
#include "tile.cuh"

// CTAs of kMaxWarps warps that must fit one SM: caps registers per thread
// (65536 / (256 * kMinBlocks)); typical CTAs have 4 warps, so twice as many are resident.
#ifndef B200ICP_MIN_BLOCKS
#define B200ICP_MIN_BLOCKS 2
#endif

namespace {

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

}  // namespace

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

int launch_nn_cta_kernel(const LaunchShape& ls, const KernelArgs& args, cudaStream_t st) {
  B200ICP_DISPATCH_CTA(nn_pair_kernel)
}

int launch_align_cta_kernel(const LaunchShape& ls, const KernelArgs& args, cudaStream_t st) {
  B200ICP_DISPATCH_CTA(icp_align_kernel)
}
