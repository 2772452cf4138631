// align_cta.cu -- the CTA-per-pair kernels: nearest-neighbour search and the fused ICP loop, one
// CTA per scan pair (the latency configuration of b200icp_nn_batch / b200icp_align_batch).
//
// Reference behaviour being replaced (paths relative to the reference repo):
//   labels_segmentation/icp.py:28-53  icp()                 -> icp_align_kernel
//   labels_segmentation/icp.py:37-38  KDTree(B).query(src)   -> nn_candidates + nn_resolve
//   labels_segmentation/icp.py:5-26   best_fit_transform()   -> kabsch_increment (icp_step.cuh) in icp_align_kernel
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
//     Kabsch problem in closed form redundantly (no broadcast step); the update step itself
//     (sums, Kabsch, apply, compose, outputs) is icp_step.cuh's.
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
  int n, m;
  row_lengths(pr, srow, trow, n, m);
  int32_t* idx_out = a.nn_idx + p * pr.src_pitch;
  double* d2_out = a.nn_dist2 ? a.nn_dist2 + p * pr.src_pitch : nullptr;

  if (n <= 0 || m <= 0) {
    nn_fill_none(idx_out, d2_out, tid, pr.src_pitch, nthreads);
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
  int n, m;
  row_lengths(pr, srow, trow, n, m);

  // cumulative pose (src = Rt * A + tt) starts at the initial pose (gicp_lidar.py:32 shape)
  Se2 pose = load_init_pose(op.init_pose, p);
  Increment last{1.0, 0.0, 0.0, 0.0};
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
        double2 q = load_point(pr.src_points, pr.dtype, srow * pr.src_pitch + i);   // icp.py:32  src = copy(A)
        if (op.init_pose) q = apply(pose, q);
        sx[k] = q.x; sy[k] = q.y;
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
            add_match(r, sx[k] - t.ox, sy[k] - t.oy, b.x - t.ox, b.y - t.oy);
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
      const double mean_error = r[8] * inv;                     // icp.py:48
      const Increment d = kabsch_increment(r, inv, t.ox, t.oy, t.ox, t.oy);
      // ---- apply (icp.py:45) and compose the cumulative pose
#pragma unroll
      for (int k = 0; k < S; ++k) {
        if (valid[k]) {
          const double2 v = apply(d, make_double2(sx[k], sy[k]));
          sx[k] = v.x; sy[k] = v.y;
        }
      }
      pose = compose(d, pose);
      last = d;
      err = mean_error; mean_d2 = r[9] * inv; inl = (int)(cnt + 0.5);
      iters = it + 1;
      // ---- convergence (icp.py:49-51); identical in every thread
      if (fabs(prev_error - mean_error) < op.tolerance) break;
      prev_error = mean_error;
    }
  }

  if (tid == 0) write_pair_result(out, p, pose, last, err, mean_d2, inl, iters);
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
              v = apply(pose, load_point(pr.src_points, pr.dtype, srow * pr.src_pitch + i));
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
