// prep.cu -- the support kernels around registration: scan preparation (polar -> Cartesian),
// order-preserving point selection, best_fit_transform for matched rows, prefix composition of
// poses, and the FP32 FFMA throughput probe.
//
// Reference behaviour being replaced (paths relative to the reference repo):
//   labels_segmentation/icp.py:5-26   best_fit_transform()   -> best_fit_warp_kernel
//   duc/ICP_LIDAR/process.py:38-52    polar_to_cartesian_3d  -> polar_to_cartesian_kernel
#include <cuda_runtime.h>

#include <cstdint>
#include <cstring>

#include "common.cuh"
#include "compact.cuh"

namespace {

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
struct SelectKeep {
  const void* points;
  int dtype, mode;
  const double* key;
  double cx, cy, thr;
  __device__ __forceinline__ bool operator()(int64_t i) const {
    if (mode == 0) return key[i] < thr;
    // mainn.py:302  distances_sq < R^2, rounded as NumPy rounds it (a contracted FMA decides points
    // within an ulp of the circle differently)
    return dist2_f64(cx, cy, load_point(points, dtype, i)) < thr;
  }
};

struct CopyPoint {
  const void* points;
  int dtype;
  void* out;
  __device__ __forceinline__ void operator()(int64_t dst, int64_t i) const {
    if (dtype == B200ICP_F64) reinterpret_cast<double2*>(out)[dst] = reinterpret_cast<const double2*>(points)[i];
    else reinterpret_cast<float2*>(out)[dst] = reinterpret_cast<const float2*>(points)[i];
  }
};

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

}  // namespace

extern "C" {

int b200icp_best_fit_batch(const b200icp_problem* prob, int64_t n_pairs, double* pose_out, void* stream) {
  int rc = check_problem(prob, n_pairs);
  if (rc == B200ICP_ERR_UNSUPPORTED_SHAPE) rc = B200ICP_OK;      // no shared-memory tile: any pitch
  if (rc != B200ICP_OK) return rc;
  if (!pose_out) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "pose_out is NULL");
  if (n_pairs == 0) return B200ICP_OK;
  KernelArgs args;
  memset(&args, 0, sizeof(args));
  args.prob = *prob;
  args.out.pose_total = pose_out;
  args.n_pairs = n_pairs;
  best_fit_warp_kernel<<<(unsigned)n_pairs, 32, 0, reinterpret_cast<cudaStream_t>(stream)>>>(args);
  return check_launch("best_fit_warp_kernel");
}

int b200icp_polar_to_cartesian(const double* raw, const int32_t* raw_len, int32_t n_scans,
                               int32_t raw_pitch, const b200icp_polar_filter* filter, double* xy_out,
                               int32_t* len_out, int32_t out_pitch, void* stream) {
  if (!raw || !xy_out || !len_out) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "NULL pointer");
  if (n_scans < 0 || raw_pitch < 1 || out_pitch < 1) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "bad size");
  if (n_scans == 0) return B200ICP_OK;
  b200icp_polar_filter f;                        // process.py:45-46,49 (canonical)
  f.min_dist = 1000.0; f.max_dist = 9000.0; f.min_quality = 10.0; f.arc_lo = 135.0; f.arc_hi = 225.0;
  f.use_arc = 1; f.y_sign = -1;
  if (filter) f = *filter;
  if (f.y_sign != 1 && f.y_sign != -1) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "polar filter: y_sign must be +1 or -1");
  polar_to_cartesian_kernel<<<n_scans, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      raw, raw_len, raw_pitch, f, xy_out, len_out, out_pitch);
  return check_launch("polar_to_cartesian launch");
}

int b200icp_select_points(const void* points, int32_t dtype, int64_t n, int32_t mode, const double* key,
                          double cx, double cy, double threshold, void* out_points,
                          int64_t* count_out, int64_t* scratch, void* stream) {
  // an empty set may come with NULL points / out_points / key (an empty tensor has no storage)
  if ((n > 0 && (!points || !out_points)) || !count_out || !scratch || n < 0) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "select_points: bad arguments");
  if (dtype != B200ICP_F32 && dtype != B200ICP_F64) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "select_points: bad dtype");
  if (mode != 0 && mode != 1) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "select_points: mode must be 0 (key) or 1 (radius)");
  if (mode == 0 && !key && n > 0) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "select_points: mode 0 needs key");
  return compact(SelectKeep{points, dtype, mode, key, cx, cy, threshold}, CopyPoint{points, dtype, out_points}, n,
                 scratch, count_out, reinterpret_cast<cudaStream_t>(stream), "select");
}

int b200icp_chain_poses(const double* poses, int64_t n, double* out, void* stream) {
  if ((n > 0 && !poses) || !out || n < 0) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "chain_poses: bad arguments");
  chain_poses_kernel<<<1, 1024, 0, reinterpret_cast<cudaStream_t>(stream)>>>(poses, n, out);
  return check_launch("chain_poses_kernel");
}

int b200icp_ffma_probe(float* sink, int32_t inner_iters, int64_t* flop_out, void* stream) {
  if (!sink || inner_iters < 1) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "bad probe arguments");
  int dev = 0, sms = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return set_error(B200ICP_ERR_CUDA, "cudaGetDevice: %s", cudaGetErrorString(e));
  e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (e != cudaSuccess) return set_error(B200ICP_ERR_CUDA, "cudaDeviceGetAttribute: %s", cudaGetErrorString(e));
  const int blocks = sms * 8, threads = 256;
  ffma_probe_kernel<<<blocks, threads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(sink, inner_iters);
  if (const int rc = check_launch("ffma probe launch")) return rc;
  if (flop_out) *flop_out = (int64_t)blocks * threads * (int64_t)inner_iters * kProbeChains * 2;
  return B200ICP_OK;
}

}  // extern "C"
