// b200icp.cu -- the C ABI of the 2D ICP scan-matching path: version, error state, pitch limits,
// argument checks, and the choice between the two kernel families of b200icp_nn_batch /
// b200icp_align_batch (one CTA per pair: align_cta.cu; W warps per pair: align_pair.cu).
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <set>
#include <utility>

#include "launch.cuh"

namespace {

constexpr int64_t kAutoCtaPairs = 512;    // at or below: CTA-per-pair fused kernel (latency), above: W warps per pair (throughput)

thread_local char g_last_error[512] = "";

// Which kernel family for a batch?  b200icp.h: B200ICP_FLAG_WARP_KERNEL / _CTA_KERNEL, else by size.
bool use_cta_kernel(int64_t n_pairs, int flags, bool wants_stats) {
  if (flags & B200ICP_FLAG_WARP_KERNEL) return false;
  if (flags & B200ICP_FLAG_CTA_KERNEL) return true;
  return n_pairs <= kAutoCtaPairs && !(flags & B200ICP_FLAG_DENSE_SWEEP) && !wants_stats;
}

}  // namespace

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_last_error, sizeof(g_last_error), fmt, ap);
  va_end(ap);
  return code;
}

int check_launch(const char* what, ...) {
  const cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) return B200ICP_OK;
  char buf[256];
  va_list ap;
  va_start(ap, what);
  vsnprintf(buf, sizeof(buf), what, ap);
  va_end(ap);
  return set_error(B200ICP_ERR_CUDA, "%s: %s", buf, cudaGetErrorString(e));
}

int opt_in_dynamic_smem(const void* kern, int bytes) {
  static std::mutex mu;
  static std::set<std::pair<const void*, int>> opted_in;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return set_error(B200ICP_ERR_CUDA, "cudaGetDevice: %s", cudaGetErrorString(e));
  std::lock_guard<std::mutex> lock(mu);
  const std::pair<const void*, int> key(kern, dev);
  if (opted_in.count(key)) return B200ICP_OK;
  if (bytes < 0) cudaDeviceGetAttribute(&bytes, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess)
    return set_error(B200ICP_ERR_CUDA, "cudaFuncSetAttribute(%d bytes of dynamic smem): %s", bytes, cudaGetErrorString(e));
  opted_in.insert(key);
  return B200ICP_OK;
}

int check_problem(const b200icp_problem* pr, int64_t n_pairs, bool pitch_limit) {
  if (!pr) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "problem is NULL");
  if (n_pairs < 0) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "n_pairs < 0");
  if (!pr->src_points || !pr->tgt_points)
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "src_points / tgt_points is NULL");
  if (pr->src_pitch < 1 || pr->tgt_pitch < 1)
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "pitch must be >= 1");
  if (pr->dtype != B200ICP_F32 && pr->dtype != B200ICP_F64)
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "dtype must be B200ICP_F32 or B200ICP_F64");
  if (pr->pairing < B200ICP_PAIR_ROWWISE || pr->pairing > B200ICP_PAIR_TRIANGLE)
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "unknown pairing");
  if (pr->pairing == B200ICP_PAIR_EXPLICIT && (!pr->src_row || !pr->tgt_row))
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "EXPLICIT pairing needs src_row and tgt_row");
  if (pr->pairing == B200ICP_PAIR_TRIANGLE) {
    const int64_t rows = pr->n_rows;
    if (rows < 2 || pr->first_pair < 0 || pr->first_pair + n_pairs > rows * (rows - 1) / 2)
      return set_error(B200ICP_ERR_INVALID_ARGUMENT, "TRIANGLE pairing: pair range outside n_rows*(n_rows-1)/2");
  }
  if (pitch_limit && (pr->src_pitch > kMaxSrcPitch || pr->tgt_pitch > kMaxTgtPitch))
    return set_error(B200ICP_ERR_UNSUPPORTED_SHAPE, "pitch beyond the fused per-pair kernel (src <= 1024, tgt <= 4096)");
  if (n_pairs > 0x7fffffffLL) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "n_pairs > 2^31-1 per call");
  return B200ICP_OK;
}

extern "C" {

int b200icp_version(void) { return B200ICP_VERSION_MAJOR * 1000 + B200ICP_VERSION_MINOR; }

const char* b200icp_last_error(void) { return g_last_error; }

int b200icp_max_src_pitch(void) { return kMaxSrcPitch; }
int b200icp_max_tgt_pitch(void) { return kMaxTgtPitch; }

int b200icp_nn_batch(const b200icp_problem* prob, int64_t n_pairs, int32_t* idx_out,
                     double* dist2_out, int32_t flags, void* stream) {
  int rc = check_problem(prob, n_pairs);
  if (rc != B200ICP_OK) return rc;
  if (!idx_out) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "idx_out is NULL");
  if (n_pairs == 0) return B200ICP_OK;
  LaunchShape ls;
  if (!pick_shape(prob, ls)) return set_error(B200ICP_ERR_UNSUPPORTED_SHAPE, "unsupported src_pitch");
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
  return launch_nn_cta_kernel(ls, args, st);
}

int b200icp_align_batch(const b200icp_problem* prob, int64_t n_pairs, const b200icp_options* opt,
                        const b200icp_outputs* out, void* stream) {
  int rc = check_problem(prob, n_pairs);
  if (rc != B200ICP_OK) return rc;
  if (!opt || !out) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "options / outputs is NULL");
  if (!out->pose_total || !out->error || !out->iterations)
    return set_error(B200ICP_ERR_INVALID_ARGUMENT, "outputs.pose_total, .error and .iterations are required");
  if (opt->max_iterations < 0) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "max_iterations < 0");
  if (n_pairs == 0) return B200ICP_OK;
  LaunchShape ls;
  if (!pick_shape(prob, ls)) return set_error(B200ICP_ERR_UNSUPPORTED_SHAPE, "unsupported src_pitch");
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
  return launch_align_cta_kernel(ls, args, st);
}

}  // extern "C"
