// compact.cuh -- order-preserving compaction (count -> exclusive scan -> scatter) of the points
// i < n that a predicate keeps, shared by b200icp_select_points and b200icp_occ_filter_points.
#pragma once

#include "common.cuh"

namespace {   // kernels: instantiated in every translation unit that compacts

constexpr int kCompactBlock = 1024;      // points per CTA (256 threads x 4)

template <typename Keep>
__global__ void __launch_bounds__(256) compact_count_kernel(const Keep keep, int64_t n, int64_t* block_counts) {
  __shared__ int wc[8];
  const int64_t base = (int64_t)blockIdx.x * kCompactBlock;
  int c = 0;
  for (int k = 0; k < 4; ++k) {
    const int64_t i = base + k * 256 + threadIdx.x;
    if (i < n && keep(i)) ++c;
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
__global__ void __launch_bounds__(1024) compact_scan_kernel(int64_t* counts, int64_t n_blocks, int64_t* count_out) {
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

template <typename Keep, typename Emit>
__global__ void __launch_bounds__(256) compact_scatter_kernel(const Keep keep, int64_t n,
                                                              const int64_t* block_offsets, const Emit emit) {
  __shared__ int wc[4][8];
  const int64_t base = (int64_t)blockIdx.x * kCompactBlock;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  bool kept[4];
  unsigned ballots[4];
  for (int k = 0; k < 4; ++k) {                         // point order: k-major, then thread
    const int64_t i = base + k * 256 + threadIdx.x;
    kept[k] = i < n && keep(i);
    ballots[k] = __ballot_sync(kFull, kept[k]);
    if (lane == 0) wc[k][warp] = __popc(ballots[k]);
  }
  __syncthreads();
  int64_t off = block_offsets[blockIdx.x];
  for (int k = 0; k < 4; ++k) {
    int before = 0;
    for (int w = 0; w < warp; ++w) before += wc[k][w];
    if (kept[k]) emit(off + before + __popc(ballots[k] & ((1u << lane) - 1u)), base + k * 256 + threadIdx.x);
    int row = 0;
    for (int w = 0; w < 8; ++w) row += wc[k][w];
    off += row;
  }
}

// emit(dst, i) for the dst-th of the points i < n with keep(i), in order; the count goes to
// *count_out.  scratch: int64[ceil(n / 1024) + 1].  Launch errors name the kernels "<name>_count_kernel",
// "<name>_scan_kernel" and "<name>_scatter_kernel".
template <typename Keep, typename Emit>
int compact(const Keep& keep, const Emit& emit, int64_t n, int64_t* scratch, int64_t* count_out,
            cudaStream_t st, const char* name) {
  const int64_t blocks = (n + kCompactBlock - 1) / kCompactBlock;
  if (blocks > 0) {
    compact_count_kernel<<<(unsigned)blocks, 256, 0, st>>>(keep, n, scratch);
    if (const int rc = check_launch("%s_count_kernel", name)) return rc;
  }
  compact_scan_kernel<<<1, 1024, 0, st>>>(scratch, blocks, count_out);
  if (const int rc = check_launch("%s_scan_kernel", name)) return rc;
  if (blocks > 0) {
    compact_scatter_kernel<<<(unsigned)blocks, 256, 0, st>>>(keep, n, scratch, emit);
    return check_launch("%s_scatter_kernel", name);
  }
  return B200ICP_OK;
}

}  // namespace
