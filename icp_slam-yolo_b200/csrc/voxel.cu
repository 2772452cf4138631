// voxel.cu -- 2D voxel-grid down-sampling on the device (sm_100a).
//
// The reference down-samples both clouds before every registration
// (duc/ICP_LIDAR/gicp_lidar.py:8-11,20-21: point_cloud.voxel_down_sample(voxel_size)) and removes
// duplicates the same way (duc/ICP_LIDAR/process.py:68-73); labels_segmentation/d.py:10-16 spells
// the 2D grid out: cell = floor(p / voxel_size).  Open3D keeps ONE point per occupied voxel, the
// mean of the points that fell into it.  Its output order is the iteration order of a hash map
// (unspecified); here the voxels come out sorted by (cell_y, cell_x), which is the order d.py
// builds with lexsort.  Parity-unpinned against Open3D (not vendored by the reference): the
// semantics are pinned by oracle.icp_oracle.voxel_down_sample_2d.
//
// cells (cell_y, cell_x), int64 per axis -> two stable cub radix sorts of (key, index): by cell_x,
// then by cell_y -> order (cell_y, cell_x, input order) -> one thread per point: segment heads
// average their run in the original point order (deterministic).  Points whose cell is not an
// int64 (non-finite coordinates, |p / voxel_size| >= 2^63) are skipped, as b200icp_occ_update
// skips non-finite points.
#include <cuda_runtime.h>

#include <cub/device/device_radix_sort.cuh>
#include <cstdint>
#include <cstdio>

#include "common.cuh"

namespace {

// sort key of a skipped point: above every biased int64 cell (the largest cell of a double below
// 2^63 is 2^63 - 1024), so skipped points sort last and never join a cell's run
constexpr uint64_t kSkipKey = ~0ull;

__device__ __forceinline__ double2 vx_load(const void* base, int dtype, int64_t i) {
  if (dtype == B200ICP_F64) return reinterpret_cast<const double2*>(base)[i];
  const float2 v = reinterpret_cast<const float2*>(base)[i];
  return make_double2((double)v.x, (double)v.y);
}

// cell = floor(p / voxel) (d.py:11-12), biased to unsigned so that the radix order is the signed
// order; kSkipKey for both axes unless both cells are int64
__device__ __forceinline__ void vx_cell(const void* points, int dtype, int64_t i, double inv_voxel,
                                        uint64_t& kx, uint64_t& ky) {
  const double2 q = vx_load(points, dtype, i);
  const double fx = floor(q.x * inv_voxel), fy = floor(q.y * inv_voxel);
  const double lim = 9223372036854775808.0;                 // 2^63
  if (!(fabs(fx) < lim && fabs(fy) < lim)) { kx = ky = kSkipKey; return; }
  kx = (uint64_t)(int64_t)fx ^ 0x8000000000000000ull;
  ky = (uint64_t)(int64_t)fy ^ 0x8000000000000000ull;
}

__global__ void voxel_key_x_kernel(const void* points, int dtype, int64_t n, double inv_voxel,
                                   uint64_t* keys, int32_t* idx) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t kx, ky;
  vx_cell(points, dtype, i, inv_voxel, kx, ky);
  keys[i] = kx;
  idx[i] = (int32_t)i;
}

// cell_y of the points in cell_x order, for the second (stable) pass
__global__ void voxel_key_y_kernel(const void* points, int dtype, int64_t n, double inv_voxel,
                                   const int32_t* idx, uint64_t* keys) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t kx, ky;
  vx_cell(points, dtype, idx[i], inv_voxel, kx, ky);
  keys[i] = ky;
}

// head of a run: a kept point whose cell differs from its predecessor's in sorted order
__global__ void voxel_head_kernel(const void* points, int dtype, int64_t n, double inv_voxel,
                                  const uint64_t* keys_y, const int32_t* idx, int32_t* head_flag) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (keys_y[i] == kSkipKey) { head_flag[i] = 0; return; }
  int flag = 1;
  if (i > 0) {
    uint64_t ax, ay, bx, by;
    vx_cell(points, dtype, idx[i], inv_voxel, ax, ay);
    vx_cell(points, dtype, idx[i - 1], inv_voxel, bx, by);
    flag = (ax != bx || ay != by) ? 1 : 0;
  }
  head_flag[i] = flag;
}

// one thread per sorted position; heads walk their run (both sorts are stable, so a run lists its
// points in the original order) and write the mean to the slot given by the scanned head count
__global__ void voxel_emit_kernel(const void* points, int dtype, int64_t n, const uint64_t* keys_y,
                                  const int32_t* idx, const int32_t* head_flag,
                                  const int32_t* head_rank, void* out, int64_t* count_out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (i == n - 1) *count_out = head_rank[i] + (int64_t)1;     // inclusive scan - 1 = slot
  if (!head_flag[i]) return;
  double sx = 0.0, sy = 0.0;
  int64_t k = i;
  do {
    const double2 q = vx_load(points, dtype, idx[k]);
    sx += q.x; sy += q.y;
    ++k;
  } while (k < n && !head_flag[k] && keys_y[k] != kSkipKey);
  const double inv = 1.0 / (double)(k - i);
  const int64_t slot = head_rank[i];
  if (dtype == B200ICP_F64) reinterpret_cast<double2*>(out)[slot] = make_double2(sx * inv, sy * inv);
  else reinterpret_cast<float2*>(out)[slot] = make_float2((float)(sx * inv), (float)(sy * inv));
}

// inclusive scan of head flags minus one (single CTA, a contiguous segment per thread)
__global__ void __launch_bounds__(1024) voxel_scan_kernel(const int32_t* flag, int64_t n, int32_t* rank) {
  __shared__ int32_t tot[1024];
  const int tid = threadIdx.x;
  const int64_t per = (n + 1023) / 1024, b = min(n, tid * per), e = min(n, b + per);
  int32_t s = 0;
  for (int64_t k = b; k < e; ++k) s += flag[k];
  const int lane = tid & 31, warp = tid >> 5;
  int32_t inc = s;                                      // warp-shuffle scan of the segment sums
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int32_t v = __shfl_up_sync(kFull, inc, o);
    if (lane >= o) inc += v;
  }
  if (lane == 31) tot[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const int32_t w = tot[lane];
    int32_t winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int32_t v = __shfl_up_sync(kFull, winc, o);
      if (lane >= o) winc += v;
    }
    tot[lane] = winc - w;
  }
  __syncthreads();
  int32_t run = tot[warp] + inc - s;
  for (int64_t k = b; k < e; ++k) { run += flag[k]; rank[k] = run - 1; }
}

struct VoxelWs {
  int64_t keys_in, keys_out, idx_in, idx_out, flags, rank, cub, total;
  size_t cub_bytes;
};

VoxelWs voxel_layout(int64_t n) {
  auto up = [](int64_t b) { return (b + 255) / 256 * 256; };
  VoxelWs w;
  size_t cub_bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const uint64_t*)nullptr, (uint64_t*)nullptr,
                                  (const int32_t*)nullptr, (int32_t*)nullptr, (int)n);
  w.cub_bytes = cub_bytes;
  int64_t off = 0;
  w.keys_in = off;  off += up(n * 8);
  w.keys_out = off; off += up(n * 8);
  w.idx_in = off;   off += up(n * 4);
  w.idx_out = off;  off += up(n * 4);
  w.flags = off;    off += up(n * 4);
  w.rank = off;     off += up(n * 4);
  w.cub = off;      off += up((int64_t)cub_bytes);
  w.total = off;
  return w;
}

}  // namespace

extern "C" {

int64_t b200icp_voxel_workspace_bytes(int64_t n) {
  if (n < 0 || n > 0x7fffffffLL) return -1;
  return voxel_layout(n > 0 ? n : 1).total;
}

int b200icp_voxel_downsample(const void* points, int32_t dtype, int64_t n, double voxel_size,
                             void* out_points, int64_t* count_out, void* workspace,
                             int64_t workspace_bytes, void* stream) {
  if (!points || !out_points || !count_out || !workspace) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "voxel_downsample: NULL pointer");
  if (dtype != B200ICP_F32 && dtype != B200ICP_F64) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "voxel_downsample: bad dtype");
  if (n < 1 || n > 0x7fffffffLL || !(voxel_size > 0.0)) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "voxel_downsample: need n >= 1 and voxel_size > 0");
  const VoxelWs w = voxel_layout(n);
  if (workspace_bytes < w.total) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "voxel_downsample: workspace too small");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  unsigned char* base = reinterpret_cast<unsigned char*>(workspace);
  uint64_t* keys_in = reinterpret_cast<uint64_t*>(base + w.keys_in);
  uint64_t* keys_out = reinterpret_cast<uint64_t*>(base + w.keys_out);
  int32_t* idx_in = reinterpret_cast<int32_t*>(base + w.idx_in);
  int32_t* idx_out = reinterpret_cast<int32_t*>(base + w.idx_out);
  int32_t* flags = reinterpret_cast<int32_t*>(base + w.flags);
  int32_t* rank = reinterpret_cast<int32_t*>(base + w.rank);
  const unsigned blocks = (unsigned)((n + 255) / 256);
  const double inv = 1.0 / voxel_size;
  // pass 1 by cell_x: keys_in, idx_in -> keys_out, idx_out; pass 2 by cell_y of that order:
  // keys_in, idx_out -> keys_out, idx_in.  Stable, so the result is (cell_y, cell_x, input order).
  voxel_key_x_kernel<<<blocks, 256, 0, st>>>(points, dtype, n, inv, keys_in, idx_in);
  size_t cub_bytes = w.cub_bytes;
  cudaError_t e = cub::DeviceRadixSort::SortPairs(base + w.cub, cub_bytes, keys_in, keys_out, idx_in, idx_out,
                                                  (int)n, 0, 64, st);
  if (e != cudaSuccess) return set_error(B200ICP_ERR_CUDA, "%s", cudaGetErrorString(e));
  voxel_key_y_kernel<<<blocks, 256, 0, st>>>(points, dtype, n, inv, idx_out, keys_in);
  cub_bytes = w.cub_bytes;
  e = cub::DeviceRadixSort::SortPairs(base + w.cub, cub_bytes, keys_in, keys_out, idx_out, idx_in, (int)n, 0, 64, st);
  if (e != cudaSuccess) return set_error(B200ICP_ERR_CUDA, "%s", cudaGetErrorString(e));
  voxel_head_kernel<<<blocks, 256, 0, st>>>(points, dtype, n, inv, keys_out, idx_in, flags);
  voxel_scan_kernel<<<1, 1024, 0, st>>>(flags, n, rank);
  voxel_emit_kernel<<<blocks, 256, 0, st>>>(points, dtype, n, keys_out, idx_in, flags, rank, out_points, count_out);
  e = cudaGetLastError();
  if (e != cudaSuccess) return set_error(B200ICP_ERR_CUDA, "%s", cudaGetErrorString(e));
  return B200ICP_OK;
}

}  // extern "C"
