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
// then by cell_y -> order (cell_y, cell_x, input order) -> compact() over the sorted points: every
// run head averages its run in the original point order (deterministic).  Points whose cell is not
// an int64 (non-finite coordinates, |p / voxel_size| >= 2^63) are skipped, as b200icp_occ_update
// skips non-finite points.
#include <cuda_runtime.h>

#include <cstdint>

#include "compact.cuh"
#include "workspace.cuh"

namespace {

// sort key of a skipped point: above every biased int64 cell (the largest cell of a double below
// 2^63 is 2^63 - 1024), so skipped points sort last and never join a cell's run
constexpr uint64_t kSkipKey = ~0ull;

// cell = floor(p / voxel) (d.py:11-12), biased to unsigned so that the radix order is the signed
// order; kSkipKey for both axes unless both cells are int64
__device__ __forceinline__ void vx_cell(double2 q, double inv_voxel, uint64_t& kx, uint64_t& ky) {
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
  vx_cell(load_point(points, dtype, i), inv_voxel, kx, ky);
  keys[i] = kx;
  idx[i] = (int32_t)i;
}

// cell_y of the points in cell_x order, for the second (stable) pass
__global__ void voxel_key_y_kernel(const void* points, int dtype, int64_t n, double inv_voxel,
                                   const int32_t* idx, uint64_t* keys) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t kx, ky;
  vx_cell(load_point(points, dtype, idx[i]), inv_voxel, kx, ky);
  keys[i] = ky;
}

// head of a run: a kept point whose cell differs from its predecessor's in sorted order.  The
// sorted cell_y keys decide most points without loading them; only equal cell_y compares cell_x.
struct VoxelHead {
  const void* points;
  int dtype;
  double inv_voxel;
  const uint64_t* keys_y;     // sorted
  const int32_t* idx;         // sorted position -> point
  __device__ __forceinline__ bool operator()(int64_t i) const {
    const uint64_t ky = keys_y[i];
    if (ky == kSkipKey) return false;
    if (i == 0 || ky != keys_y[i - 1]) return true;
    uint64_t ax, ay, bx, by;
    vx_cell(load_point(points, dtype, idx[i]), inv_voxel, ax, ay);
    vx_cell(load_point(points, dtype, idx[i - 1]), inv_voxel, bx, by);
    return ax != bx;
  }
};

// the mean of the run that starts at head i, summed in sorted order (both sorts are stable, so a
// run lists its points in the original order); skipped points sort last and end the last run
struct VoxelMean {
  const void* points;
  int dtype;
  double inv_voxel;
  const uint64_t* keys_y;
  const int32_t* idx;
  int64_t n;
  void* out;
  __device__ __forceinline__ void operator()(int64_t dst, int64_t i) const {
    double2 q = load_point(points, dtype, idx[i]);
    uint64_t hx, hy, kx, ky;
    vx_cell(q, inv_voxel, hx, hy);
    double sx = 0.0, sy = 0.0;
    int64_t k = i;
    for (;;) {
      sx += q.x; sy += q.y;
      if (++k == n || keys_y[k] != hy) break;     // the sorted cell_y ends most runs without a load
      q = load_point(points, dtype, idx[k]);
      vx_cell(q, inv_voxel, kx, ky);
      if (kx != hx) break;
    }
    const double inv = 1.0 / (double)(k - i);
    if (dtype == B200ICP_F64) reinterpret_cast<double2*>(out)[dst] = make_double2(sx * inv, sy * inv);
    else reinterpret_cast<float2*>(out)[dst] = make_float2((float)(sx * inv), (float)(sy * inv));
  }
};

struct VoxelBuffers {
  uint64_t *keys_in, *keys_out;
  int32_t *idx_in, *idx_out;
  int64_t* scratch;      // compact()
  SortTemp sort;
  int64_t bytes;
};

VoxelBuffers voxel_buffers(void* base, int64_t n) {
  Carver c(base);
  VoxelBuffers b;
  b.keys_in = c.take<uint64_t>(n);
  b.keys_out = c.take<uint64_t>(n);
  b.idx_in = c.take<int32_t>(n);
  b.idx_out = c.take<int32_t>(n);
  b.scratch = c.take<int64_t>(compact_scratch_len(n));
  b.sort = take_sort_temp<uint64_t, int32_t>(c, n);
  b.bytes = c.total;
  return b;
}

}  // namespace

extern "C" {

int64_t b200icp_voxel_workspace_bytes(int64_t n) {
  if (n < 0 || n > 0x7fffffffLL) return -1;
  return voxel_buffers(nullptr, n > 0 ? n : 1).bytes;
}

int b200icp_voxel_downsample(const void* points, int32_t dtype, int64_t n, double voxel_size,
                             void* out_points, int64_t* count_out, void* workspace,
                             int64_t workspace_bytes, void* stream) {
  if (!points || !out_points || !count_out || !workspace) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "voxel_downsample: NULL pointer");
  if (dtype != B200ICP_F32 && dtype != B200ICP_F64) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "voxel_downsample: bad dtype");
  if (n < 1 || n > 0x7fffffffLL || !(voxel_size > 0.0)) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "voxel_downsample: need n >= 1 and voxel_size > 0");
  const VoxelBuffers b = voxel_buffers(workspace, n);
  if (workspace_bytes < b.bytes) return set_error(B200ICP_ERR_INVALID_ARGUMENT, "voxel_downsample: workspace too small");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const unsigned blocks = (unsigned)((n + 255) / 256);
  const double inv = 1.0 / voxel_size;
  // pass 1 by cell_x: keys_in, idx_in -> keys_out, idx_out; pass 2 by cell_y of that order:
  // keys_in, idx_out -> keys_out, idx_in.  Stable, so the result is (cell_y, cell_x, input order).
  voxel_key_x_kernel<<<blocks, 256, 0, st>>>(points, dtype, n, inv, b.keys_in, b.idx_in);
  if (const int rc = radix_sort_pairs(b.sort, b.keys_in, b.keys_out, b.idx_in, b.idx_out, n, 0, 64, st,
                                      "voxel_downsample: radix sort"))
    return rc;
  voxel_key_y_kernel<<<blocks, 256, 0, st>>>(points, dtype, n, inv, b.idx_out, b.keys_in);
  if (const int rc = radix_sort_pairs(b.sort, b.keys_in, b.keys_out, b.idx_out, b.idx_in, n, 0, 64, st,
                                      "voxel_downsample: radix sort"))
    return rc;
  return compact(VoxelHead{points, dtype, inv, b.keys_out, b.idx_in},
                 VoxelMean{points, dtype, inv, b.keys_out, b.idx_in, n, out_points}, n, b.scratch, count_out, st, "voxel");
}

}  // extern "C"
