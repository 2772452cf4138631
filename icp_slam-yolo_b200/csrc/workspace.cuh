// workspace.cuh -- the caller-provided device workspace of the entry points that sort
// (b200icp_voxel_downsample, b200icp_s2m_prepare_map, b200icp_pose_graph_optimize) and the cub radix
// sort they share.  Each entry point carves its buffers in one function; run on nullptr that function
// answers the matching *_workspace_bytes query, so the query and the launch cannot disagree.
#pragma once

#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"

// Hands out consecutive 256-byte-aligned parts of `base` (nullptr: sizes only, every part is nullptr);
// `total` is the size of the parts taken so far.
struct Carver {
  explicit Carver(void* b) : base(static_cast<unsigned char*>(b)) {}
  void* take_bytes(size_t n) {
    void* p = base ? base + total : nullptr;
    total += (int64_t)((n + 255) & ~(size_t)255);
    return p;
  }
  template <typename T>
  T* take(int64_t count) { return static_cast<T*>(take_bytes(sizeof(T) * (size_t)count)); }
  unsigned char* base;
  int64_t total = 0;
};

struct SortTemp {        // cub's temporary storage of one sort
  void* ptr;
  size_t bytes;
};

// Temporary storage for stable radix sorts of up to n (K, V) pairs over any bit range of K.
template <typename K, typename V>
SortTemp take_sort_temp(Carver& c, int64_t n) {
  size_t bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const K*)nullptr, (K*)nullptr, (const V*)nullptr, (V*)nullptr,
                                  (int)n);
  return SortTemp{c.take_bytes(bytes), bytes};
}

// Stable sort of n (key, value) pairs by bits [begin_bit, end_bit) of the key; a CUDA error becomes
// B200ICP_ERR_CUDA with the message "<what>: <CUDA error string>".
template <typename K, typename V>
int radix_sort_pairs(SortTemp t, const K* keys_in, K* keys_out, const V* vals_in, V* vals_out, int64_t n,
                     int begin_bit, int end_bit, cudaStream_t st, const char* what) {
  size_t bytes = t.bytes;
  const cudaError_t e = cub::DeviceRadixSort::SortPairs(t.ptr, bytes, keys_in, keys_out, vals_in, vals_out, (int)n,
                                                        begin_bit, end_bit, st);
  if (e != cudaSuccess) return set_error(B200ICP_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
  return B200ICP_OK;
}
