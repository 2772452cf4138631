// launch.cuh -- launch functions of the pair-batch kernel families (align_cta.cu, align_pair.cu),
// called by the dispatch of b200icp_nn_batch / b200icp_align_batch in b200icp.cu.
#pragma once

#include <mutex>
#include <set>
#include <utility>

#include "common.cuh"

struct LaunchShape {
  int S;           // CTA-per-pair kernels: source points per lane
  int warps;
  size_t smem;
  int mcap;
};

// Launch shape of the CTA-per-pair kernels; false if src_pitch needs more than kMaxWarps warps.
bool pick_shape(const b200icp_problem* pr, LaunchShape& ls);

// align_cta.cu: one CTA per pair
int launch_nn_cta_kernel(const LaunchShape& ls, const KernelArgs& args, cudaStream_t st);
int launch_align_cta_kernel(const LaunchShape& ls, const KernelArgs& args, cudaStream_t st);

// align_pair.cu: W warps per pair (fused ICP loop) and one warp per pair (search only)
int launch_pair_kernel(const b200icp_problem* prob, const LaunchShape& ls, KernelArgs& args, bool dense,
                       int forced_warps, cudaStream_t st);
int launch_nn_warp_kernel(const b200icp_problem* prob, const LaunchShape& ls, KernelArgs& args, bool dense,
                          cudaStream_t st);

// One launch per call.  The opt-in to more than 48 KB of dynamic shared memory is made once per
// kernel and device (the largest size the device allows), not on every launch.
template <typename Kern, typename Args>
int launch_pairs(Kern kern, const LaunchShape& ls, const Args& args, cudaStream_t st) {
  if (ls.smem > 48 * 1024) {
    // (all kernels share the function-pointer type, so the memo is keyed by pointer and device)
    static std::mutex mu;
    static std::set<std::pair<const void*, int>> opted_in;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lock(mu);
    const std::pair<const void*, int> key(reinterpret_cast<const void*>(kern), dev);
    if (!opted_in.count(key)) {
      int max_optin = 0;
      cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin);
      if (e != cudaSuccess)
        return set_error(B200ICP_ERR_CUDA, "cudaFuncSetAttribute(max dynamic smem): %s", cudaGetErrorString(e));
      opted_in.insert(key);
    }
  }
  kern<<<(unsigned)args.n_pairs, ls.warps * 32, ls.smem, st>>>(args);
  return check_launch("kernel launch");
}

// The CTA-per-pair kernels are instantiated for S = 1..4 source points per lane.
#define B200ICP_DISPATCH_CTA(KERNEL)                                         \
  switch (ls.S) {                                                            \
    case 1: return launch_pairs(KERNEL<1>, ls, args, st);                    \
    case 2: return launch_pairs(KERNEL<2>, ls, args, st);                    \
    case 3: return launch_pairs(KERNEL<3>, ls, args, st);                    \
    default: return launch_pairs(KERNEL<4>, ls, args, st);                   \
  }
