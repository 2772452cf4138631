// launch.cuh -- launch functions of the pair-batch kernel families (align_cta.cu, align_pair.cu),
// called by the dispatch of b200icp_nn_batch / b200icp_align_batch in b200icp.cu.
#pragma once

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

// One launch per call, opted in to the most dynamic shared memory the device allows when the shape
// needs more than 48 KB.
template <typename Kern, typename Args>
int launch_pairs(Kern kern, const LaunchShape& ls, const Args& args, cudaStream_t st) {
  if (ls.smem > 48 * 1024)
    if (const int rc = opt_in_dynamic_smem(reinterpret_cast<const void*>(kern), -1)) return rc;
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
