// Launch of the n=32, m=8 Riccati sweep on the FP64 tensor cores (lqr_dmma_warp.cuh): its own translation unit so that
// the 255-register kernel compiles in parallel with the generic kernels.  Compiled once per dtype (-DDMPC_REAL).
// R = float: the same kernel with float tensors in HBM and in the staging buffers, fp64 arithmetic.
#include <cstdlib>
#include "launch.h"
#include "lqr_dmma_warp.cuh"

#ifndef DMPC_REAL
#define DMPC_REAL double
#endif

namespace dmpc {

template <typename R>
int launch_lqr_solve_dmma(const LqrParams<R>& p, cudaStream_t st, long long* nl) {
  if (p.flags & LQR_DO_FACTOR) {
    constexpr int WPC = 4;
    const size_t smem = (size_t)WPC * WarpCfg::TOTAL * sizeof(double);
    auto kern = lqr_factor_dmma_warp_kernel<WPC, R>;
    if (set_smem(kern, smem)) return DMPC_ERR_CUDA;
    static int n_sm = 0;
    if (n_sm == 0) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev); }
    int grid = (p.B + WPC - 1) / WPC;                            // persistent: at most the 2 resident CTAs per SM
    if (grid > 2 * n_sm) grid = 2 * n_sm;
    return launch(kern, grid, WPC * 32, smem, st, nl, p);         // the rollout (if requested) is fused in
  }
  if (p.flags & LQR_DO_ROLLOUT) return launch_lqr_rollout_32_8<R>(p, st, nl);   // rollout-only: compact generic launch
  return DMPC_OK;
}

template int launch_lqr_solve_dmma<DMPC_REAL>(const LqrParams<DMPC_REAL>&, cudaStream_t, long long*);

}  // namespace dmpc
