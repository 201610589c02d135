// Launches of the large-system LQR kernels (lqr_large_kernels.cuh).  Compiled once per dtype (-DDMPC_REAL).
#include "launch.h"
#include "lqr_large_kernels.cuh"

#ifndef DMPC_REAL
#define DMPC_REAL double
#endif

namespace dmpc {

// launch_lqr_solve, launch_lqr_adjoint and launch_adjoint_out (lqr_launch.cu) take these kernels where the per-element
// kernels' layout does not fit one CTA's shared memory.
template <typename R>
int launch_lqr_large_solve(const LqrParams<R>& p, cudaStream_t st, long long* nl) {
  const int n = p.n, m = p.m, s = n + m, B = p.B, T = p.T;
  if (!lqr_large_shape_ok(n, m)) return DMPC_ERR_UNSUPPORTED;
  int rc = DMPC_OK;
  if (p.flags & LQR_DO_FACTOR) {
    // V_t | v_t into the caller's factor cache (the slot dmpc_lqr_fac_elems reserves) or the shared path's Vsave
    R* Vdst = p.Vsave ? p.Vsave : ((p.flags & LQR_SAVE_FAC) && p.fac ? p.fac + (size_t)T * B * (m * m + n * m) : nullptr);
    double* ws = nullptr;
    if (cudaMallocAsync((void**)&ws, large_fwd_ws_bytes(B, n, m), st) != cudaSuccess) return DMPC_ERR_CUDA;
    const size_t smf = sizeof(double) * (m * m + m * (n + 1 + m));
    rc = set_smem(lqr_large_factor_kernel<R>, smf);
    if (!rc) rc = large_riccati_steps<R>(p, ws, Vdst, [&](const LargeFwdWs& w, int t) {
      return launch(lqr_large_factor_kernel<R>, B, kLargeThreads, smf, st, nl, p, w, t);
    }, st, nl);
    if (cudaFreeAsync(ws, st) != cudaSuccess && !rc) rc = DMPC_ERR_CUDA;
    if (rc) return rc;
  }
  if (p.flags & LQR_DO_ROLLOUT) rc = launch(lqr_large_rollout_kernel<R>, B, kLargeThreads, sizeof(double) * (s + n), st, nl, p);
  return rc;
}

// stage: 0 = everything, 1 = the d-tau sweeps only, 2 = lambda recursion and outer products only (re-using dtau)
template <typename R>
int launch_lqr_large_adjoint(const AdjOutParams<R>& a, const R* Ks, const R* fac, int stage, cudaStream_t st, long long* nl) {
  const int n = a.n, m = a.m, s = n + m, B = a.B, T = a.T;
  if (!lqr_large_shape_ok(n, m)) return DMPC_ERR_UNSUPPORTED;
  const bool red = (a.flags & ADJ_REDUCE_TB) != 0;
  double* ws = nullptr;
  if (cudaMallocAsync((void**)&ws, sizeof(double) * 2 * (size_t)T * B * n, st) != cudaSuccess) return DMPC_ERR_CUDA;
  LargeAdjWs w{ws, ws + (size_t)T * B * n};
  int rc = launch(lqr_large_adj_kernel<R>, B, kLargeThreads, sizeof(double) * (3 * s + 4 * n + m), st, nl, a, Ks, fac, w,
                  stage != 2, stage != 1);
  if (!rc && stage != 1) {
    if (red) rc = launch(lqr_large_red_kernel<R>, dim3(B, (s + kLargePanel - 1) / kLargePanel), kLargeThreads, 0, st, nl, a, w);
    else rc = launch(lqr_large_outer_kernel<R>, dim3(B, T), kLargeThreads, 0, st, nl, a, w);
  }
  if (cudaFreeAsync(ws, st) != cudaSuccess && !rc) rc = DMPC_ERR_CUDA;
  return rc;
}

template int launch_lqr_large_solve<DMPC_REAL>(const LqrParams<DMPC_REAL>&, cudaStream_t, long long*);
template int launch_lqr_large_adjoint<DMPC_REAL>(const AdjOutParams<DMPC_REAL>&, const DMPC_REAL*, const DMPC_REAL*, int, cudaStream_t, long long*);

}  // namespace dmpc
