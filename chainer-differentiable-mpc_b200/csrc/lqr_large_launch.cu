// Selection and launches of the large-system LQR kernels (lqr_large_kernels.cuh).  Compiled once per dtype (-DDMPC_REAL).
#include "launch.h"
#include "lqr_large_kernels.cuh"

#ifndef DMPC_REAL
#define DMPC_REAL double
#endif

namespace dmpc {

// A call takes these kernels only where the per-element kernels cannot run it for shared memory: the same layout
// functions and the same kMaxSmem test as do_launch (one element per CTA at s > 24; smaller systems always fit).
// LQR_MASKED calls (the MPC step backward, LQR_active) are selected by the same test.
template <typename R>
bool lqr_large_solve_selected(int n, int m, int flags) {
  const LqrLayout L = lqr_layout<R>(n, m, (flags & LQR_SAVE_FAC) != 0, !(flags & LQR_DO_FACTOR));
  return m > 32 || (size_t)L.stride * sizeof(R) > (size_t)kMaxSmem;
}

// (the compile-time shapes' reduced adjoint keeps its sums in registers; all of them fit either way)
template <typename R>
bool lqr_large_adjoint_selected(int n, int m, bool reduced) {
  return (size_t)dtau_layout<R>(n, m).stride * sizeof(R) > (size_t)kMaxSmem ||
         (size_t)adj_layout<R>(n, m, reduced).stride * sizeof(R) > (size_t)kMaxSmem;
}

// The lambda / d-lambda stage alone (the MPC step backward, whose dtau comes from the masked solve): adjoint_out_kernel's
// layout test.
template <typename R>
bool lqr_large_adj_out_selected(int n, int m, bool reduced) {
  return (size_t)adj_layout<R>(n, m, reduced).stride * sizeof(R) > (size_t)kMaxSmem;
}

namespace {
template <typename K>
int set_smem(K kernel, size_t bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) == cudaSuccess ? DMPC_OK : DMPC_ERR_CUDA;
}
inline int launched(long long* nl) {
  if (nl) ++*nl;
  return cudaGetLastError() == cudaSuccess ? DMPC_OK : DMPC_ERR_CUDA;
}
}  // namespace

template <typename R>
int launch_lqr_large_solve(const LqrParams<R>& p, cudaStream_t st, long long* nl) {
  const int n = p.n, m = p.m, s = n + m, B = p.B, T = p.T;
  if (!lqr_large_shape_ok(n, m)) return DMPC_ERR_UNSUPPORTED;
  int rc = DMPC_OK;
  if (p.flags & LQR_DO_FACTOR) {
    // V_t | v_t into the caller's factor cache (the slot dmpc_lqr_fac_elems reserves) or the shared path's Vsave
    R* Vdst = p.Vsave ? p.Vsave : ((p.flags & LQR_SAVE_FAC) && p.fac ? p.fac + (size_t)T * B * (m * m + n * m) : nullptr);
    const size_t nV = (size_t)n * (n + 1), nQ = (size_t)s * (s + 1), nK = (size_t)m * (n + 1);
    double* ws = nullptr;
    if (cudaMallocAsync((void**)&ws, sizeof(double) * B * (nV + nQ + 2 * nK), st) != cudaSuccess) return DMPC_ERR_CUDA;
    LargeFwdWs w{ws, ws + (size_t)B * nV, ws + (size_t)B * (nV + nQ), ws + (size_t)B * (nV + nQ + nK)};
    const size_t smq = sizeof(double) * n * kLargePanel, smf = sizeof(double) * (m * m + m * (n + 1 + m));
    rc = set_smem(lqr_large_q_kernel<R>, smq);
    if (!rc) rc = set_smem(lqr_large_factor_kernel<R>, smf);
    const dim3 gq(B, (s + 1 + kLargePanel - 1) / kLargePanel), gv(B, (n + 1 + kLargePanel - 1) / kLargePanel);
    for (int t = T - 1; t >= 0 && !rc; --t) {
      lqr_large_q_kernel<R><<<gq, kLargeThreads, smq, st>>>(p, w, t);
      rc = launched(nl);
      if (rc) break;
      lqr_large_factor_kernel<R><<<B, kLargeThreads, smf, st>>>(p, w, t);
      rc = launched(nl);
      if (rc || t == 0) break;
      lqr_large_v_kernel<R><<<gv, kLargeThreads, 0, st>>>(p, w, Vdst, t);
      rc = launched(nl);
    }
    if (cudaFreeAsync(ws, st) != cudaSuccess && !rc) rc = DMPC_ERR_CUDA;
    if (rc) return rc;
  }
  if (p.flags & LQR_DO_ROLLOUT) {
    lqr_large_rollout_kernel<R><<<B, kLargeThreads, sizeof(double) * (s + n), st>>>(p);
    rc = launched(nl);
  }
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
  lqr_large_adj_kernel<R><<<B, kLargeThreads, sizeof(double) * (3 * s + 4 * n + m), st>>>(a, Ks, fac, w, stage != 2, stage != 1);
  int rc = launched(nl);
  if (!rc && stage != 1) {
    if (red) lqr_large_red_kernel<R><<<dim3(B, (s + kLargePanel - 1) / kLargePanel), kLargeThreads, 0, st>>>(a, w);
    else lqr_large_outer_kernel<R><<<dim3(B, T), kLargeThreads, 0, st>>>(a, w);
    rc = launched(nl);
  }
  if (cudaFreeAsync(ws, st) != cudaSuccess && !rc) rc = DMPC_ERR_CUDA;
  return rc;
}

template bool lqr_large_solve_selected<DMPC_REAL>(int, int, int);
template bool lqr_large_adjoint_selected<DMPC_REAL>(int, int, bool);
template bool lqr_large_adj_out_selected<DMPC_REAL>(int, int, bool);
template int launch_lqr_large_solve<DMPC_REAL>(const LqrParams<DMPC_REAL>&, cudaStream_t, long long*);
template int launch_lqr_large_adjoint<DMPC_REAL>(const AdjOutParams<DMPC_REAL>&, const DMPC_REAL*, const DMPC_REAL*, int, cudaStream_t, long long*);

}  // namespace dmpc
