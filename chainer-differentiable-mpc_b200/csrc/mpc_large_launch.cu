// Launch sequences of the large-system MPC step forward and get_traj (mpc_large_kernels.cuh, DESIGN.md §4.9).
// Compiled once per dtype (-DDMPC_REAL).  mpc_launch.cu selects them where the per-element kernels do not fit.
#include <cstring>
#include "launch.h"
#include "mpc_large_kernels.cuh"
#include "mpc_launch.h"

#ifndef DMPC_REAL
#define DMPC_REAL double
#endif

namespace dmpc {

namespace {
template <typename K>
int set_smem(K kernel, size_t bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) == cudaSuccess ? DMPC_OK : DMPC_ERR_CUDA;
}
inline int launched(long long* nl) {
  if (nl) ++*nl;
  return cudaGetLastError() == cudaSuccess ? DMPC_OK : DMPC_ERR_CUDA;
}
inline size_t al256(size_t v) { return (v + 255) & ~(size_t)255; }
}  // namespace

// chat (need_expand), then per t = T-1 ... 0 the Q step, the PNQP factor step and the V step (t >= 1), then the line
// search.  Scratch: LargeFwdWs (fp64), c_hat [T,B,s] in R, the per-element flags [B].
template <typename R>
int launch_mpc_large_forward(const MpcFwdParams<R>& p, cudaStream_t st, long long* nl) {
  const int n = p.n, m = p.m, s = n + m, B = p.B, T = p.T;
  if (!lqr_large_shape_ok(n, m) || p.coupling == DMPC_COUPLING_BATCH || p.dynamics != DMPC_DYN_LINEAR) return DMPC_ERR_UNSUPPORTED;
  const bool expand = p.need_expand != 0;
  const size_t nV = (size_t)n * (n + 1), nQ = (size_t)s * (s + 1), nK = (size_t)m * (n + 1);
  const size_t o_chat = al256(sizeof(double) * B * (nV + nQ + 2 * nK));
  const size_t o_fl = al256(o_chat + (expand ? sizeof(R) * (size_t)T * B * s : 0));
  char* ws = nullptr;
  if (cudaMallocAsync((void**)&ws, o_fl + sizeof(int) * B, st) != cudaSuccess) return DMPC_ERR_CUDA;
  double* d = (double*)ws;
  LargeFwdWs w{d, d + (size_t)B * nV, d + (size_t)B * (nV + nQ), d + (size_t)B * (nV + nQ + nK)};
  R* chat = expand ? (R*)(ws + o_chat) : nullptr;
  int* eflags = (int*)(ws + o_fl);
  int rc = cudaMemsetAsync(eflags, 0, sizeof(int) * B, st) == cudaSuccess ? DMPC_OK : DMPC_ERR_CUDA;
  // the Riccati steps of lqr_large_kernels.cuh on the model (C, c_hat or c, F, f unless need_expand: mpc_step.py:317)
  LqrParams<R> q;
  memset(&q, 0, sizeof(q));
  q.T = T; q.B = B; q.n = n; q.m = m; q.flags = LQR_DO_FACTOR;
  q.C = p.C; q.c = expand ? chat : p.c; q.c_scale = R(1); q.F = p.F; q.f = expand ? nullptr : p.f; q.skip = p.skip;
  const size_t smq = sizeof(double) * n * kLargePanel, smp = sizeof(double) * mpc_large_pnqp_smem(n, m);
  const size_t sml = sizeof(double) * (3 * s + 2 * n + 1);
  if (!rc) rc = set_smem(lqr_large_q_kernel<R>, smq);
  if (!rc) rc = set_smem(mpc_large_pnqp_kernel<R>, smp);
  if (!rc && expand) {
    mpc_large_chat_kernel<R><<<dim3(B, T), kLargeThreads, sizeof(double) * s, st>>>(p, chat);
    rc = launched(nl);
  }
  const dim3 gq(B, (s + 1 + kLargePanel - 1) / kLargePanel), gv(B, (n + 1 + kLargePanel - 1) / kLargePanel);
  for (int t = T - 1; t >= 0 && !rc; --t) {
    lqr_large_q_kernel<R><<<gq, kLargeThreads, smq, st>>>(q, w, t);
    rc = launched(nl);
    if (rc) break;
    mpc_large_pnqp_kernel<R><<<B, kLargeThreads, smp, st>>>(p, w, eflags, t);
    rc = launched(nl);
    if (rc || t == 0) break;
    lqr_large_v_kernel<R><<<gv, kLargeThreads, 0, st>>>(q, w, (R*)nullptr, t);
    rc = launched(nl);
  }
  if (!rc) {
    mpc_large_ls_kernel<R><<<B, kLargeThreads, sml, st>>>(p, eflags);
    rc = launched(nl);
  }
  if (cudaFreeAsync(ws, st) != cudaSuccess && !rc) rc = DMPC_ERR_CUDA;
  return rc;
}

template <typename R>
int launch_traj_large(const TrajParams<R>& p, cudaStream_t st, long long* nl) {
  if (!lqr_large_shape_ok(p.n, p.m) || p.dynamics != DMPC_DYN_LINEAR) return DMPC_ERR_UNSUPPORTED;
  traj_large_kernel<R><<<p.B, kLargeThreads, sizeof(double) * (p.n + p.m + p.n), st>>>(p);
  return launched(nl);
}

template int launch_mpc_large_forward<DMPC_REAL>(const MpcFwdParams<DMPC_REAL>&, cudaStream_t, long long*);
template int launch_traj_large<DMPC_REAL>(const TrajParams<DMPC_REAL>&, cudaStream_t, long long*);

}  // namespace dmpc
