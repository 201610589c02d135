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

// chat (need_expand), then per t = T-1 ... 0 the Q step, the PNQP factor step and the V step (t >= 1), then the line
// search.  Scratch: large_fwd_ws_bytes (fp64), c_hat [T,B,s] in R, the per-element flags [B].
template <typename R>
int launch_mpc_large_forward(const MpcFwdParams<R>& p, cudaStream_t st, long long* nl) {
  const int n = p.n, m = p.m, s = n + m, B = p.B, T = p.T;
  if (!lqr_large_shape_ok(n, m) || p.coupling == DMPC_COUPLING_BATCH || p.dynamics != DMPC_DYN_LINEAR) return DMPC_ERR_UNSUPPORTED;
  const bool expand = p.need_expand != 0;
  const size_t o_chat = al256(large_fwd_ws_bytes(B, n, m));
  const size_t o_fl = al256(o_chat + (expand ? sizeof(R) * (size_t)T * B * s : 0));
  char* ws = nullptr;
  if (cudaMallocAsync((void**)&ws, o_fl + sizeof(int) * B, st) != cudaSuccess) return DMPC_ERR_CUDA;
  R* chat = expand ? (R*)(ws + o_chat) : nullptr;
  int* eflags = (int*)(ws + o_fl);
  int rc = cudaMemsetAsync(eflags, 0, sizeof(int) * B, st) == cudaSuccess ? DMPC_OK : DMPC_ERR_CUDA;
  // the Riccati steps of lqr_large_kernels.cuh on the model (C, c_hat or c, F, f unless need_expand: mpc_step.py:317)
  LqrParams<R> q;
  memset(&q, 0, sizeof(q));
  q.T = T; q.B = B; q.n = n; q.m = m; q.flags = LQR_DO_FACTOR;
  q.C = p.C; q.c = expand ? chat : p.c; q.c_scale = R(1); q.F = p.F; q.f = expand ? nullptr : p.f; q.skip = p.skip;
  const size_t smp = sizeof(double) * mpc_large_pnqp_smem(n, m), sml = sizeof(double) * (3 * s + 2 * n + 1);
  if (!rc) rc = set_smem(mpc_large_pnqp_kernel<R>, smp);
  if (!rc && expand) rc = launch(mpc_large_chat_kernel<R>, dim3(B, T), kLargeThreads, sizeof(double) * s, st, nl, p, chat);
  if (!rc) rc = large_riccati_steps<R>(q, (double*)ws, (R*)nullptr, [&](const LargeFwdWs& w, int t) {
    return launch(mpc_large_pnqp_kernel<R>, B, kLargeThreads, smp, st, nl, p, w, eflags, t);
  }, st, nl);
  if (!rc) rc = launch(mpc_large_ls_kernel<R>, B, kLargeThreads, sml, st, nl, p, eflags);
  if (cudaFreeAsync(ws, st) != cudaSuccess && !rc) rc = DMPC_ERR_CUDA;
  return rc;
}

template <typename R>
int launch_traj_large(const TrajParams<R>& p, cudaStream_t st, long long* nl) {
  if (!lqr_large_shape_ok(p.n, p.m) || p.dynamics != DMPC_DYN_LINEAR) return DMPC_ERR_UNSUPPORTED;
  return launch(traj_large_kernel<R>, p.B, kLargeThreads, sizeof(double) * (p.n + p.m + p.n), st, nl, p);
}

template int launch_mpc_large_forward<DMPC_REAL>(const MpcFwdParams<DMPC_REAL>&, cudaStream_t, long long*);
template int launch_traj_large<DMPC_REAL>(const TrajParams<DMPC_REAL>&, cudaStream_t, long long*);

}  // namespace dmpc
