// Launches of the shared-parameter LQR kernels (lqr_shared_kernels.cuh).  Compiled once per dtype (-DDMPC_REAL).
#include "launch.h"

#ifndef DMPC_REAL
#define DMPC_REAL double
#endif

namespace dmpc {

template <typename K, typename P>
static int shared_launch(K kernel, const P& p, size_t smem, cudaStream_t st, long long* nl) {
  if (set_smem(kernel, smem)) return DMPC_ERR_CUDA;
  return launch(kernel, (p.B + p.NB - 1) / p.NB, kSharedThreads, smem, st, nl, p);
}

template <typename R>
int launch_lqr_shared_fwd(const LqrSharedParams<R>& p, cudaStream_t st, long long* nl) {
  const size_t smem = (size_t)SharedFwdLayout(p.n, p.m, p.NB).total * sizeof(R);
  if (p.c_shared && !p.f) return shared_launch(lqr_shared_rollout_kernel<R>, p, smem, st, nl);   // k_t is the sweep's ks
  return shared_launch(lqr_shared_fwd_kernel<R>, p, smem, st, nl);
}

template <typename R>
int launch_lqr_shared_adj(const LqrSharedParams<R>& p, cudaStream_t st, long long* nl) {
  const size_t smem = (size_t)SharedAdjLayout(p.n, p.m, p.NB).total * sizeof(R);
  int rc = shared_launch(lqr_shared_adj_kernel<R>, p, smem, st, nl);
  if (rc) return rc;
  const size_t total = shared_reduce_outputs(p);
  const int tpb = 256;
  return launch(lqr_shared_reduce_kernel<R>, (unsigned)((total + tpb - 1) / tpb), tpb, 0, st, nl, p, (p.B + p.NB - 1) / p.NB);
}

template int launch_lqr_shared_fwd<DMPC_REAL>(const LqrSharedParams<DMPC_REAL>&, cudaStream_t, long long*);
template int launch_lqr_shared_adj<DMPC_REAL>(const LqrSharedParams<DMPC_REAL>&, cudaStream_t, long long*);

}  // namespace dmpc
