#pragma once
#include "mpc_kernels.cuh"
namespace dmpc {
template <typename R> int launch_mpc_forward(const MpcFwdParams<R>& p, cudaStream_t st, long long* nl);
template <typename R> int launch_pnqp(const PnqpParams<R>& p, cudaStream_t st, long long* nl);
template <typename R> int launch_active_mask(const R* u, const R* lo, const R* hi, unsigned char* out, size_t count,
                                             cudaStream_t st, long long* nl);
template <typename R> int launch_traj(const TrajParams<R>& p, cudaStream_t st, long long* nl);
// systems whose per-element step does not fit one CTA (mpc_large_launch.cu, DESIGN.md §4.9): element coupling and
// LinDx only, n <= 128, m <= 32; DMPC_ERR_UNSUPPORTED otherwise, before launching anything
template <typename R> int launch_mpc_large_forward(const MpcFwdParams<R>& p, cudaStream_t st, long long* nl);
template <typename R> int launch_traj_large(const TrajParams<R>& p, cudaStream_t st, long long* nl);
}  // namespace dmpc
