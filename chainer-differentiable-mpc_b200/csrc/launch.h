// Host-side launch interfaces between capi.cu and the kernel translation units.
#pragma once
#include <cuda_runtime.h>
#include "lqr_kernels.cuh"
#include "lqr_adjoint_fused.cuh"
#include "lqr_shared_kernels.cuh"

namespace dmpc {

// Which (n, m) shapes have compile-time-specialised kernels (everything else runs the
// runtime-shape instantiation of the same code).
struct ShapeInfo { int n, m, G; bool specialised; };

template <typename R> int launch_lqr_solve(const LqrParams<R>& p, cudaStream_t st, long long* nlaunch);
// n=32, m=8: warp-per-element DMMA Riccati sweep + fused rollout (lqr_dmma_launch.cu)
template <typename R> int launch_lqr_solve_dmma(const LqrParams<R>& p, cudaStream_t st, long long* nlaunch);
// rollout-only launch of the generic kernel at n=32, m=8 (lqr_launch.cu)
template <typename R> int launch_lqr_rollout_32_8(const LqrParams<R>& p, cudaStream_t st, long long* nlaunch);
template <typename R> int launch_lqr_dtau(const DtauParams<R>& p, cudaStream_t st, long long* nlaunch);
// two-sweep adjoint (lqr_adjoint_fused.cuh); DMPC_ERR_UNSUPPORTED when the shape has no instantiation
#define DMPC_FUSED_SHAPES(X) X(32, 8)
// stage: 0 = both sweeps, 1 = sweep 1 only, 2 = sweep 2 only (bench.py's per-kernel timing)
template <typename R> int launch_adjoint_fused(const DtauParams<R>& d, const AdjFusedParams<R>& a, int stage, cudaStream_t st, long long* nlaunch);
template <typename R> int launch_adjoint_out(const AdjOutParams<R>& p, cudaStream_t st, long long* nlaunch);
template <typename R> int launch_expand_time_batch(const R* src, R* dst, int count, size_t total, cudaStream_t st, long long* nlaunch);
// C and F shared by the batch (lqr_shared_launch.cu): the chunked vector sweeps + rollout; the adjoint + reduction
template <typename R> int launch_lqr_shared_fwd(const LqrSharedParams<R>& p, cudaStream_t st, long long* nlaunch);
template <typename R> int launch_lqr_shared_adj(const LqrSharedParams<R>& p, cudaStream_t st, long long* nlaunch);
template <typename R> int launch_reduce_partials(const R* red, int B, int rsz, R* out, cudaStream_t st, long long* nlaunch);

constexpr int kMaxSmem = 227 * 1024;

// Systems whose per-element step does not fit one CTA (lqr_large_launch.cu, DESIGN.md §4.8, §4.9).  *_selected: the
// per-element kernels would return DMPC_ERR_UNSUPPORTED for shared memory; the launchers return DMPC_ERR_UNSUPPORTED
// outside n <= 128, m <= 32 before launching anything.
inline bool lqr_large_shape_ok(int n, int m) { return n >= 1 && n <= 128 && m >= 1 && m <= 32; }
template <typename R> bool lqr_large_solve_selected(int n, int m, int lqr_flags);
template <typename R> bool lqr_large_adjoint_selected(int n, int m, bool reduced);
// adjoint_out_kernel alone (lambda / d-lambda stage of the MPC step backward)
template <typename R> bool lqr_large_adj_out_selected(int n, int m, bool reduced);
template <typename R> int launch_lqr_large_solve(const LqrParams<R>& p, cudaStream_t st, long long* nlaunch);
// stage: 0 = whole adjoint, 1 = d-tau sweeps only, 2 = lambda recursion + gradients only
template <typename R> int launch_lqr_large_adjoint(const AdjOutParams<R>& a, const R* Ks, const R* fac, int stage,
                                                   cudaStream_t st, long long* nlaunch);

}  // namespace dmpc
