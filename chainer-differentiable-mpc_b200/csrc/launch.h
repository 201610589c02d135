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

constexpr int kMaxSmem = 227 * 1024;

inline size_t al256(size_t v) { return (v + 255) & ~(size_t)255; }

// Raise a kernel's dynamic shared-memory limit to `bytes` (needed above 48 KB).  Each call costs host time: the
// large-system launchers, which step the horizon from the host, set it once per call.
template <typename K>
int set_smem(K kernel, size_t bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) == cudaSuccess ? DMPC_OK : DMPC_ERR_CUDA;
}

// Launch, count the launch in *nl, and report a launch error.
template <typename K, typename... A>
int launch(K kernel, dim3 grid, dim3 block, size_t smem, cudaStream_t st, long long* nl, A... args) {
  kernel<<<grid, block, smem, st>>>(args...);
  if (nl) ++*nl;
  return cudaGetLastError() == cudaSuccess ? DMPC_OK : DMPC_ERR_CUDA;
}

// launch_lqr_solve, launch_lqr_adjoint and launch_adjoint_out pick the kernel family themselves: the per-element kernels,
// or the large-system kernels where the per-element layout does not fit one CTA's shared memory (DESIGN.md §4.8, §4.9).
// DMPC_ERR_UNSUPPORTED: no kernel runs the shape, and nothing was launched.
template <typename R> int launch_lqr_solve(const LqrParams<R>& p, cudaStream_t st, long long* nlaunch);
// n=32, m=8: warp-per-element DMMA Riccati sweep + fused rollout (lqr_dmma_launch.cu)
template <typename R> int launch_lqr_solve_dmma(const LqrParams<R>& p, cudaStream_t st, long long* nlaunch);
// rollout-only launch of the generic kernel at n=32, m=8 (lqr_launch.cu)
template <typename R> int launch_lqr_rollout_32_8(const LqrParams<R>& p, cudaStream_t st, long long* nlaunch);
// Shapes whose adjoint runs as two sweeps on the V_t, v_t saved by the forward (lqr_adjoint_fused.cuh); the solve saves
// them (LqrParams::Vsave) exactly where this holds.  DMPC_ADJ_UNFUSED=1 turns it off for A/B runs.
template <typename R> bool adjoint_fused_available(int n, int m);
// The whole adjoint of dmpc_lqr_adjoint[_reduced]: the two sweeps where adjoint_fused_available (full gradients with a
// df buffer, or the (T,B)-reduction), the large-system kernels, or lqr_dtau + adjoint_out; then, when a.red is set, the
// reduction of the per-element partials into `sums`.  stage: 0 = everything, 1 = the d-tau stage only, 2 = the rest only
// (bench.py's per-kernel timing).  On an error *failed is the message naming the launch, or nullptr when the shape is
// outside the large-system kernels' range.
template <typename R> int launch_lqr_adjoint(const DtauParams<R>& d, const AdjFusedParams<R>& f, const AdjOutParams<R>& a,
                                             int stage, R* sums, cudaStream_t st, long long* nlaunch, const char** failed);
// The lambda / d-lambda stage alone, on a d-tau the caller computed (the MPC step backward's masked solve), then the
// reduction into `sums` when p.red is set.  On an error *failed is the message naming the launch.
template <typename R> int launch_adjoint_out(const AdjOutParams<R>& p, R* sums, cudaStream_t st, long long* nlaunch,
                                             const char** failed);
template <typename R> int launch_expand_time_batch(const R* src, R* dst, int count, size_t total, cudaStream_t st, long long* nlaunch);
// C and F shared by the batch (lqr_shared_launch.cu): the chunked vector sweeps + rollout; the adjoint + reduction
template <typename R> int launch_lqr_shared_fwd(const LqrSharedParams<R>& p, cudaStream_t st, long long* nlaunch);
template <typename R> int launch_lqr_shared_adj(const LqrSharedParams<R>& p, cudaStream_t st, long long* nlaunch);

// Systems whose per-element step does not fit one CTA (lqr_large_launch.cu): DMPC_ERR_UNSUPPORTED outside n <= 128,
// m <= 32, before launching anything.
inline bool lqr_large_shape_ok(int n, int m) { return n >= 1 && n <= 128 && m >= 1 && m <= 32; }
template <typename R> int launch_lqr_large_solve(const LqrParams<R>& p, cudaStream_t st, long long* nlaunch);
// stage: 0 = whole adjoint, 1 = d-tau sweeps only, 2 = lambda recursion + gradients only
template <typename R> int launch_lqr_large_adjoint(const AdjOutParams<R>& a, const R* Ks, const R* fac, int stage,
                                                   cudaStream_t st, long long* nlaunch);

}  // namespace dmpc
