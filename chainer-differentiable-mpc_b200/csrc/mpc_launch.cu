// Kernel instantiation + shape dispatch for the MPC kernels (mpc_kernels.cuh).
// Compiled once per dtype (-DDMPC_REAL=double|float) so the two builds run in parallel.
#include "launch.h"
#include "mpc_kernels.cuh"
#include "mpc_tpe_kernel.cuh"
#include "mpc_launch.h"
#include <cstdlib>
#include <cstring>
#include <cstdio>

#ifndef DMPC_REAL
#define DMPC_REAL double
#endif

namespace dmpc {

typedef DMPC_REAL Rr;

// Launch `grid` CTAs as ONE thread-block cluster (batch coupling across CTAs: common.cuh batch_or).  Clusters of more than
// 8 CTAs are "non-portable" sizes the kernel has to opt in to; 16 is the hardware maximum on sm_100.
template <typename K, typename P>
static int launch_cluster(K kernel, const P& p, int grid, int tpb, size_t smem, cudaStream_t st) {
  if (grid > 8 && cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) return DMPC_ERR_CUDA;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3((unsigned)tpb); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)grid; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  P pc = p;
  const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, pc);
  if (e != cudaSuccess) fprintf(stderr, "diffmpc: cluster launch (%d CTAs x %d threads, %zu B smem) failed: %s\n", grid, tpb, smem, cudaGetErrorString(e));
  return e == cudaSuccess ? DMPC_OK : DMPC_ERR_CUDA;
}

static int check_launch(const char* what) {
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) fprintf(stderr, "diffmpc: %s launch failed: %s\n", what, cudaGetErrorString(e));
  return e == cudaSuccess ? DMPC_OK : DMPC_ERR_CUDA;
}

constexpr int kMaxClusterCtas = 16;
constexpr size_t kMpcMaxSmem = (size_t)kMaxSmem - 256;   // dynamic shared memory: the kernels also hold a few static words (batch_or flags)

template <typename K, typename P>
static int launch_elems(K kernel, const P& p, int G, size_t stride_bytes, int B, bool one_cta, cudaStream_t st,
                        long long* nl) {
  int tpb, epb, grid;
  bool cluster = false;
  if (G > 32) { tpb = G; epb = 1; grid = B; }
  else if (one_cta) {
    // batch coupling: the whole batch in one CTA, or spread evenly over the CTAs of one thread-block cluster
    cudaFuncAttributes fa;                          // the CTA size is capped by the kernel's register count too
    if (cudaFuncGetAttributes(&fa, kernel) != cudaSuccess) return DMPC_ERR_CUDA;
    int max_threads = fa.maxThreadsPerBlock;
    const int regs = ((fa.numRegs + 7) / 8) * 8;
    if (regs > 0 && 65536 / regs < max_threads) max_threads = 65536 / regs;
    max_threads = (max_threads / 32) * 32;
    if (max_threads > 1024) max_threads = 1024;
    int epb_max = max_threads / G;
    if ((size_t)epb_max * stride_bytes > kMpcMaxSmem) epb_max = (int)(kMpcMaxSmem / stride_bytes);
    if (epb_max < 1) return DMPC_ERR_UNSUPPORTED;
    grid = (B + epb_max - 1) / epb_max;
    if (grid > kMaxClusterCtas) return DMPC_ERR_UNSUPPORTED;    // batch coupling needs the batch resident in one cluster
    epb = (B + grid - 1) / grid;
    tpb = ((epb * G + 31) / 32) * 32;
    epb = tpb / G;                                 // padded groups replicate element B-1 in their own region
    if ((size_t)epb * stride_bytes > kMpcMaxSmem || tpb > max_threads) {
      epb = (epb_max * G / 32) * 32 / G;           // largest warp-multiple CTA within the limits
      if (epb < 1) return DMPC_ERR_UNSUPPORTED;
      tpb = ((epb * G + 31) / 32) * 32; grid = (B + epb - 1) / epb;
    }
    if (tpb > max_threads || grid > kMaxClusterCtas) return DMPC_ERR_UNSUPPORTED;
    cluster = grid > 1;
  } else {
    tpb = 128; epb = tpb / G;
    while ((size_t)epb * stride_bytes > kMpcMaxSmem && tpb > 32) { tpb /= 2; epb = tpb / G; }
    while (tpb > 32 && (B + epb - 1) / epb < 148 * 2) { tpb /= 2; epb = tpb / G; }
    grid = (B + epb - 1) / epb;
  }
  const size_t smem = (size_t)epb * stride_bytes;
  if (smem > kMpcMaxSmem) return DMPC_ERR_UNSUPPORTED;
  if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return DMPC_ERR_CUDA;
  if (nl) ++*nl;
  if (cluster) return launch_cluster(kernel, p, grid, tpb, smem, st);
  kernel<<<grid, tpb, smem, st>>>(p);
  return check_launch("element-group kernel");
}

#define MPC_SHAPES(X) X(3, 1, 4) X(4, 2, 8) X(8, 4, 16)

// m = 1, n <= 3: one thread per element, everything in registers (mpc_tpe_kernel.cuh).  DMPC_MPC_GROUP=1 selects the
// group-per-element kernel for A/B runs.
template <int N>
static int launch_mpc_tpe(const MpcFwdParams<Rr>& p_in, bool batch, cudaStream_t st, long long* nl) {
  // four candidate lanes per element (speculative parallel line search) while the K_t, k_t hand-over fits shared memory
  // and - for batch coupling - the whole batch still fits one 256-thread CTA; otherwise one lane per element.  When the
  // candidate trajectories of lanes 1..3 fit too, they are stashed there (the winner copies instead of re-rolling).
  MpcFwdParams<Rr> p = p_in;
  const size_t kk = (size_t)tpe_kk_stride(p.T, N) * sizeof(Rr);            // bytes per element
  const size_t ks = kk + 3 * (size_t)tpe_stash_stride(p.T, N) * sizeof(Rr);
  static int spec = -1, stash_ok = -1;
  if (spec < 0) { const char* e = getenv("DMPC_MPC_NO_SPEC"); spec = (e && e[0] == '1') ? 0 : 1; }
  if (stash_ok < 0) { const char* e = getenv("DMPC_MPC_NO_STASH"); stash_ok = (e && e[0] == '1') ? 0 : 1; }
  if (batch) {
    const int t4 = ((p.B * 4 + 31) / 32) * 32, t1 = ((p.B + 31) / 32) * 32;
    if (spec && t4 <= 256 && (t4 / 4) * kk <= (size_t)kMaxSmem) {
      auto k = mpc_forward_tpe_kernel<Rr, N, true, 256, 4>;
      p.tpe_stash = (stash_ok && (t4 / 4) * ks <= (size_t)kMaxSmem) ? 1 : 0;
      const size_t sm = (t4 / 4) * (p.tpe_stash ? ks : kk);
      if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm) != cudaSuccess) return DMPC_ERR_CUDA;
      k<<<1, t4, sm, st>>>(p);
    } else if (t1 <= 256) mpc_forward_tpe_kernel<Rr, N, true, 256, 1><<<1, t1, 0, st>>>(p);
    else {
      // the batch spread over the CTAs of one thread-block cluster, 256 threads (255 registers) per CTA
      const int grid = (p.B + 255) / 256;
      if (grid > kMaxClusterCtas) return DMPC_ERR_UNSUPPORTED;   // batch coupling: at most 16 x 256 elements
      const int tpb = ((((p.B + grid - 1) / grid) + 31) / 32) * 32;
      if (nl) ++*nl;
      return launch_cluster(mpc_forward_tpe_kernel<Rr, N, true, 256, 1>, p, grid, tpb, 0, st);
    }
  } else {
    const int epb = 16;                                            // elements per CTA: many small CTAs spread over the SMs
    if (spec && epb * kk <= (size_t)kMaxSmem) {
      auto k = mpc_forward_tpe_kernel<Rr, N, false, 256, 4>;
      p.tpe_stash = (stash_ok && epb * ks <= (size_t)kMaxSmem / 3) ? 1 : 0;      // keep three CTAs per SM resident
      const size_t sm = epb * (p.tpe_stash ? ks : kk);
      if (cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm) != cudaSuccess) return DMPC_ERR_CUDA;
      k<<<(p.B + epb - 1) / epb, epb * 4, sm, st>>>(p);
    } else {
      const int tpb = p.B >= 148 * 128 ? 64 : 32;
      mpc_forward_tpe_kernel<Rr, N, false, 256, 1><<<(p.B + tpb - 1) / tpb, tpb, 0, st>>>(p);
    }
  }
  if (nl) ++*nl;
  return check_launch("mpc_forward_tpe_kernel");
}

static bool mpc_tpe_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("DMPC_MPC_GROUP"); v = (e && e[0] == '1') ? 0 : 1; }
  return v == 1;
}

template <>
int launch_mpc_forward<Rr>(const MpcFwdParams<Rr>& p, cudaStream_t st, long long* nl) {
  if (p.m == 1 && mpc_tpe_enabled() && (p.dynamics == DMPC_DYN_LINEAR || p.n == 3)) {
    const bool b = p.coupling == DMPC_COUPLING_BATCH;
    if (!(b && p.B > kMaxClusterCtas * 256)) {
      if (p.n == 3) return launch_mpc_tpe<3>(p, b, st, nl);
      if (p.n == 2) return launch_mpc_tpe<2>(p, b, st, nl);
    }
  }
  const MpcLayout L = mpc_layout<Rr>(p.n, p.m);
  const size_t sb = (size_t)L.stride * sizeof(Rr);
  const bool batch = p.coupling == DMPC_COUPLING_BATCH;
  if (p.m > 32) return DMPC_ERR_UNSUPPORTED;
#define X(N_, M_, G_)                                                                                              \
  if (p.n == N_ && p.m == M_) {                                                                                    \
    if (batch) return launch_elems(mpc_forward_kernel<Rr, N_, M_, G_, true>, p, G_, sb, p.B, true, st, nl);        \
    return launch_elems(mpc_forward_kernel<Rr, N_, M_, G_, false>, p, G_, sb, p.B, false, st, nl);                 \
  }
  MPC_SHAPES(X)
#undef X
  const int s = p.n + p.m;
  if (s <= 6 && p.m <= 8) {
    if (batch) return launch_elems(mpc_forward_kernel<Rr, 0, 0, 8, true>, p, 8, sb, p.B, true, st, nl);
    return launch_elems(mpc_forward_kernel<Rr, 0, 0, 8, false>, p, 8, sb, p.B, false, st, nl);
  }
  if (s <= 14 && p.m <= 16) {
    if (batch) return launch_elems(mpc_forward_kernel<Rr, 0, 0, 16, true>, p, 16, sb, p.B, true, st, nl);
    return launch_elems(mpc_forward_kernel<Rr, 0, 0, 16, false>, p, 16, sb, p.B, false, st, nl);
  }
  if (s <= 24) {
    if (batch) return launch_elems(mpc_forward_kernel<Rr, 0, 0, 32, true>, p, 32, sb, p.B, true, st, nl);
    return launch_elems(mpc_forward_kernel<Rr, 0, 0, 32, false>, p, 32, sb, p.B, false, st, nl);
  }
  if (batch) return DMPC_ERR_UNSUPPORTED;
  // one element per CTA does not fit shared memory (launch_elems' test): the host-stepped large-system kernels
  if (sb > kMpcMaxSmem) return launch_mpc_large_forward<Rr>(p, st, nl);
  return launch_elems(mpc_forward_kernel<Rr, 0, 0, 256, false>, p, 256, sb, p.B, false, st, nl);
}

template <>
int launch_pnqp<Rr>(const PnqpParams<Rr>& p, cudaStream_t st, long long* nl) {
  const bool batch = p.coupling == DMPC_COUPLING_BATCH;
  const size_t sb = (size_t)pnqp_stride<Rr>(p.m) * sizeof(Rr);
  if (p.m > 32) return DMPC_ERR_UNSUPPORTED;
  const int SG = p.m <= 4 ? 4 : (p.m <= 8 ? 8 : (p.m <= 16 ? 16 : 32));
#define PN(SG_)                                                                                      \
  if (SG == SG_) {                                                                                   \
    if (batch) return launch_elems(pnqp_kernel<Rr, 0, SG_, true>, p, SG_, sb, p.B, true, st, nl);    \
    return launch_elems(pnqp_kernel<Rr, 0, SG_, false>, p, SG_, sb, p.B, false, st, nl);             \
  }
  PN(4) PN(8) PN(16) PN(32)
#undef PN
  return DMPC_ERR_UNSUPPORTED;
}

template <>
int launch_active_mask<Rr>(const Rr* u, const Rr* lo, const Rr* hi, unsigned char* out, size_t count, cudaStream_t st,
                           long long* nl) {
  const int tpb = 256;
  return launch(active_mask_kernel<Rr>, (unsigned)((count + tpb - 1) / tpb), tpb, 0, st, nl, u, lo, hi, out, count);
}

template <>
int launch_traj<Rr>(const TrajParams<Rr>& p, cudaStream_t st, long long* nl) {
  if (p.n + p.m > 64) return launch_traj_large<Rr>(p, st, nl);     // traj_kernel keeps [x; u] in registers
  const int tpb = 64;
  return launch(traj_kernel<Rr, 64>, (p.B + tpb - 1) / tpb, tpb, 0, st, nl, p);
}

}  // namespace dmpc
