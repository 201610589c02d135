// Kernel instantiation + shape dispatch for the LQR kernels (lqr_kernels.cuh).
#include <cstdlib>
#include <type_traits>
#include "launch.h"
#include "lqr_tpe_kernel.cuh"

#ifndef DMPC_REAL
#define DMPC_REAL double
#endif

namespace dmpc {

// Compile-time shapes: the BASELINE.json configs + the reference's examples.
//   (3,1) pendulum / Boyd / LQRnet   (2,1) one-variable example   (4,2) c2   (8,4) c3   (32,8) c5
#define DMPC_SHAPES(X) X(2, 1, 4) X(3, 1, 4) X(4, 2, 8) X(8, 4, 16) X(32, 8, 256)

inline ShapeInfo pick_shape_impl(int n, int m) {
#define X(N_, M_, G_) if (n == N_ && m == M_) return ShapeInfo{N_, M_, G_, true};
  DMPC_SHAPES(X)
#undef X
  const int s = n + m;
  int G = s <= 6 ? 8 : (s <= 14 ? 16 : (s <= 24 ? 32 : 256));
  return ShapeInfo{n, m, G, false};
}

template <typename K, typename P>
static int do_launch(K kernel, const P& p, int G, size_t stride_bytes, int B, cudaStream_t st, long long* nl) {
  int tpb = (G <= 32) ? 128 : G;
  int epb = (G <= 32) ? tpb / G : 1;
  while (G <= 32 && (size_t)epb * stride_bytes > (size_t)kMaxSmem && tpb > 32) { tpb /= 2; epb = tpb / G; }
  // small batches: fewer elements per CTA so the grid covers more SMs
  while (G <= 32 && tpb > 32 && (B + epb - 1) / epb < 148 * 2) { tpb /= 2; epb = tpb / G; }
  const size_t smem = (size_t)epb * stride_bytes;
  if (smem > (size_t)kMaxSmem) return DMPC_ERR_UNSUPPORTED;
  if (set_smem(kernel, smem)) return DMPC_ERR_CUDA;
  return launch(kernel, (B + epb - 1) / epb, tpb, smem, st, nl, p);
}

static bool dmma_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("DMPC_DISABLE_DMMA"); v = (e && e[0] == '1') ? 0 : 1; }
  return v == 1;
}

static bool lqr_tpe_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("DMPC_LQR_GROUP"); v = (e && e[0] == '1') ? 0 : 1; }
  return v == 1;
}

// elements per warp of the thread-per-element kernels (lqr_tpe_kernel.cuh).  32 is the measured default.
// DMPC_LQR_TPE_EPW=auto spreads a small batch over thin warps (8 elements per warp up to B = 148 SMs x 4 schedulers x 8,
// 16 up to twice that), which shortens each warp's operand staging (about 30 % of its instruction stream at config 2;
// the recursion itself does not shrink); tests/test_gpu_dispatch_matrix.py checks every setting against the oracle, but it
// has not been timed, so it stays opt-in.  DMPC_LQR_TPE_EPW=8|16|32 forces a value.
static int tpe_elems_per_warp(int B) {
  static int forced = -2;
  if (forced == -2) {
    const char* e = getenv("DMPC_LQR_TPE_EPW");
    forced = !e ? 32 : ((e[0] == 'a') ? -1 : atoi(e));
    if (forced != -1 && forced != 8 && forced != 16 && forced != 32) forced = 32;
  }
  if (forced > 0) return forced;
  return B <= 148 * 4 * 8 ? 8 : (B <= 148 * 4 * 16 ? 16 : 32);
}

// adjoint_out_tpe_kernel has its own switch (DMPC_ADJ_GROUP=1 -> adjoint_out_kernel) on top of DMPC_LQR_GROUP
static bool lqr_tpe_adj_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("DMPC_ADJ_GROUP"); v = (e && e[0] == '1') ? 0 : 1; }
  return v == 1 && lqr_tpe_enabled();
}

#define DMPC_FUSED_SHAPES(X) X(32, 8)

template <typename R>
bool adjoint_fused_available(int n, int m) {
  static int off = -1;
  if (off < 0) { const char* e = getenv("DMPC_ADJ_UNFUSED"); off = (e && e[0] == '1') ? 1 : 0; }
  if (off) return false;
#define X(N_, M_) if (n == N_ && m == M_) return true;
  DMPC_FUSED_SHAPES(X)
#undef X
  return false;
}

// s <= 6: one thread per element, registers only (lqr_tpe_kernel.cuh); `warp_reals` of shared memory per warp
template <typename K, template <typename> class P, typename R>
static int tpe_launch(K kernel, const P<R>& p, int warp_reals, cudaStream_t st, long long* nl) {
  const int tpb = p.B >= 148 * 64 * 2 ? 64 : 32;            // small batches: more, smaller CTAs so the grid covers the SMs
  const int epw = tpe_elems_per_warp(p.B);
  const size_t sm = (size_t)(tpb / 32) * warp_reals * sizeof(R);
  if (set_smem(kernel, sm)) return DMPC_ERR_CUDA;
  return launch(kernel, (p.B + epw * (tpb / 32) - 1) / (epw * (tpb / 32)), tpb, sm, st, nl, p, epw);
}

template <typename R>
int launch_lqr_rollout_32_8(const LqrParams<R>& p, cudaStream_t st, long long* nl) {
  LqrParams<R> q = p;
  q.flags = LQR_DO_ROLLOUT;
  const LqrLayout L = lqr_layout<R>(q.n, q.m, false, true);
  return do_launch(lqr_solve_kernel<R, 32, 8, 32>, q, 32, (size_t)L.stride * sizeof(R), q.B, st, nl);
}

template <typename R>
int launch_lqr_solve(const LqrParams<R>& p, cudaStream_t st, long long* nl) {
  const ShapeInfo si = pick_shape_impl(p.n, p.m);
  // the DMMA kernel moves C, c, F, f, K_t, k_t with 16-byte cp.async / bulk copies and stores the factors with 16-byte
  // stores: every such pointer must be 16-byte aligned (include/diffmpc_b200.h); otherwise the generic kernel (which
  // checks alignment per copy) takes the call
  auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
  const bool aligned = al16(p.C) && al16(p.c) && al16(p.F) && al16(p.f) && al16(p.Ks) && al16(p.ks) && al16(p.fac) && al16(p.Vsave);
  if (p.n == 32 && p.m == 8 && !(p.flags & LQR_MASKED) && p.c && p.c_scale == R(1) && dmma_enabled() && aligned)
    return launch_lqr_solve_dmma<R>(p, st, nl);
  // DMPC_LQR_GROUP=1 keeps the group kernel (A/B)
  if (lqr_tpe_enabled()) {
#define X(N_, M_) if (p.n == N_ && p.m == M_) return tpe_launch(lqr_tpe_kernel<R, N_, M_, 64, 2, 3>, p, tpe_lqr_warp_reals(N_, M_, 2, 3), st, nl);
    X(2, 1) X(3, 1) X(4, 2)
#undef X
  }
  const bool compact = !(p.flags & LQR_DO_FACTOR);
  const LqrLayout L = lqr_layout<R>(p.n, p.m, (p.flags & LQR_SAVE_FAC) != 0, compact);
  const size_t sb = (size_t)L.stride * sizeof(R);
  // one element per CTA does not fit (do_launch's test; s > 24 runs one element per CTA, smaller systems always fit) or
  // m > 32: the host-stepped large-system kernels (lqr_large_launch.cu), masked solves included
  if (p.m > 32 || sb > (size_t)kMaxSmem) return launch_lqr_large_solve<R>(p, st, nl);
#define X(N_, M_, G_) if (si.specialised && p.n == N_ && p.m == M_) return do_launch(lqr_solve_kernel<R, N_, M_, G_>, p, G_, sb, p.B, st, nl);
  DMPC_SHAPES(X)
#undef X
  switch (si.G) {
    case 8: return do_launch(lqr_solve_kernel<R, 0, 0, 8>, p, 8, sb, p.B, st, nl);
    case 16: return do_launch(lqr_solve_kernel<R, 0, 0, 16>, p, 16, sb, p.B, st, nl);
    case 32: return do_launch(lqr_solve_kernel<R, 0, 0, 32>, p, 32, sb, p.B, st, nl);
    default: return do_launch(lqr_solve_kernel<R, 0, 0, 256>, p, 256, sb, p.B, st, nl);
  }
}

template <typename R>
static int launch_lqr_dtau(const DtauParams<R>& p, cudaStream_t st, long long* nl) {
  const ShapeInfo si = pick_shape_impl(p.n, p.m);
  if (lqr_tpe_enabled()) {
#define X(N_, M_) if (p.n == N_ && p.m == M_) return tpe_launch(lqr_dtau_tpe_kernel<R, N_, M_, 64, 3>, p, tpe_dtau_warp_reals(N_, M_, 3), st, nl);
    X(2, 1) X(3, 1) X(4, 2)
#undef X
  }
  const DtauLayout L = dtau_layout<R>(p.n, p.m);
  const size_t sb = (size_t)L.stride * sizeof(R);
#define X(N_, M_, G_) if (si.specialised && p.n == N_ && p.m == M_) return do_launch(lqr_dtau_kernel<R, N_, M_, (G_ > 32 ? 64 : G_)>, p, (G_ > 32 ? 64 : G_), sb, p.B, st, nl);
  DMPC_SHAPES(X)
#undef X
  switch (si.G) {
    case 8: return do_launch(lqr_dtau_kernel<R, 0, 0, 8>, p, 8, sb, p.B, st, nl);
    case 16: return do_launch(lqr_dtau_kernel<R, 0, 0, 16>, p, 16, sb, p.B, st, nl);
    case 32: return do_launch(lqr_dtau_kernel<R, 0, 0, 32>, p, 32, sb, p.B, st, nl);
    default: return do_launch(lqr_dtau_kernel<R, 0, 0, 64>, p, 64, sb, p.B, st, nl);
  }
}

// Two-sweep adjoint: sweep 1 (lqr_dtau_kernel<FUSED>) then adjoint_fused_kernel, one CTA per element each.
// stage as launch_lqr_adjoint's; DMPC_ERR_UNSUPPORTED when the shape has no instantiation
template <typename R>
static int launch_adjoint_fused(const DtauParams<R>& d, const AdjFusedParams<R>& a, int stage, cudaStream_t st, long long* nl) {
#define X(N_, M_)                                                                                                     \
  if (d.n == N_ && d.m == M_) {                                                                                       \
    const DtauLayout L1 = dtau_layout<R>(N_, M_);                                                                     \
    int rc = DMPC_OK;                                                                                                 \
    if (stage != 2) rc = do_launch(lqr_dtau_kernel<R, N_, M_, 64, true>, d, 64, (size_t)L1.stride * sizeof(R), d.B, st, nl); \
    if (rc || stage == 1) return rc;                                                                                  \
    const AdjFusedLayout L2 = adj_fused_layout<R>(N_, M_);                                                            \
    if (a.red) return do_launch(adjoint_fused_kernel<R, N_, M_, 128, true>, a, 128, (size_t)L2.total * sizeof(R), a.B, st, nl); \
    return do_launch(adjoint_fused_kernel<R, N_, M_, 128, false>, a, 128, (size_t)L2.total * sizeof(R), a.B, st, nl); \
  }
  DMPC_FUSED_SHAPES(X)
#undef X
  return DMPC_ERR_UNSUPPORTED;
}

// adjoint_out_kernel / adjoint_out_tpe_kernel
template <typename R>
static int launch_adjoint_out_group(const AdjOutParams<R>& p, cudaStream_t st, long long* nl) {
  const ShapeInfo si = pick_shape_impl(p.n, p.m);
  const bool red = (p.flags & ADJ_REDUCE_TB) != 0;
  if (!red && lqr_tpe_adj_enabled()) {                        // s <= 6, materialised gradients: thread per element
#define X(N_, M_) if (p.n == N_ && p.m == M_) return tpe_launch(adjoint_out_tpe_kernel<R, N_, M_, 64>, p, tpe_adj_warp_reals(N_, M_), st, nl);
    X(2, 1) X(3, 1) X(4, 2)
#undef X
  }
  const AdjLayout L = adj_layout<R>(p.n, p.m, red && !si.specialised);
  const size_t sb = (size_t)L.stride * sizeof(R);
#define X(N_, M_, G_) if (si.specialised && p.n == N_ && p.m == M_) \
    return red ? do_launch(adjoint_out_kernel<R, N_, M_, (G_ > 32 ? 128 : G_), true>, p, (G_ > 32 ? 128 : G_), sb, p.B, st, nl) \
               : do_launch(adjoint_out_kernel<R, N_, M_, (G_ > 32 ? 128 : G_), false>, p, (G_ > 32 ? 128 : G_), sb, p.B, st, nl);
  DMPC_SHAPES(X)
#undef X
#define Y(G_) return red ? do_launch(adjoint_out_kernel<R, 0, 0, G_, true>, p, G_, sb, p.B, st, nl) \
                         : do_launch(adjoint_out_kernel<R, 0, 0, G_, false>, p, G_, sb, p.B, st, nl);
  switch (si.G) {
    case 8: Y(8)
    case 16: Y(16)
    case 32: Y(32)
    default: Y(128)
  }
#undef Y
}

// The last step of the (T,B)-reduced adjoint: the per-element partial records a.red summed into `sums`.
template <typename R>
static int reduce_partials(const AdjOutParams<R>& a, R* sums, cudaStream_t st, long long* nl, const char** failed) {
  if (!a.red) return DMPC_OK;
  *failed = "reduce_partials launch failed";
  const int wpb = 4, rsz = adj_red_elems(a.n, a.m);
  return launch(reduce_partials_kernel<R>, (rsz + wpb - 1) / wpb, wpb * 32, 0, st, nl, (const R*)a.red, a.B, rsz, sums);
}

// The per-element kernels run where one element's layout fits one CTA's shared memory (do_launch's test).  (The
// compile-time shapes' reduced adjoint keeps its sums in registers; all of them fit either way.)
template <typename R>
static bool fits(int stride) { return (size_t)stride * sizeof(R) <= (size_t)kMaxSmem; }

template <typename R>
int launch_lqr_adjoint(const DtauParams<R>& d, const AdjFusedParams<R>& f, const AdjOutParams<R>& a, int stage, R* sums,
                       cudaStream_t st, long long* nl, const char** failed) {
  int rc;
  if ((a.red || a.df) && adjoint_fused_available<R>(a.n, a.m)) {
    *failed = "adjoint_fused launch failed";
    rc = launch_adjoint_fused<R>(d, f, stage, st, nl);
  } else if (!fits<R>(dtau_layout<R>(a.n, a.m).stride) || !fits<R>(adj_layout<R>(a.n, a.m, a.red != nullptr).stride)) {
    // m > 32 alone does not select these: the per-element adjoint kernels have no limit on m
    if (!lqr_large_shape_ok(a.n, a.m)) { *failed = nullptr; return DMPC_ERR_UNSUPPORTED; }
    *failed = "lqr_adjoint large-system launch failed";
    rc = launch_lqr_large_adjoint<R>(a, d.Ks, d.fac, stage, st, nl);
  } else {
    *failed = "lqr_dtau launch failed";
    rc = stage == 2 ? DMPC_OK : launch_lqr_dtau<R>(d, st, nl);
    if (!rc && stage != 1) {
      *failed = "adjoint_out launch failed";
      rc = launch_adjoint_out_group<R>(a, st, nl);
    }
  }
  if (rc || stage == 1) return rc;
  return reduce_partials<R>(a, sums, st, nl, failed);
}

template <typename R>
int launch_adjoint_out(const AdjOutParams<R>& p, R* sums, cudaStream_t st, long long* nl, const char** failed) {
  int rc;
  if (fits<R>(adj_layout<R>(p.n, p.m, p.red != nullptr).stride)) {
    *failed = "adjoint_out launch failed";
    rc = launch_adjoint_out_group<R>(p, st, nl);
  } else {
    *failed = "mpc_step_backward large-system adjoint launch failed";
    rc = launch_lqr_large_adjoint<R>(p, nullptr, nullptr, 2, st, nl);
  }
  if (rc) return rc;
  return reduce_partials<R>(p, sums, st, nl, failed);
}

template <typename R>
int launch_expand_time_batch(const R* src, R* dst, int count, size_t total, cudaStream_t st, long long* nl) {
  const int tpb = 256;
  size_t blocks = (total + tpb - 1) / tpb;
  if (blocks > 148 * 32) blocks = 148 * 32;               // grid-stride: 32 CTAs per SM keep the store queues full
  return launch(expand_time_batch_kernel<R>, (unsigned)blocks, tpb, 0, st, nl, src, dst, count, total);
}

template bool adjoint_fused_available<DMPC_REAL>(int, int);
template int launch_expand_time_batch<DMPC_REAL>(const DMPC_REAL*, DMPC_REAL*, int, size_t, cudaStream_t, long long*);
template int launch_lqr_rollout_32_8<DMPC_REAL>(const LqrParams<DMPC_REAL>&, cudaStream_t, long long*);
template int launch_lqr_solve<DMPC_REAL>(const LqrParams<DMPC_REAL>&, cudaStream_t, long long*);
template int launch_lqr_adjoint<DMPC_REAL>(const DtauParams<DMPC_REAL>&, const AdjFusedParams<DMPC_REAL>&,
                                           const AdjOutParams<DMPC_REAL>&, int, DMPC_REAL*, cudaStream_t, long long*, const char**);
template int launch_adjoint_out<DMPC_REAL>(const AdjOutParams<DMPC_REAL>&, DMPC_REAL*, cudaStream_t, long long*, const char**);

}  // namespace dmpc
