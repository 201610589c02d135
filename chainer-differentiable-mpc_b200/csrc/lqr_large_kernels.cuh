// LQR kernels for systems whose per-element step does not fit one CTA's shared memory (DESIGN.md §4.8).
//
// The other LQR kernels keep one element's C_t, F_t, Q_t, V_t in the shared memory of one CTA for the whole horizon.
// Here the horizon is stepped from the host and every step is spread over many CTAs:
//
//   lqr_large_q_kernel       grid (B, column panels): W = V_{t+1} [F_t | f_t] + [0 | v_{t+1}],  [Q | q] = [C | c] + F_t^T W
//   lqr_large_factor_kernel  grid B: pivoted LU of Quu, [K | k], Quu^-1 | Qxu (factor cache), P = [Qux | qu] + Quu [K | k]
//   lqr_large_v_kernel       grid (B, column panels): [V | v] = [Qxx | qx] + Qxu [K | k] + K^T P
//   lqr_large_rollout_kernel grid B: u_t = K_t x_t + k_t, x_{t+1} = F_t [x_t; u_t] + f_t
//   lqr_large_adj_kernel     grid B: the d-tau sweeps of lqr_dtau_kernel and the lambda / d-lambda recursion of
//                            adjoint_out_kernel, matrix-vector products read from L2 / HBM
//   lqr_large_outer_kernel   grid (B, T): dC_t, dF_t, df_t written per (t, b)
//   lqr_large_red_kernel     grid (B, column panels): per-element sums over t of the same outer products, as
//                            contractions over t, into the partial-record layout of reduce_partials_kernel
//
// Every product runs in fp64 on mma.m8n8k4.f64 (DMMA); fp32 tensors are widened on load and rounded once on store.
// Scratch (V | v, Q | q, [K | k], P, lambda, d-lambda) is fp64 and per element.
#pragma once
#include "launch.h"
#include "lqr_kernels.cuh"
#include "lqr_shared_kernels.cuh"

namespace dmpc {

constexpr int kLargeThreads = 256;   // 8 warps
constexpr int kLargePanel = 32;      // output columns per CTA of the tile-parallel stages
constexpr int kLargeMaxM = 32;        // register copy of the pivot column in g_lu_factor

// fp64 scratch of the forward, per element: V | v [n][n+1], Q | q [s][s+1], [K | k] [m][n+1], P [m][n+1]
struct LargeFwdWs { double* V; double* Q; double* KK; double* P; };
// fp64 scratch of the adjoint: lambda_t, d-lambda_t [T][B][n]
struct LargeAdjWs { double* lam; double* dlam; };

// out(i,j) = base(i,j) + sum_{k<K} A(i,k) Bm(k,j) for i < I, j < J on 8x8 tiles spread over the CTA's warps.
// Fragments of mma.m8n8k4.f64: lane (g, q) holds A(g, q), B(q, g), D(g, 2q..2q+1).  Out-of-range rows, columns and k
// read as zero, so ragged edges need no padding.
template <class FA, class FB, class FC, class FO>
__device__ __forceinline__ void large_gemm(int I, int J, int K, FA A, FB Bm, FC base, FO out) {
  const int warp = threadIdx.x >> 5, nw = blockDim.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
  const int ti = (I + 7) >> 3, tj = (J + 7) >> 3;
  for (int tile = warp; tile < ti * tj; tile += nw) {
    const int i = (tile / tj) * 8 + g, j0 = (tile % tj) * 8, ja = j0 + 2 * q, jb = ja + 1, jB = j0 + g;
    double acc[2];
    acc[0] = (i < I && ja < J) ? base(i, ja) : 0.0;
    acc[1] = (i < I && jb < J) ? base(i, jb) : 0.0;
    for (int k0 = 0; k0 < K; k0 += 4) {
      const int k = k0 + q;
      const double a = (i < I && k < K) ? A(i, k) : 0.0;
      const double b = (k < K && jB < J) ? Bm(k, jB) : 0.0;
      dmma_f64(acc, a, b);
    }
    if (i < I && ja < J) out(i, ja, acc[0]);
    if (i < I && jb < J) out(i, jb, acc[1]);
  }
}

// y_i = init(i) + sum_{k<K} A(i,k) x_k for i < I: one warp per row (coalesced along a row of A), fixed-order lane
// partial sums and shuffle tree, so the result does not depend on the launch.  Callers synchronise afterwards.
template <class FA, class FI, class FO>
__device__ __forceinline__ void cta_rowdot(int I, int K, FA A, const double* x, FI init, FO out) {
  const int warp = threadIdx.x >> 5, nw = blockDim.x >> 5, lane = threadIdx.x & 31;
  for (int i = warp; i < I; i += nw) {
    double a = 0.0;
    for (int k = lane; k < K; k += 32) a += A(i, k) * x[k];
    for (int d = 16; d > 0; d >>= 1) a += __shfl_xor_sync(0xffffffffu, a, d);
    if (lane == 0) out(i, init(i) + a);
  }
}

// y_i = init(i) + sum_{k<K} A(k,i) x_k for i < I: one thread per output (coalesced along a row of A across threads)
template <class FA, class FI, class FO>
__device__ __forceinline__ void cta_coldot(int I, int K, FA A, const double* x, FI init, FO out) {
  for (int i = threadIdx.x; i < I; i += blockDim.x) {
    double a0 = init(i), a1 = 0.0;
    int k = 0;
    for (; k + 1 < K; k += 2) { a0 += A(k, i) * x[k]; a1 += A(k + 1, i) * x[k + 1]; }
    if (k < K) a0 += A(k, i) * x[k];
    out(i, a0 + a1);
  }
}

// ---------------------------------------------------------------------------------------------- forward
// Q step of time t.  Column j < s of [Q | q] is column j of Q, column s is q.
// c is p.c, or the split form p.cx | p.cu (NULL parts are zero), times p.c_scale.
template <typename R>
__global__ void __launch_bounds__(kLargeThreads) lqr_large_q_kernel(LqrParams<R> p, LargeFwdWs w, int t) {
  extern __shared__ double Wp[];                        // [n][kLargePanel]: W(:, panel)
  if (p.skip && *p.skip) return;
  const int n = p.n, m = p.m, s = n + m, e = blockIdx.x, j0 = blockIdx.y * kLargePanel;
  const int J = min(kLargePanel, s + 1 - j0);
  const size_t idx = (size_t)t * p.B + e;
  const R* Ct = p.C + idx * s * s;
  const double cs = (double)p.c_scale;
  auto cval = [&](int i) -> double {
    if (p.c) return cs * (double)p.c[idx * s + i];
    const R* part = i < n ? p.cx : p.cu;
    return part ? cs * (double)(i < n ? part[idx * n + i] : part[idx * m + i - n]) : 0.0;
  };
  double* Q = w.Q + (size_t)e * s * (s + 1);
  auto base = [&](int i, int j) -> double { return j0 + j < s ? (double)Ct[i * s + j0 + j] : cval(i); };
  auto out = [&](int i, int j, double v) { Q[i * (s + 1) + j0 + j] = v; };
  if (t == p.T - 1) {
    auto zero = [](int, int) -> double { return 0.0; };
    large_gemm(s, J, 0, zero, zero, base, out);
    return;
  }
  const R* Ft = p.F + idx * n * s;
  const R* ft = p.f ? p.f + idx * n : nullptr;
  const double* V = w.V + (size_t)e * n * (n + 1);
  large_gemm(n, J, n,
             [&](int i, int k) -> double { return V[i * (n + 1) + k]; },
             [&](int k, int j) -> double { const int jj = j0 + j; return jj < s ? (double)Ft[k * s + jj] : (ft ? (double)ft[k] : 0.0); },
             [&](int i, int j) -> double { return j0 + j == s ? V[i * (n + 1) + n] : 0.0; },
             [&](int i, int j, double v) { Wp[i * kLargePanel + j] = v; });
  __syncthreads();
  large_gemm(s, J, n,
             [&](int i, int k) -> double { return (double)Ft[k * s + i]; },
             [&](int k, int j) -> double { return Wp[k * kLargePanel + j]; },
             base, out);
}

// Factor step of time t: one CTA per element, pivoted LU of Quu (m <= 32) carrying -[Qux | qu | I] (no symmetric
// shortcut: C need not be symmetric).  Writes K_t, k_t, the factor cache, [K | k] and P for the V step.
template <typename R>
__global__ void __launch_bounds__(kLargeThreads) lqr_large_factor_kernel(LqrParams<R> p, LargeFwdWs w, int t) {
  extern __shared__ double fsm[];
  const int n = p.n, m = p.m, s = n + m, e = blockIdx.x, ldr = n + 1 + m, ldq = s + 1;
  double* H = fsm;
  double* Rhs = fsm + m * m;
  const double* Q = w.Q + (size_t)e * s * ldq;
  const size_t idx = (size_t)t * p.B + e;
  // LQR_MASKED (LQR_active, active_constrained_lqr.py:113-126): cross terms of active controls zeroed with 1e-8 on their
  // diagonal, their rows of Qux and qu zeroed; P below keeps the unmasked Quu, Qux, qu
  const unsigned char* act = (p.flags & LQR_MASKED) ? p.active + idx * m : nullptr;
  for (int o = threadIdx.x; o < m * m; o += blockDim.x) {
    const int i = o / m, j = o - i * m;
    double hv = Q[(n + i) * ldq + n + j];
    if (act && (act[i] || act[j])) hv = i == j && act[i] ? 1e-8 : 0.0;
    H[o] = hv;
  }
  for (int o = threadIdx.x; o < m * ldr; o += blockDim.x) {
    const int i = o / ldr, j = o - i * ldr;
    double rv = j < n ? -Q[(n + i) * ldq + j] : (j == n ? -Q[(n + i) * ldq + s] : (j - n - 1 == i ? 1.0 : 0.0));
    if (act && j <= n && act[i]) rv = 0.0;
    Rhs[o] = rv;
  }
  __syncthreads();
  const Grp<kLargeThreads> g;
  g_lu_factor<kLargeThreads, kLargeMaxM>(g, m, H, m, Rhs, ldr, ldr, (int*)nullptr);
  g_back_subst(g, m, H, m, Rhs, ldr, ldr);
  __syncthreads();
  double* KK = w.KK + (size_t)e * m * (n + 1);
  double* P = w.P + (size_t)e * m * (n + 1);
  for (int o = threadIdx.x; o < m * (n + 1); o += blockDim.x) {
    const int i = o / (n + 1), j = o - i * (n + 1);
    const double kv = Rhs[i * ldr + j];
    double a = j < n ? Q[(n + i) * ldq + j] : Q[(n + i) * ldq + s];
    for (int l = 0; l < m; ++l) a += Q[(n + i) * ldq + n + l] * Rhs[l * ldr + j];
    KK[o] = kv;
    P[o] = a;
    if (j < n) p.Ks[idx * m * n + i * n + j] = (R)kv; else p.ks[idx * m + i] = (R)kv;
  }
  if ((p.flags & LQR_SAVE_FAC) && p.fac) {
    R* fg = p.fac + idx * (m * m + n * m);
    for (int o = threadIdx.x; o < m * m; o += blockDim.x) { const int i = o / m, j = o - i * m; fg[o] = (R)Rhs[i * ldr + n + 1 + j]; }
    for (int o = threadIdx.x; o < n * m; o += blockDim.x) { const int i = o / m, j = o - i * m; fg[m * m + o] = (R)Q[i * ldq + n + j]; }
  }
}

// V step of time t (t >= 1): [V | v] = [Qxx | qx] + Qxu [K | k] + K^T P as one contraction of length 2m.
// Vdst (nullable): V_t | v_t per (t, b) in the factor-cache layout.
template <typename R>
__global__ void __launch_bounds__(kLargeThreads) lqr_large_v_kernel(LqrParams<R> p, LargeFwdWs w, R* Vdst, int t) {
  if (p.skip && *p.skip) return;
  const int n = p.n, m = p.m, s = n + m, e = blockIdx.x, j0 = blockIdx.y * kLargePanel, ldq = s + 1;
  const int J = min(kLargePanel, n + 1 - j0);
  const double* Q = w.Q + (size_t)e * s * ldq;
  const double* KK = w.KK + (size_t)e * m * (n + 1);
  const double* P = w.P + (size_t)e * m * (n + 1);
  double* V = w.V + (size_t)e * n * (n + 1);
  R* vd = Vdst ? Vdst + ((size_t)t * p.B + e) * (n * n + n) : nullptr;
  large_gemm(n, J, 2 * m,
             [&](int i, int k) -> double { return k < m ? Q[i * ldq + n + k] : KK[(k - m) * (n + 1) + i]; },
             [&](int k, int j) -> double { return k < m ? KK[k * (n + 1) + j0 + j] : P[(k - m) * (n + 1) + j0 + j]; },
             [&](int i, int j) -> double { return j0 + j < n ? Q[i * ldq + j0 + j] : Q[i * ldq + s]; },
             [&](int i, int j, double v) {
               const int jj = j0 + j;
               V[i * (n + 1) + jj] = v;
               if (vd) vd[jj < n ? i * n + jj : n * n + i] = (R)v;
             });
}

// Rollout: one CTA per element over the horizon.  LQR_MASKED: u of active controls is zero
// (active_constrained_lqr.py:175); tau_out (nullable) gets [x; u].
template <typename R>
__global__ void __launch_bounds__(kLargeThreads) lqr_large_rollout_kernel(LqrParams<R> p) {
  extern __shared__ double rsm[];
  const int n = p.n, m = p.m, s = n + m, e = blockIdx.x, T = p.T;
  double* xu = rsm;           // [x; u]
  double* xn = rsm + s;       // next x
  for (int o = threadIdx.x; o < n; o += blockDim.x) xu[o] = (double)p.x0[(size_t)e * n + o];
  __syncthreads();
  for (int t = 0; t < T; ++t) {
    const size_t idx = (size_t)t * p.B + e;
    const R* Kt = p.Ks + idx * m * n;
    const R* kt = p.ks + idx * m;
    const unsigned char* act = (p.flags & LQR_MASKED) ? p.active + idx * m : nullptr;
    cta_rowdot(m, n, [&](int i, int k) -> double { return (double)Kt[i * n + k]; }, xu,
               [&](int i) -> double { return (double)kt[i]; },
               [&](int i, double v) { xu[n + i] = act && act[i] ? 0.0 : v; });
    __syncthreads();
    if (p.x) for (int o = threadIdx.x; o < n; o += blockDim.x) p.x[idx * n + o] = (R)xu[o];
    if (p.u) for (int o = threadIdx.x; o < m; o += blockDim.x) p.u[idx * m + o] = (R)xu[n + o];
    if (p.tau_out) for (int o = threadIdx.x; o < s; o += blockDim.x) p.tau_out[idx * s + o] = (R)xu[o];
    if (t < T - 1) {
      const R* Ft = p.F + idx * n * s;
      const R* ft = p.f ? p.f + idx * n : nullptr;
      cta_rowdot(n, s, [&](int i, int k) -> double { return (double)Ft[i * s + k]; }, xu,
                 [&](int i) -> double { return ft ? (double)ft[i] : 0.0; }, [&](int i, double v) { xn[i] = v; });
      __syncthreads();
      for (int o = threadIdx.x; o < n; o += blockDim.x) xu[o] = xn[o];
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------- adjoint
// One CTA per element; the same three recursions as lqr_dtau_kernel + adjoint_out_kernel (the MPC step backward runs
// sweep 3 only, on the masked solve's dtau, with ADJ_NEGATE / ADJ_NEG_RHS as in adjoint_out_kernel):
//   sweep 1 (t down): q = [gx | gu] + F_t^T v';  k' = -Quu^-1 q_u;  v' = q_x + Qxu k'      (k' parked in dtau[t, n:])
//   sweep 2 (t up):   du = K_t dx + k';  dtau_t = [dx; du];  dx' = F_t dtau_t
//   sweep 3 (t down): lambda_t = c_t[:n] + C_t[:n,:] tau_t + F_t[:, :n]^T lambda_{t+1}, d-lambda the same on dtau and gx
// lambda_t, d-lambda_t go to scratch for the outer-product stage; dx0 = d-lambda_0.
template <typename R>
__global__ void __launch_bounds__(kLargeThreads) lqr_large_adj_kernel(AdjOutParams<R> a, const R* Ks, const R* fac,
                                                                       LargeAdjWs w, int do_dtau, int do_lam) {
  extern __shared__ double asm_[];
  const int n = a.n, m = a.m, s = n + m, e = blockIdx.x, T = a.T, B = a.B, fsz = m * m + n * m;
  double* q = asm_;              // [s]
  double* vp = q + s;            // [n]  v' / lambda
  double* kp = vp + n;           // [m]
  double* dx = kp + m;           // [s]  dtau_t / tau_t
  double* tmp = dx + s;          // [n]
  double* dl = tmp + n;          // [n]  d-lambda
  double* tmp2 = dl + n;         // [n]
  double* dt = tmp2 + n;         // [s]
  R* dtau = const_cast<R*>(a.dtau);
  if (do_dtau) {
    for (int t = T - 1; t >= 0; --t) {
      const size_t idx = (size_t)t * B + e;
      const R* Ft = a.F + idx * n * s;
      const int Kf = t < T - 1 ? n : 0;
      cta_coldot(s, Kf, [&](int k, int i) -> double { return (double)Ft[k * s + i]; }, vp,
                 [&](int i) -> double { return i < n ? (a.gx ? (double)a.gx[idx * n + i] : 0.0) : (a.gu ? (double)a.gu[idx * m + i - n] : 0.0); },
                 [&](int i, double v) { q[i] = v; });
      __syncthreads();
      const R* Qi = fac + idx * fsz;
      cta_rowdot(m, m, [&](int i, int k) -> double { return (double)Qi[i * m + k]; }, q + n,
                 [](int) -> double { return 0.0; }, [&](int i, double v) { kp[i] = -v; dtau[idx * s + n + i] = (R)(-v); });
      __syncthreads();
      const R* Qxu = Qi + m * m;
      cta_rowdot(n, m, [&](int i, int k) -> double { return (double)Qxu[i * m + k]; }, kp,
                 [&](int i) -> double { return q[i]; }, [&](int i, double v) { vp[i] = v; });
      __syncthreads();
    }
    for (int o = threadIdx.x; o < n; o += blockDim.x) dx[o] = 0.0;
    __syncthreads();
    for (int t = 0; t < T; ++t) {
      const size_t idx = (size_t)t * B + e;
      const R* Kt = Ks + idx * m * n;
      cta_rowdot(m, n, [&](int i, int k) -> double { return (double)Kt[i * n + k]; }, dx,
                 [&](int i) -> double { return (double)dtau[idx * s + n + i]; }, [&](int i, double v) { kp[i] = v; });
      __syncthreads();
      for (int o = threadIdx.x; o < m; o += blockDim.x) dx[n + o] = kp[o];
      __syncthreads();
      for (int o = threadIdx.x; o < s; o += blockDim.x) dtau[idx * s + o] = (R)dx[o];
      if (t < T - 1) {
        const R* Ft = a.F + idx * n * s;
        cta_rowdot(n, s, [&](int i, int k) -> double { return (double)Ft[i * s + k]; }, dx,
                   [](int) -> double { return 0.0; }, [&](int i, double v) { tmp[i] = v; });
        __syncthreads();
        for (int o = threadIdx.x; o < n; o += blockDim.x) dx[o] = tmp[o];
      }
      __syncthreads();
    }
  }
  if (!do_lam) return;
  for (int t = T - 1; t >= 0; --t) {
    const size_t idx = (size_t)t * B + e;
    for (int o = threadIdx.x; o < s; o += blockDim.x) {
      dx[o] = o < n ? (double)a.x[idx * n + o] : (double)a.u[idx * m + o - n];
      dt[o] = (double)a.dtau[idx * s + o];
    }
    __syncthreads();
    const R* Ct = a.C + idx * s * s;
    const R* ct = a.c + idx * s;
    cta_rowdot(n, s, [&](int i, int k) -> double { return (double)Ct[i * s + k]; }, dx,
               [&](int i) -> double { return (double)ct[i]; }, [&](int i, double v) { tmp[i] = v; });
    cta_rowdot(n, s, [&](int i, int k) -> double { return (double)Ct[i * s + k]; }, dt,
               [&](int i) -> double {
                 const double gv = a.gx ? (double)a.gx[idx * n + i] : 0.0;
                 return (a.flags & ADJ_NEG_RHS) ? -gv : gv;
               }, [&](int i, double v) { tmp2[i] = v; });
    __syncthreads();
    const R* Ft = a.F + idx * n * s;
    const int Kf = t < T - 1 ? n : 0;
    // lambda_{t+1} sits in vp, d-lambda_{t+1} in dl; the new values go to q and dt (free after the barrier above)
    // and replace them after the next one
    cta_coldot(n, Kf, [&](int k, int i) -> double { return (double)Ft[k * s + i]; }, vp,
               [&](int i) -> double { return tmp[i]; }, [&](int i, double v) { q[i] = v; });
    cta_coldot(n, Kf, [&](int k, int i) -> double { return (double)Ft[k * s + i]; }, dl,
               [&](int i) -> double { return tmp2[i]; }, [&](int i, double v) { dt[i] = v; });
    __syncthreads();
    for (int o = threadIdx.x; o < n; o += blockDim.x) {
      vp[o] = q[o];
      dl[o] = dt[o];
      w.lam[idx * n + o] = q[o];
      w.dlam[idx * n + o] = dt[o];
      if (t == 0) a.dx0[(size_t)e * n + o] = (R)((a.flags & ADJ_NEGATE) ? -dt[o] : dt[o]);
    }
    __syncthreads();
  }
}

// dC_t, dF_t (t < T-1), df_t (t < T-1, nullable) per (t, b).  dc_t is dtau_t: the LQR adjoint's dtau is the caller's dc
// buffer; ADJ_NEGATE (MPC step) writes dc = -dtau and negates every gradient, and F with T rows (F_T == T) gets a zero
// row T-1 of dF (mpc_step.py:428).
template <typename R>
__global__ void __launch_bounds__(kLargeThreads) lqr_large_outer_kernel(AdjOutParams<R> a, LargeAdjWs w) {
  const int n = a.n, m = a.m, s = n + m, e = blockIdx.x, t = blockIdx.y, T = a.T, B = a.B;
  const size_t idx = (size_t)t * B + e;
  const bool quirk_c = (a.flags & ADJ_QUIRK_DC) != 0, quirk_f = (a.flags & ADJ_QUIRK_DF) != 0;
  const double sgn = (a.flags & ADJ_NEGATE) ? -1.0 : 1.0;
  auto tau = [&](int j) -> double { return j < n ? (double)a.x[idx * n + j] : (double)a.u[idx * m + j - n]; };
  const R* dt = a.dtau + idx * s;
  R* dC = a.dC + idx * s * s;
  for (int o = threadIdx.x; o < s * s; o += blockDim.x) {
    const int i = o / s, j = o - i * s;
    const double x = (double)dt[i] * tau(j), y = tau(i) * (double)dt[j];
    dC[o] = (R)(quirk_c ? 0.5 * x + y : sgn * (0.5 * (x + y)));
  }
  if (a.dc != a.dtau) for (int o = threadIdx.x; o < s; o += blockDim.x) a.dc[idx * s + o] = (R)(sgn * (double)dt[o]);
  if (t >= T - 1) {
    if (a.F_T == T && a.dF) for (int o = threadIdx.x; o < n * s; o += blockDim.x) a.dF[idx * n * s + o] = R(0);
    return;
  }
  const double* ln = w.lam + (idx + B) * n;
  const double* dln = w.dlam + (idx + B) * n;
  R* dF = a.dF + idx * n * s;
  for (int o = threadIdx.x; o < n * s; o += blockDim.x) {
    const int i = o / s, j = o - i * s;
    dF[o] = (R)(sgn * (dln[i] * tau(j) + ln[i] * (double)dt[j]));
  }
  if (a.df) {
    const double* src = quirk_f ? w.dlam + idx * n : dln;
    for (int o = threadIdx.x; o < n; o += blockDim.x) a.df[idx * n + o] = (R)(sgn * src[o]);
  }
}

// Per-element sums over t into a.red[e] = (sum dC [s,s] | sum dc [s] | sum dF [n,s] | sum df [n]): contractions over
// t of length 2T (dC) and 2(T-1) (dF) on DMMA, column panels of [dC; dF] over the CTAs.
template <typename R>
__global__ void __launch_bounds__(kLargeThreads) lqr_large_red_kernel(AdjOutParams<R> a, LargeAdjWs w) {
  const int n = a.n, m = a.m, s = n + m, e = blockIdx.x, j0 = blockIdx.y * kLargePanel, T = a.T, B = a.B;
  const int J = min(kLargePanel, s - j0);
  const bool quirk_c = (a.flags & ADJ_QUIRK_DC) != 0, quirk_f = (a.flags & ADJ_QUIRK_DF) != 0;
  const double sgn = (a.flags & ADJ_NEGATE) ? -1.0 : 1.0;    // ADJ_NEGATE never comes with the quirks
  const double c1 = sgn * 0.5, c2 = quirk_c ? 1.0 : sgn * 0.5;
  auto tau = [&](int t, int j) -> double {
    const size_t idx = (size_t)t * B + e;
    return j < n ? (double)a.x[idx * n + j] : (double)a.u[idx * m + j - n];
  };
  auto dt = [&](int t, int j) -> double { return (double)a.dtau[((size_t)t * B + e) * s + j]; };
  auto lam = [&](int t, int i) -> double { return w.lam[((size_t)t * B + e) * n + i]; };
  auto dlam = [&](int t, int i) -> double { return w.dlam[((size_t)t * B + e) * n + i]; };
  R* out = a.red + (size_t)e * adj_red_elems(n, m);
  auto zero = [](int, int) -> double { return 0.0; };
  // sum_t (c1 dtau_t tau_t^T + c2 tau_t dtau_t^T)
  large_gemm(s, J, 2 * T,
             [&](int i, int k) -> double { return k < T ? dt(k, i) : tau(k - T, i); },
             [&](int k, int j) -> double { return k < T ? c1 * tau(k, j0 + j) : c2 * dt(k - T, j0 + j); },
             zero, [&](int i, int j, double v) { out[i * s + j0 + j] = (R)v; });
  // sum_{t<T-1} (d-lambda_{t+1} tau_t^T + lambda_{t+1} dtau_t^T)
  const int T1 = T - 1;
  large_gemm(n, J, 2 * T1,
             [&](int i, int k) -> double { return k < T1 ? dlam(k + 1, i) : lam(k - T1 + 1, i); },
             [&](int k, int j) -> double { return k < T1 ? tau(k, j0 + j) : dt(k - T1, j0 + j); },
             zero, [&](int i, int j, double v) { out[s * s + s + i * s + j0 + j] = (R)(sgn * v); });
  if (blockIdx.y != 0) return;
  for (int o = threadIdx.x; o < s + n; o += blockDim.x) {
    double acc = 0.0;
    if (o < s) {
      for (int t = 0; t < T; ++t) acc += dt(t, o);
      out[s * s + o] = (R)(sgn * acc);
    } else {
      const int i = o - s;
      for (int t = 0; t < T1; ++t) acc += quirk_f ? dlam(t, i) : dlam(t + 1, i);
      out[s * s + s + n * s + i] = (R)(sgn * acc);
    }
  }
}

// ---- host: the Riccati steps of the large-system LQR solve and MPC step forward

inline size_t large_fwd_ws_bytes(int B, int n, int m) {
  const size_t s = (size_t)(n + m);
  return sizeof(double) * B * ((size_t)n * (n + 1) + s * (s + 1) + 2 * (size_t)m * (n + 1));
}

// Per t = T-1 ... 0: lqr_large_q_kernel, then factor(w, t) (the factor step, which launches one kernel), then for t >= 1
// lqr_large_v_kernel, which also writes V_t | v_t to Vdst when it is not null.  `ws` holds large_fwd_ws_bytes.
// factor's kernel has its shared-memory limit set by the caller.
template <typename R, typename Factor>
int large_riccati_steps(const LqrParams<R>& q, double* ws, R* Vdst, Factor factor, cudaStream_t st, long long* nl) {
  const int n = q.n, s = n + q.m, B = q.B;
  const size_t nV = (size_t)n * (n + 1), nQ = (size_t)s * (s + 1), nK = (size_t)q.m * (n + 1);
  const LargeFwdWs w{ws, ws + (size_t)B * nV, ws + (size_t)B * (nV + nQ), ws + (size_t)B * (nV + nQ + nK)};
  const size_t smq = sizeof(double) * n * kLargePanel;
  int rc = set_smem(lqr_large_q_kernel<R>, smq);
  const dim3 gq(B, (s + 1 + kLargePanel - 1) / kLargePanel), gv(B, (n + 1 + kLargePanel - 1) / kLargePanel);
  for (int t = q.T - 1; t >= 0 && !rc; --t) {
    rc = launch(lqr_large_q_kernel<R>, gq, kLargeThreads, smq, st, nl, q, w, t);
    if (!rc) rc = factor(w, t);
    if (!rc && t > 0) rc = launch(lqr_large_v_kernel<R>, gv, kLargeThreads, 0, st, nl, q, w, Vdst, t);
  }
  return rc;
}

}  // namespace dmpc
