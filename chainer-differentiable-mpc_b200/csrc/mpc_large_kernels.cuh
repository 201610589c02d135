// MPC step forward and get_traj for systems whose per-element step does not fit one CTA's shared memory
// (DESIGN.md §4.9).  The horizon is stepped from the host, as for the large LQR solve (lqr_large_kernels.cuh):
//
//   mpc_large_chat_kernel   grid (B, T): Taylor shift c_hat_t = C_t tau_nom,t + c_t (mpc_step.py:305-316) into an
//                           R-typed [T,B,s] scratch, read by lqr_large_q_kernel as its c
//   per t = T-1 ... 0:  lqr_large_q_kernel, mpc_large_pnqp_kernel, lqr_large_v_kernel (t >= 1)
//   mpc_large_pnqp_kernel   grid B: PNQP on (Quu, qu, lo - u_nom, hi - u_nom) warm-started from k_{t+1} (one warp),
//                           K = -(LU)^-1 Qux with the rows of clamped controls zeroed, P = [Qux | qu] + Quu [K | k]
//   mpc_large_ls_kernel     grid B: forward_rec (mpc_step.py:175-286), every line-search pass over the whole horizon
//   traj_large_kernel       grid B: util.get_traj for LinDx with the line search's row-dot order
//
// Every product runs in fp64; fp32 tensors are widened on load and rounded once on store.  The line search and the
// rollout round the state and the controls to R as they produce them, so get_traj of the accepted controls reproduces
// the accepted trajectory bit for bit in both dtypes.
#pragma once
#include "lqr_large_kernels.cuh"
#include "mpc_kernels.cuh"

namespace dmpc {

template <typename R>
__global__ void __launch_bounds__(kLargeThreads) mpc_large_chat_kernel(MpcFwdParams<R> p, R* chat) {
  extern __shared__ double csm[];                       // tau_nom [s]
  if (p.skip && *p.skip) return;
  const int n = p.n, m = p.m, s = n + m, e = blockIdx.x, t = blockIdx.y;
  const size_t idx = (size_t)t * p.B + e;
  for (int o = threadIdx.x; o < s; o += blockDim.x) csm[o] = o < n ? (double)p.x_nom[idx * n + o] : (double)p.u_nom[idx * m + o - n];
  __syncthreads();
  const R* Ct = p.C + idx * s * s;
  const R* ct = p.c + idx * s;
  cta_rowdot(s, s, [&](int i, int k) -> double { return (double)Ct[i * s + k]; }, csm,
             [&](int i) -> double { return (double)ct[i]; }, [&](int i, double v) { chat[idx * s + i] = (R)v; });
}

// shared memory of mpc_large_pnqp_kernel, in doubles
__host__ __device__ inline int mpc_large_pnqp_smem(int n, int m) { return 2 * m * m + m * (n + 1) + 8 * m; }

// PNQP factor step of time t (mpc_step.py:136-157).  Reads [Q | q] of the Q step and k_{t+1} from [K | k] (the warm
// start, :141-146; at t = T-1 the clamped unconstrained solve), writes K_t, k_t, n_qp, free and [K | k], P for the V step.
// Per-element flags accumulate into eflags over the steps.
template <typename R>
__global__ void __launch_bounds__(kLargeThreads) mpc_large_pnqp_kernel(MpcFwdParams<R> p, LargeFwdWs w, int* eflags, int t) {
  extern __shared__ double psm[];
  __shared__ unsigned sh_fm;
  __shared__ int sh_it, sh_status;
  if (p.skip && *p.skip) return;
  const int n = p.n, m = p.m, s = n + m, e = blockIdx.x, ldq = s + 1, ldr = n + 1, T = p.T;
  const size_t idx = (size_t)t * p.B + e;
  double* Huu = psm;
  double* Hf = Huu + m * m;
  double* Rhs = Hf + m * m;
  double* qu = Rhs + m * ldr;
  double* lb = qu + m;
  double* ub = lb + m;
  double* kp = ub + m;
  double* rhs1 = kp + m;
  double* gb = rhs1 + m;
  double* xh = gb + m;
  int* piv = reinterpret_cast<int*>(xh + m);
  const double* Q = w.Q + (size_t)e * s * ldq;
  double* KK = w.KK + (size_t)e * m * ldr;
  double* P = w.P + (size_t)e * m * ldr;
  for (int o = threadIdx.x; o < m * m; o += blockDim.x) { const int i = o / m, j = o - i * m; Huu[o] = Q[(n + i) * ldq + n + j]; }
  for (int o = threadIdx.x; o < m; o += blockDim.x) {
    const double un = (double)p.u_nom[idx * m + o];
    qu[o] = Q[(n + o) * ldq + s];
    lb[o] = (double)p.lo[idx * m + o] - un;                                      // :136-138
    ub[o] = (double)p.hi[idx * m + o] - un;
    kp[o] = t < T - 1 ? KK[o * ldr + n] : 0.0;
  }
  __syncthreads();
  if (threadIdx.x < 32) {
    const Grp<32> sg;
    if (t == T - 1) {
      for (int o = sg.lane; o < m * m; o += 32) Hf[o] = Huu[o];
      for (int o = sg.lane; o < m; o += 32) rhs1[o] = -qu[o];
      sg.sync();
      g_lu_factor<32, kLargeMaxM>(sg, m, Hf, m, rhs1, 1, 1, (int*)nullptr);
      g_back_subst(sg, m, Hf, m, rhs1, 1, 1);
      sg.sync();
      for (int o = sg.lane; o < m; o += 32) kp[o] = fmin(fmax(rhs1[o], lb[o]), ub[o]);
    } else {
      for (int o = sg.lane; o < m; o += 32) kp[o] = fmin(fmax(kp[o], lb[o]), ub[o]);
    }
    sg.sync();
    unsigned fm = 0, bphase = 0;
    int status = 0;
    const int it = g_pnqp<32, kLargeMaxM, false>(sg, m, Huu, m, qu, lb, ub, kp, Hf, piv, rhs1, gb, xh, p.n_qp_iter, &fm,
                                                 &status, bphase);
    for (int o = 0; o < m; ++o) if (p.lo[idx * m + o] > p.hi[idx * m + o]) status |= FLAG_BAD_BOUNDS;   // the reference asserts (:139)
    if (sg.lane == 0) { sh_fm = fm; sh_it = it; sh_status = status; }
  }
  __syncthreads();
  const unsigned fm = sh_fm;
  // K = -(LU)^-1 Qux with the rows of clamped controls zeroed (:147-157); column n carries k
  for (int o = threadIdx.x; o < m * ldr; o += blockDim.x) {
    const int i = o / ldr, j = o - i * ldr;
    Rhs[o] = j == n ? kp[i] : (((fm >> i) & 1u) ? -Q[(n + i) * ldq + j] : 0.0);
  }
  __syncthreads();
  g_lu_solve(Grp<kLargeThreads>(), m, Hf, m, piv, Rhs, ldr, n);
  __syncthreads();
  for (int o = threadIdx.x; o < m * ldr; o += blockDim.x) {          // P = [Qux | qu] + Quu [K | k]  (unmasked, Q6)
    const int i = o / ldr, j = o - i * ldr;
    const double kv = Rhs[o];
    double a = j < n ? Q[(n + i) * ldq + j] : qu[i];
    for (int l = 0; l < m; ++l) a += Huu[i * m + l] * Rhs[l * ldr + j];
    KK[o] = kv;
    P[o] = a;
    if (j < n) p.Ks[idx * m * n + i * n + j] = (R)kv;
    else {
      p.ks[idx * m + i] = (R)kv;
      if (p.free_mask) p.free_mask[idx * m + i] = (unsigned char)((fm >> i) & 1u);
    }
  }
  if (threadIdx.x == 0) {
    if (p.n_qp) p.n_qp[idx] = 1 + sh_it;
    eflags[e] |= sh_status;
  }
}

// 0.5 v^T C v + c . v for one element: C v by rows (cta_rowdot), then sum_k v_k (0.5 (C v)_k + c_k) on warp 0 in a fixed
// order.  Every thread gets the value; y [s] and red [1] are scratch.
template <typename R>
__device__ __forceinline__ double large_quad_cost(int s, const R* Ct, const R* ct, const double* v, double* y, double* red) {
  cta_rowdot(s, s, [&](int i, int k) -> double { return (double)Ct[i * s + k]; }, v, [](int) -> double { return 0.0; },
             [&](int i, double a) { y[i] = a; });
  __syncthreads();
  if (threadIdx.x < 32) {
    double a = 0.0;
    for (int k = threadIdx.x; k < s; k += 32) a += v[k] * (0.5 * y[k] + (double)ct[k]);
    for (int d = 16; d > 0; d >>= 1) a += __shfl_xor_sync(0xffffffffu, a, d);
    if (threadIdx.x == 0) *red = a;
  }
  __syncthreads();
  const double r = *red;
  __syncthreads();
  return r;
}

// forward_rec (mpc_step.py:175-286): passes at alpha = ls_decay^pass until cost <= old cost or max_ls_trials passes
// (Q5).  The nominal trajectory's cost (:191) is evaluated inside the first pass.  max_ls_trials < 0: the gains only;
// the flags of the sweep are written and nothing else.
template <typename R>
__global__ void __launch_bounds__(kLargeThreads) mpc_large_ls_kernel(MpcFwdParams<R> p, const int* eflags) {
  extern __shared__ double lsm[];
  if (p.skip && *p.skip) return;
  const int n = p.n, m = p.m, s = n + m, e = blockIdx.x, T = p.T;
  int status = eflags[e];
  if (p.max_ls_trials < 0) {
    if (threadIdx.x == 0 && p.flags) p.flags[e] = status;
    return;
  }
  double* tau = lsm;            // [s]  [x; u] of this pass
  double* tau0 = tau + s;       // [s]  nominal [x; u] (first pass)
  double* y = tau0 + s;         // [s]
  double* xnew = y + s;         // [n]
  double* dxv = xnew + n;       // [n]
  double* red = dxv + n;        // [1]
  const double decay = (double)p.ls_decay;
  double alpha = 1.0, old_cost = 0.0, cost = 0.0;
  int trial = 0;
  for (;;) {
    const bool first = trial == 0;
    cost = 0.0;
    for (int t = 0; t < T; ++t) {
      const size_t idx = (size_t)t * p.B + e;
      for (int o = threadIdx.x; o < n; o += blockDim.x) {
        const double xn = (double)p.x_nom[idx * n + o];
        const double xv = t == 0 ? xn : xnew[o];                                  // new_x[0] = states[0]
        tau[o] = xv;
        dxv[o] = t == 0 ? 0.0 : xv - xn;
      }
      if (first) for (int o = threadIdx.x; o < s; o += blockDim.x) tau0[o] = o < n ? (double)p.x_nom[idx * n + o] : (double)p.u_nom[idx * m + o - n];
      __syncthreads();
      const R* Kt = p.Ks + idx * m * n;
      const R* kt = p.ks + idx * m;
      cta_rowdot(m, n, [&](int i, int k) -> double { return (double)Kt[i * n + k]; }, dxv,
                 [&](int i) -> double { return (double)p.u_nom[idx * m + i]; },
                 [&](int i, double v) {
                   double nu = v + alpha * (double)kt[i];                                // :209-219
                   nu = fmin(fmax(nu, (double)p.lo[idx * m + i]), (double)p.hi[idx * m + i]);   // :221
                   tau[n + i] = (double)(R)nu;
                 });
      __syncthreads();
      const R* Ct = p.tC + idx * s * s;
      const R* ct = p.tc + idx * s;
      const double obj = large_quad_cost(s, Ct, ct, tau, y, red);                  // :251
      cost += obj;
      if (first) old_cost += large_quad_cost(s, Ct, ct, tau0, y, red);
      for (int o = threadIdx.x; o < n; o += blockDim.x) p.x[idx * n + o] = (R)tau[o];
      for (int o = threadIdx.x; o < m; o += blockDim.x) {
        p.u[idx * m + o] = (R)tau[n + o];
        if (first && p.u_first) p.u_first[idx * m + o] = (R)tau[n + o];
      }
      if (threadIdx.x == 0 && p.objs) p.objs[idx] = (R)obj;
      if (t < T - 1) {
        const R* Ft = p.tF + idx * n * s;
        const R* ft = p.tf ? p.tf + idx * n : nullptr;
        cta_rowdot(n, s, [&](int i, int k) -> double { return (double)Ft[i * s + k]; }, tau,
                   [&](int i) -> double { return ft ? (double)ft[i] : 0.0; }, [&](int i, double v) { xnew[i] = (double)(R)v; });
      }
      __syncthreads();
    }
    if (!(cost > old_cost)) break;                   // NaN -> accepted, as in the reference
    if (trial + 1 >= p.max_ls_trials) { status |= FLAG_LS_CAPPED; break; }   // alpha stays the one of the trajectory just written
    alpha *= decay;
    ++trial;
  }
  if (threadIdx.x == 0) {
    p.costs[e] = (R)cost;
    if (p.old_costs) p.old_costs[e] = (R)old_cost;
    p.alphas[e] = (R)alpha;
    if (p.n_ls) p.n_ls[e] = trial + 1;
    if (p.flags) p.flags[e] = status;
  }
}

// util.get_traj for LinDx past n + m = 64: one CTA per element, the line search's row dots and rounding
template <typename R>
__global__ void __launch_bounds__(kLargeThreads) traj_large_kernel(TrajParams<R> p) {
  extern __shared__ double tsm[];
  if (p.skip && *p.skip) return;
  const int n = p.n, m = p.m, s = n + m, e = blockIdx.x, T = p.T;
  double* tau = tsm;            // [x; u]
  double* xnew = tsm + s;
  for (int o = threadIdx.x; o < n; o += blockDim.x) tau[o] = (double)p.x0[(size_t)e * n + o];
  __syncthreads();
  for (int t = 0; t < T; ++t) {
    const size_t idx = (size_t)t * p.B + e;
    for (int o = threadIdx.x; o < n; o += blockDim.x) p.x[idx * n + o] = (R)tau[o];
    if (t == T - 1) break;
    for (int o = threadIdx.x; o < m; o += blockDim.x) tau[n + o] = (double)p.u[idx * m + o];
    __syncthreads();
    const R* Ft = p.F + idx * n * s;
    const R* ft = p.f ? p.f + idx * n : nullptr;
    cta_rowdot(n, s, [&](int i, int k) -> double { return (double)Ft[i * s + k]; }, tau,
               [&](int i) -> double { return ft ? (double)ft[i] : 0.0; }, [&](int i, double v) { xnew[i] = (double)(R)v; });
    __syncthreads();
    for (int o = threadIdx.x; o < n; o += blockDim.x) tau[o] = xnew[o];
    __syncthreads();
  }
}

}  // namespace dmpc
