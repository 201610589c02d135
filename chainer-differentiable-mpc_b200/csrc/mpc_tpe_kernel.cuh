// MPCstep.forward for single-input systems with a small state (m = 1, n <= 4: the pendulum of env_dx/il_exp.py, the
// reference's one-variable example): ONE THREAD owns one batch element and keeps the whole recursion in registers.
//
// Why (profiles/r1/r2b_mpc_forward_c1.summary.txt): the group-per-element kernel (mpc_forward_kernel, 4 lanes per element,
// state in shared memory, a group barrier between every few flops, the generic LU-based g_pnqp) spends 52 k warp
// instructions at ~9 cycles each on the batch-64 pendulum step - 239 us of dependent-chain latency on ONE CTA.  For
// s = n + m = 4 a step of the Riccati recursion is ~250 flops: it fits a thread's registers, needs no barrier, no shared
// memory and no LU - PNQP for m = 1 is the scalar branch of the reference (mpc/pnqp.py:77-78, 133-134).
//
// Same semantics as mpc_forward_kernel (reference mpc/mpc_step.py:70-328), including both couplings: with BATCH the CTA
// (or the CTAs of one thread-block cluster) hold the whole batch and PNQP's convergence test / line-search exit are
// batch_or reductions (common.cuh), exactly where the reference has xp.sum / xp.max over the batch (pnqp.py:139-144, 172-187).
#pragma once
#include "mpc_kernels.cuh"

namespace dmpc {

// scalar projected-Newton box QP: minimise 0.5 H x^2 + q x on [lo, hi]; x in = clamped start, out = solution.
// Returns the iteration index like g_pnqp; *Hf_out = last masked Hessian + REG (the "factor"), *is_free = control is free.
template <bool BATCH, typename R>
__device__ __forceinline__ int pnqp_scalar(R H, R q, R lo, R hi, R& x, R* Hf_out, bool* is_free, int n_iter, int* status,
                                           unsigned& bphase) {
  bool act = false;
  R Hf = H;
  int it = 0;
  for (it = 0; it < n_iter; ++it) {
    const R g = q + H * x;
    act = ((x == lo) && (g > R(0))) || ((x == hi) && (g < R(0)));            // pnqp.py:110
    Hf = (act ? R(0) : H) + R(DMPC_PNQP_REG);
    // a zero numerator sends the compiler's double division down its slow path (~60 dependent instructions, taken by
    // the whole warp); 0 / Hf is 0 (Hf = H + reg > 0 or the quotient's sign is irrelevant: only |dx| and x + alpha dx are used)
    const R dx = (act || g == R(0)) ? R(0) : -g / Hf;
    // pnqp.py:139-140 tests sqrt(dx^2) >= tol.  sqrt(dx*dx) is within 2 ulp of |dx|, so away from the threshold |dx| decides
    // (same answer, no square root on the dependent chain); within ~50 ulp of it the literal expression is evaluated.
    const R adx = fabs(dx);
    constexpr double mg = sizeof(R) == 8 ? 1e-14 : 1e-5;
    bool large;
    if (adx >= R(DMPC_PNQP_TOL * (1.0 + mg))) large = true;
    else if (adx <= R(DMPC_PNQP_TOL * (1.0 - mg))) large = false;
    else large = sqrt(dx * dx) >= R(DMPC_PNQP_TOL);
    bool any_large = large;
    if (BATCH) any_large = batch_or(large ? 1 : 0, bphase) != 0;
    if (!any_large) break;                                                    // x is returned before dx is applied (Q4)
    R alpha = R(1);
    const R f0 = R(0.5) * ((x * H) * x) + q * x;
    int count = 0;
    bool go = true;
    R xh = x;
    while (go) {                                                              // Armijo backtracking, pnqp.py:162-190
      xh = fmin(fmax(x + alpha * dx, lo), hi);
      R lhs;
      if (large) lhs = (f0 - (R(0.5) * ((xh * H) * xh) + q * xh)) / (g * (x - xh));
      else lhs = R(DMPC_PNQP_GAMMA + 1e-6);
      const bool fail = lhs <= R(DMPC_PNQP_GAMMA);                            // NaN -> not fail
      if (fail) alpha *= R(DMPC_PNQP_DECAY);
      ++count;
      bool stop = !fail;
      if (BATCH) stop = batch_or(stop ? 1 : 0, bphase) != 0;
      go = !stop && count < DMPC_PNQP_MAX_LS;
    }
    x = xh;
  }
  if (it >= n_iter) { it = n_iter - 1; if (status) *status |= FLAG_QP_NOT_CONVERGED; }
  *Hf_out = Hf;
  *is_free = !act;
  return it;
}

// Operands of one Riccati step / one rollout step, loaded at the top of the step.  (Requesting step t-1's operands before
// step t is computed - a register double buffer - was measured and is slower: 255 registers + spills, 96-101 us against
// 90 us on the batch-64 step, profiles/r2/tpe_variants_ab.txt.)
template <typename R, int N>
struct TpeSweepOps {
  R C[N + 1][N + 1], c[N + 1], tau[N + 1], lo, hi, F[N][N + 1], f[N];
};
template <typename R, int N>
struct TpeRollOps {
  R xn[N], un, lo, hi, C[(N + 1) * (N + 1)], c[N + 1];
};

template <typename R, int N>
__device__ __forceinline__ void tpe_load_sweep(const MpcFwdParams<R>& p, int t, int e, bool have_f, TpeSweepOps<R, N>& o) {
  constexpr int n = N, s = N + 1;
  const size_t idx = (size_t)t * p.B + e;
  const R* Cg = p.C + idx * s * s; const R* cg = p.c + idx * s;
#pragma unroll
  for (int i = 0; i < s; ++i) {
#pragma unroll
    for (int j = 0; j < s; ++j) o.C[i][j] = Cg[i * s + j];
    o.c[i] = cg[i];
  }
#pragma unroll
  for (int i = 0; i < n; ++i) o.tau[i] = p.x_nom[idx * n + i];
  o.tau[n] = p.u_nom[idx];
  o.lo = p.lo[idx]; o.hi = p.hi[idx];
  if (t < p.T - 1) {
    const R* Fg = p.F + idx * n * s;
#pragma unroll
    for (int i = 0; i < n; ++i)
#pragma unroll
      for (int j = 0; j < s; ++j) o.F[i][j] = Fg[i * s + j];
#pragma unroll
    for (int i = 0; i < n; ++i) o.f[i] = have_f ? p.f[idx * n + i] : R(0);
  }
}

template <typename R, int N>
__device__ __forceinline__ void tpe_load_roll(const MpcFwdParams<R>& p, int t, int e, TpeRollOps<R, N>& o) {
  constexpr int n = N, s = N + 1;
  const size_t idx = (size_t)t * p.B + e;
#pragma unroll
  for (int i = 0; i < n; ++i) o.xn[i] = p.x_nom[idx * n + i];
  o.un = p.u_nom[idx]; o.lo = p.lo[idx]; o.hi = p.hi[idx];
  const R* Cg = p.tC + idx * s * s; const R* cg = p.tc + idx * s;
#pragma unroll
  for (int i = 0; i < s * s; ++i) o.C[i] = Cg[i];
#pragma unroll
  for (int i = 0; i < s; ++i) o.c[i] = cg[i];
}

// shared-memory strides (in elements), odd so that the lanes of a warp fall into different banks
__host__ __device__ inline int tpe_kk_stride(int T, int n) { return (T * (n + 1)) | 1; }        // K_t | k_t per element
__host__ __device__ inline int tpe_stash_stride(int T, int n) { return (T * (n + 2)) | 1; }     // x_t | u_t | obj_t per lane

// MAXT = largest CTA the instantiation is launched with (register budget: 256 threads leave 255 registers per thread).
// NA   = lanes per element.  NA = 1: plain thread-per-element.  NA = 4: SPECULATIVE PARALLEL LINE SEARCH - the four
//        adjacent lanes of an element run the Riccati sweep redundantly (same registers, no communication) and then roll
//        out the four candidates alpha = decay^(4 r + a), a = 0..3, of round r at the same time; the first candidate (in
//        the reference's order) whose cost does not exceed the old cost wins (mpc_step.py:196, Q5).  The reference
//        evaluates the candidates one after the other; each one is independent of the previous ones, so the selected
//        alpha and trajectory are the same - the dependent chain is one horizon pass instead of (1 + trials) passes.
//        Lane 0 writes its candidate straight to x, u, objs; lanes 1..3 keep theirs in shared memory (p.tpe_stash) and the
//        winner copies it out - without the stash the winner rolls the horizon a second time.
template <typename R, int N, bool BATCH, int MAXT, int NA>
__global__ void __launch_bounds__(MAXT) mpc_forward_tpe_kernel(MpcFwdParams<R> p) {
  static_assert(NA == 1 || NA == 4, "lanes per element");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int n = N, s = N + 1;
  const int T = p.T, B = p.B;
  if (p.skip && *p.skip) return;                            // device-resident BoxDDP loop already exited (uniform)
  const int gt = blockIdx.x * blockDim.x + threadIdx.x;
  const int a = (NA > 1) ? (threadIdx.x % NA) : 0;          // candidate lane
  int e = gt / NA;
  const bool valid = e < B;
  if (!valid) { if (!BATCH && NA == 1) return; e = B - 1; } // padding threads shadow element B-1 (barrier / shuffle uniform)
  const bool writer = valid && a == 0;
  const size_t tb = (size_t)B;
  const bool expand = p.need_expand != 0;
  const bool have_f = (p.f != nullptr) && !expand;          // f_hat = None after the Taylor shift (mpc_step.py:317)
  int status = 0;
  unsigned bphase = 0;                                      // batch_or flag slot (BATCH coupling over a cluster)
  // NA > 1: K_t, k_t of the element are handed from the sweep to its candidate lanes through shared memory
  R* Kk = reinterpret_cast<R*>(smem_raw) + (size_t)(threadIdx.x / NA) * tpe_kk_stride(T, n);
  const bool use_stash = NA > 1 && p.tpe_stash != 0;
  R* stash = reinterpret_cast<R*>(smem_raw) + (size_t)(blockDim.x / NA) * tpe_kk_stride(T, n) +
             (size_t)((threadIdx.x / NA) * (NA - 1) + (a > 0 ? a - 1 : 0)) * tpe_stash_stride(T, n);

  // =========================== backward_rec (mpc_step.py:70-173) ===========================
  {
    R V[n][n], v[n];
    R kprev = R(0);
    for (int t = T - 1; t >= 0; --t) {
      const size_t idx = (size_t)t * tb + e;
      TpeSweepOps<R, N> cur;
      tpe_load_sweep<R, N>(p, t, e, have_f, cur);
      const R lb = cur.lo - cur.tau[n], ub = cur.hi - cur.tau[n];             // :136-138
      if (lb > ub) status |= FLAG_BAD_BOUNDS;                                  // the reference asserts (:139)
      R Q[s][s], q[s];
#pragma unroll
      for (int o = 0; o < s; ++o) {                                            // Taylor shift c_hat = C tau + c (:305-316)
        R acc = cur.c[o];
        if (expand) {
#pragma unroll
          for (int j = 0; j < s; ++j) acc += cur.C[o][j] * cur.tau[j];
        }
        q[o] = acc;
      }
      if (t == T - 1) {
#pragma unroll
        for (int i = 0; i < s; ++i)
#pragma unroll
          for (int j = 0; j < s; ++j) Q[i][j] = cur.C[i][j];
      } else {
        R Mx[n][s], mv[n];
#pragma unroll
        for (int i = 0; i < n; ++i) {                                          // Mx = V F ; mv = V f + v
#pragma unroll
          for (int j = 0; j < s; ++j) {
            R acc = R(0);
#pragma unroll
            for (int k = 0; k < n; ++k) acc += V[i][k] * cur.F[k][j];
            Mx[i][j] = acc;
          }
          R acc = v[i];
          if (have_f) {
#pragma unroll
            for (int k = 0; k < n; ++k) acc += V[i][k] * cur.f[k];
          }
          mv[i] = acc;
        }
#pragma unroll
        for (int i = 0; i < s; ++i) {                                          // Q = C + F^T Mx ; q = c_hat + F^T mv
#pragma unroll
          for (int j = 0; j < s; ++j) {
            R acc = cur.C[i][j];
#pragma unroll
            for (int k = 0; k < n; ++k) acc += cur.F[k][i] * Mx[k][j];
            Q[i][j] = acc;
          }
#pragma unroll
          for (int k = 0; k < n; ++k) q[i] += cur.F[k][i] * mv[k];
        }
      }
      // ---- PNQP on (Quu, qu, lb, ub), warm start k_{t+1} (:141-146)
      const R Huu = Q[n][n], quu = q[n];
      if (t == T - 1) kprev = fmin(fmax(-quu / Huu, lb), ub);
      else kprev = fmin(fmax(kprev, lb), ub);
      R Hf; bool is_free;
      const int it = pnqp_scalar<BATCH>(Huu, quu, lb, ub, kprev, &Hf, &is_free, p.n_qp_iter, &status, bphase);
      R K[n], P[s];
#pragma unroll
      for (int j = 0; j < n; ++j)                                              // rows of clamped controls zeroed (:147-157)
        K[j] = (is_free && Q[n][j] != R(0)) ? -Q[n][j] / Hf : R(0);            // (0 / Hf without the division's slow path)
#pragma unroll
      for (int j = 0; j < n; ++j) P[j] = Q[n][j] + Huu * K[j];                // P = [Qux | qu] + Quu [K | k]  (unmasked, Q6)
      P[n] = quu + Huu * kprev;
      if (writer) {
#pragma unroll
        for (int j = 0; j < n; ++j) p.Ks[idx * n + j] = K[j];
        p.ks[idx] = kprev;
        if (p.free_mask) p.free_mask[idx] = (unsigned char)(is_free ? 1 : 0);
        if (p.n_qp) p.n_qp[idx] = 1 + it;
      }
      if (NA > 1 && a == 0) {
#pragma unroll
        for (int j = 0; j < n; ++j) Kk[t * (n + 1) + j] = K[j];
        Kk[t * (n + 1) + n] = kprev;
      }
      if (t > 0) {
#pragma unroll
        for (int i = 0; i < n; ++i) {                                          // [V | v] = [Qxx | qx] + Qxu [K | k] + K^T P
#pragma unroll
          for (int j = 0; j < n; ++j) V[i][j] = (Q[i][j] + Q[i][n] * K[j]) + K[i] * P[j];
          v[i] = (q[i] + Q[i][n] * kprev) + K[i] * P[n];
        }
      }
    }
  }
  if (BATCH) batch_or_finish();                             // the last batch-wide decision is behind us
  if (p.max_ls_trials < 0) {                                // backward_rec only: the line search runs on the host
    if (writer && p.flags) p.flags[e] = status;
    return;
  }
  if (NA > 1) __syncwarp();                                 // K_t, k_t of lane a = 0 are visible to its candidate lanes
  else if (!valid) return;                                  // padding threads were only needed for the PNQP barriers

  // =========================== forward_rec (mpc_step.py:175-286) ===========================
  // One horizon pass evaluates the cost of the nominal trajectory (xpget_cost, :191) AND the candidate alpha of this
  // lane.  mode 0: evaluate only; 1: write x, u, objs (+ u_first on the first pass); 2: keep x, u, objs in the stash.
  const bool linear = p.dynamics == DMPC_DYN_LINEAR;
  R old_cost = R(0), cost = R(0), alpha = R(1);
  auto rollout = [&](R al, int mode, bool first) {
    R oc = R(0), cc = R(0);
    R xnew[n];
    for (int t = 0; t < T; ++t) {
      const size_t idx = (size_t)t * tb + e;
      TpeRollOps<R, N> cur;
      tpe_load_roll<R, N>(p, t, e, cur);
      R Fr[n][s], fr[n];
      if (linear && t < T - 1) {                                               // true dynamics of this step, requested early
#pragma unroll
        for (int o = 0; o < n; ++o) {
#pragma unroll
          for (int j = 0; j < s; ++j) Fr[o][j] = p.tF[idx * n * s + o * s + j];
          fr[o] = p.tf ? p.tf[idx * n + o] : R(0);
        }
      }
      R tau[s], tn[s];
      R dxv[n];
#pragma unroll
      for (int i = 0; i < n; ++i) {
        if (t == 0) xnew[i] = cur.xn[i];                                       // new_x[0] = states[0]
        tau[i] = xnew[i]; tn[i] = cur.xn[i];
        dxv[i] = (t == 0) ? R(0) : xnew[i] - cur.xn[i];
      }
      tn[n] = cur.un;
      R Kt[n], kt;
      if (NA > 1) {
#pragma unroll
        for (int i = 0; i < n; ++i) Kt[i] = Kk[t * (n + 1) + i];
        kt = Kk[t * (n + 1) + n];
      } else {
#pragma unroll
        for (int i = 0; i < n; ++i) Kt[i] = p.Ks[idx * n + i];
        kt = p.ks[idx];
      }
      R nu = dot2(Kt, 1, dxv, n, R(0)) + cur.un;                               // :209
      nu += al * kt;                                                           // :213-219
      nu = fmin(fmax(nu, cur.lo), cur.hi);                                     // :221
      tau[n] = nu;
      // objectives 0.5 (tau^T C) tau + tau . c   (:251) of the candidate and (first pass) of the nominal trajectory
      R quad = R(0), lin = R(0), quad0 = R(0), lin0 = R(0);
#pragma unroll
      for (int j = 0; j < s; ++j) {
        R tj = R(0), tj0 = R(0);
#pragma unroll
        for (int i = 0; i < s; ++i) { const R cij = cur.C[i * s + j]; tj += tau[i] * cij; tj0 += tn[i] * cij; }
        quad += tj * tau[j]; quad0 += tj0 * tn[j];
        lin += tau[j] * cur.c[j]; lin0 += tn[j] * cur.c[j];
      }
      const R obj = R(0.5) * quad + lin;
      cc += obj;
      if (first) oc += R(0.5) * quad0 + lin0;
      if (mode == 1) {
#pragma unroll
        for (int i = 0; i < n; ++i) p.x[idx * n + i] = tau[i];
        p.u[idx] = tau[n];
        if (first && p.u_first) p.u_first[idx] = tau[n];
        if (p.objs) p.objs[idx] = obj;
      } else if (mode == 2) {
#pragma unroll
        for (int i = 0; i < s; ++i) stash[t * (n + 2) + i] = tau[i];
        stash[t * (n + 2) + s] = obj;
      }
      if (t < T - 1) {
        if (linear) {
#pragma unroll
          for (int o = 0; o < n; ++o) xnew[o] = dot2(Fr[o], 1, tau, s, fr[o]);
        } else {
          if constexpr (N == 3) {
            R nx[3];
            pendulum_step(p.dyn_params, tau, tau[n], nx);
            xnew[0] = nx[0]; xnew[1] = nx[1]; xnew[2] = nx[2];
          }
        }
      }
    }
    if (first) old_cost = oc;
    cost = cc;
  };

  int trial = 0;                                            // index of the accepted (or, capped, the last) candidate
  if (NA == 1) {
    bool done = false;
    while (!done) {
      rollout(alpha, valid ? 1 : 0, trial == 0);
      const bool worse = cost > old_cost;                   // NaN -> accepted, as in the reference
      if (!worse) done = true;
      else if (trial + 1 >= p.max_ls_trials) { status |= FLAG_LS_CAPPED; done = true; }   // alpha = the one written
      else { alpha *= p.ls_decay; ++trial; }
    }
  } else {
    const unsigned full = 0xffffffffu;
    const int qbase = (threadIdx.x & 31) & ~(NA - 1);
    int win = -1;                                           // winning candidate index
    R wcost = R(0), walpha = R(1);
    // warp-uniform loop: a quad whose winner is known idles (but keeps voting) until every quad of the warp is done
    for (int round = 0; __any_sync(full, win < 0); ++round) {
      const bool open = win < 0;
      const int k = NA * round + a;
      R al = R(1);
      for (int i = 0; i < k; ++i) al *= p.ls_decay;         // the reference's repeated multiplication (bit-identical)
      const bool in_range = k < p.max_ls_trials;
      // lane 0 writes its candidate in place (round 0: it also is u_first); a later winner overwrites it
      const int mode = (a == 0) ? (valid ? 1 : 0) : (use_stash ? 2 : 0);
      if (open && in_range) rollout(al, mode, round == 0);
      if (round == 0) old_cost = __shfl_sync(full, old_cost, qbase);            // every lane computed the same value
      const bool ok = open && in_range && !(cost > old_cost);                   // NaN -> accepted, as in the reference
      const unsigned bal = (__ballot_sync(full, ok) >> qbase) & ((1u << NA) - 1u);
      int wa = -1;
      bool capped = false;
      if (bal) wa = __ffs(bal) - 1;
      else if (NA * (round + 1) >= p.max_ls_trials) { wa = (p.max_ls_trials - 1) - NA * round; capped = true; }
      const int src = qbase + (wa > 0 ? wa : 0);
      const R c_w = __shfl_sync(full, cost, src), a_w = __shfl_sync(full, al, src);
      if (open && wa >= 0) {
        win = NA * round + wa;
        wcost = c_w; walpha = a_w;
        if (capped) status |= FLAG_LS_CAPPED;
        if (wa != 0 && a == wa && valid) {                  // a stashing lane won: its trajectory goes out
          if (use_stash) {
            for (int t = 0; t < T; ++t) {
              const size_t idx = (size_t)t * tb + e;
#pragma unroll
              for (int i = 0; i < n; ++i) p.x[idx * n + i] = stash[t * (n + 2) + i];
              p.u[idx] = stash[t * (n + 2) + n];
              if (p.objs) p.objs[idx] = stash[t * (n + 2) + s];
            }
          } else {
            rollout(al, 1, false);
          }
        }
      }
    }
    trial = win;
    cost = wcost; alpha = walpha;
  }
  if (writer) {
    p.costs[e] = cost;
    if (p.old_costs) p.old_costs[e] = old_cost;
    p.alphas[e] = alpha;
    if (p.n_ls) p.n_ls[e] = trial + 1;
    if (p.flags) p.flags[e] = status;
  }
}

}  // namespace dmpc
