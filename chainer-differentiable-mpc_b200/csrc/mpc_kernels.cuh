// Box-DDP / iLQR step on sm_100a: projected-Newton box QP (PNQP), the bounded Riccati
// sweep, and the fused line-search rollout.
//
//   g_pnqp             = PNQP                    (reference mpc/pnqp.py:37-201)
//   pnqp_kernel        = standalone batched PNQP (same)
//   mpc_forward_kernel = MPCstep.forward: Taylor shift (:305-317) + backward_rec (:70-173)
//                        + forward_rec line search (:175-286) in ONE launch
//   active_mask_kernel = mpc_step.py:363-364
//   traj / pendulum kernels = util.get_traj (util.py:201-236), PendulumDx.forward
//                        (env_dx/pendulum.py:65-102) and its analytic linearisation
//                        (replaces mpc/approximate.py:77-119)
//
// Coupling (SURVEY.md H2): ELEMENT = the reference's control flow with n_batch == 1 on every
// element; BATCH = the literal whole-batch control flow, available when the whole batch is
// resident in one CTA (block-wide OR-reductions stand in for the reference's xp.sum / xp.max).
#pragma once
#include "common.cuh"

namespace dmpc {

#define DMPC_PNQP_GAMMA 0.1
#define DMPC_PNQP_DECAY 0.1
#define DMPC_PNQP_REG 1e-11
#define DMPC_PNQP_TOL 1e-4
#define DMPC_PNQP_MAX_LS 10

// dot product with two interleaved accumulators; shared by every rollout so that a re-rolled
// trajectory reproduces a previous one bit for bit.
template <typename R>
__device__ __forceinline__ R dot2(const R* a, int sa, const R* b, int n, R init) {
  R a0 = init, a1 = R(0);
  int k = 0;
  for (; k + 1 < n; k += 2) { a0 = fma_rn(a[k * sa], b[k], a0); a1 = fma_rn(a[(k + 1) * sa], b[k + 1], a1); }
  if (k < n) a0 = fma_rn(a[k * sa], b[k], a0);
  return add_rn(a0, a1);
}

// 0.5 * (x^T H) x + q^T x  evaluated like util.xpbquad / xpbdot (reference pnqp.py:26-33)
template <typename R>
__device__ __forceinline__ R qp_objective(const R* H, int ldh, const R* q, const R* x, int m) {
  R quad = R(0), lin = R(0);
  for (int j = 0; j < m; ++j) {
    R t = R(0);
    for (int i = 0; i < m; ++i) t += x[i] * H[i * ldh + j];
    quad += t * x[j];
    lin += q[j] * x[j];
  }
  return R(0.5) * quad + lin;
}

// Projected-Newton box QP for ONE element, executed by the SG (<=32) lanes of `sg`.
//   H[m x m] (ld ldh), q, lo, hi: shared memory, read-only.  x: in = clamped start, out = solution.
//   On return Hf holds the LU of the last masked Hessian (+REG I), piv its pivots.
// Returns the iteration index i (as the reference) ; *free_mask bit r = control r is free;
// *status gets FLAG_QP_NOT_CONVERGED when the n_iter cap is hit.
// BATCH: decisions are OR-reduced over the CTA (all threads of the CTA must call this function).
template <int SG, int MMAX, bool BATCH, typename R>
__device__ __forceinline__ int g_pnqp(const Grp<SG>& sg, int m, const R* H, int ldh, const R* q, const R* lo,
                                      const R* hi, R* x, R* Hf, int* piv, R* rhs, R* gbuf, R* xh,
                                      int n_iter, unsigned* free_mask, int* status, unsigned& bphase) {
  const int r = sg.lane;
  unsigned act = 0;
  int it = 0;
  for (it = 0; it < n_iter; ++it) {
    // gradient (lane r -> component r), active set by ballot
    bool a_r = false;
    R g_r = R(0);
    if (r < m) {
      g_r = q[r];
      for (int j = 0; j < m; ++j) g_r += H[r * ldh + j] * x[j];
      const R xr = x[r];
      a_r = ((xr == lo[r]) && (g_r > R(0))) || ((xr == hi[r]) && (g_r < R(0)));   // pnqp.py:110
      gbuf[r] = g_r;
    }
    act = (__ballot_sync(sg.mask, a_r) >> ((threadIdx.x & 31) & ~(SG - 1))) & ((m >= 32) ? 0xffffffffu : ((1u << m) - 1u));
    // masked Hessian + regulariser, masked gradient
    for (int o = r; o < m * m; o += SG) {
      const int i = o / m, j = o - i * m;
      R hv = (((act >> i) | (act >> j)) & 1u) ? R(0) : H[i * ldh + j];
      if (i == j) hv += R(DMPC_PNQP_REG);
      Hf[o] = hv;
    }
    if (r < m) rhs[r] = a_r ? R(0) : -g_r;          // rhs = -g_f  ->  dx = Hf^-1 rhs
    sg.sync();
    g_lu_factor<SG, MMAX>(sg, m, Hf, m, rhs, 1, 1, piv);
    g_back_subst(sg, m, Hf, m, rhs, 1, 1);
    sg.sync();
    R n2 = R(0);
    for (int j = 0; j < m; ++j) n2 += rhs[j] * rhs[j];
    // pnqp.py:139-140 tests sqrt(|dx|^2) >= tol; away from the threshold |dx|^2 against tol^2 gives the same answer without
    // the square root (whose n2 == 0 case - a converged, fully clamped QP - is the compiler's out-of-line slow path)
    constexpr double mg2 = sizeof(R) == 8 ? 1e-13 : 1e-4;
    bool large;
    if (n2 >= R(DMPC_PNQP_TOL * DMPC_PNQP_TOL * (1.0 + mg2))) large = true;
    else if (n2 <= R(DMPC_PNQP_TOL * DMPC_PNQP_TOL * (1.0 - mg2))) large = false;
    else large = sqrt(n2) >= R(DMPC_PNQP_TOL);
    bool any_large = large;
    if (BATCH) any_large = batch_or(large ? 1 : 0, bphase) != 0;
    if (!any_large) break;                          // returns x *before* applying dx (Q4)
    // Armijo backtracking (pnqp.py:162-190)
    R alpha = R(1);
    const R f0 = qp_objective(H, ldh, q, x, m);
    int count = 0;
    bool go = true;
    while (go) {
      if (r < m) {
        R v = x[r] + alpha * rhs[r];
        v = fmin(fmax(v, lo[r]), hi[r]);
        xh[r] = v;
      }
      sg.sync();
      R lhs;
      if (large) {
        R den = R(0);
        for (int j = 0; j < m; ++j) den += gbuf[j] * (x[j] - xh[j]);
        lhs = (f0 - qp_objective(H, ldh, q, xh, m)) / den;
      } else {
        lhs = R(DMPC_PNQP_GAMMA + 1e-6);            // pnqp.py:174
      }
      const bool fail = lhs <= R(DMPC_PNQP_GAMMA);  // NaN -> not fail
      if (fail) alpha *= R(DMPC_PNQP_DECAY);
      ++count;
      bool stop = !fail;                            // max_lhs > GAMMA or NaN
      if (BATCH) stop = batch_or(stop ? 1 : 0, bphase) != 0;
      go = !stop && count < DMPC_PNQP_MAX_LS;
      sg.sync();
    }
    if (r < m) x[r] = xh[r];
    sg.sync();
  }
  if (it >= n_iter) { it = n_iter - 1; if (status) *status |= FLAG_QP_NOT_CONVERGED; }
  *free_mask = ~act;
  return it;
}

// ------------------------------------------------------------------------------------------
template <typename R>
struct PnqpParams {
  int B, m, n_iter, coupling;
  const R* H; const R* q; const R* lo; const R* hi; const R* x_init;   // x_init nullable
  R* x; R* LU; int* piv; R* free_out; int* iters; int* flags;
};

template <typename R>
__host__ __device__ inline int pnqp_stride(int m) {
  const int W = 16 / (int)sizeof(R);
  const int opiv = 2 * rup(m * m, W) + 8 * rup(m, W);
  return rup(opiv + rup((m * 4 + (int)sizeof(R) - 1) / (int)sizeof(R), W), 128 / (int)sizeof(R)) + W;
}

// standalone PNQP: one group of SG lanes per element, regions carved from dynamic smem
template <typename R, int M, int SG, bool BATCH>
__global__ void pnqp_kernel(PnqpParams<R> p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int m = M > 0 ? M : p.m;
  constexpr int MMAX = M > 0 ? M : 32;
  const Grp<SG> sg;
  const int epb = blockDim.x / SG;
  const int eloc = threadIdx.x / SG;
  int e = blockIdx.x * epb + eloc;
  const bool valid = e < p.B;
  if (!valid) e = p.B - 1;
  const int W = 16 / (int)sizeof(R);
  const int oH = 0, oHf = rup(m * m, W), oq = oHf + rup(m * m, W), olo = oq + rup(m, W), ohi = olo + rup(m, W);
  const int ox = ohi + rup(m, W), orhs = ox + rup(m, W), og = orhs + rup(m, W), oxh = og + rup(m, W);
  const int opiv = oxh + rup(m, W);
  const int stride = pnqp_stride<R>(m);
  R* sm = reinterpret_cast<R*>(smem_raw) + (size_t)eloc * stride;
  R* H = sm + oH; R* Hf = sm + oHf; R* q = sm + oq; R* lo = sm + olo; R* hi = sm + ohi; R* x = sm + ox;
  R* rhs = sm + orhs; R* gb = sm + og; R* xh = sm + oxh; int* piv = reinterpret_cast<int*>(sm + opiv);
  for (int o = sg.lane; o < m * m; o += SG) H[o] = p.H[(size_t)e * m * m + o];
  for (int o = sg.lane; o < m; o += SG) {
    q[o] = p.q[(size_t)e * m + o]; lo[o] = p.lo[(size_t)e * m + o]; hi[o] = p.hi[(size_t)e * m + o];
  }
  sg.sync();
  if (p.x_init) {
    for (int o = sg.lane; o < m; o += SG) x[o] = fmin(fmax(p.x_init[(size_t)e * m + o], lo[o]), hi[o]);
  } else {
    // unconstrained minimiser -H^-1 q, clamped (pnqp.py:75-93)
    for (int o = sg.lane; o < m * m; o += SG) Hf[o] = H[o];
    for (int o = sg.lane; o < m; o += SG) rhs[o] = -q[o];
    sg.sync();
    g_lu_factor<SG, MMAX>(sg, m, Hf, m, rhs, 1, 1, (int*)nullptr);
    g_back_subst(sg, m, Hf, m, rhs, 1, 1);
    sg.sync();
    for (int o = sg.lane; o < m; o += SG) x[o] = fmin(fmax(rhs[o], lo[o]), hi[o]);
  }
  sg.sync();
  unsigned fm = 0; int status = 0;
  unsigned bphase = 0;
  for (int o = 0; o < m; ++o) if (lo[o] > hi[o]) status |= FLAG_BAD_BOUNDS;                       // pnqp.py:64 asserts
  const int it = g_pnqp<SG, MMAX, BATCH>(sg, m, H, m, q, lo, hi, x, Hf, piv, rhs, gb, xh, p.n_iter, &fm, &status, bphase);
  if (BATCH) batch_or_finish();
  if (valid) {
    for (int o = sg.lane; o < m; o += SG) {
      p.x[(size_t)e * m + o] = x[o];
      p.free_out[(size_t)e * m + o] = ((fm >> o) & 1u) ? R(1) : R(0);
      if (p.piv) p.piv[(size_t)e * m + o] = piv[o];
    }
    if (p.LU) for (int o = sg.lane; o < m * m; o += SG) p.LU[(size_t)e * m * m + o] = Hf[o];
    if (sg.lane == 0) { p.iters[e] = it; if (p.flags) p.flags[e] = status; }
  }
}

// ------------------------------------------------------------------------------------------
template <typename R>
struct MpcFwdParams {
  int T, B, n, m, F_T, need_expand, dynamics, coupling, max_ls_trials, n_qp_iter;
  R ls_decay;
  const R* C; const R* c; const R* F; const R* f;          // approximated model (C_hat, c_hat, F_hat, f_hat)
  const R* x_nom; const R* u_nom;                           // current_states, controls
  const R* lo; const R* hi;                                 // [T,B,m]
  const R* tC; const R* tc;                                 // true QuadCost
  const R* tF; const R* tf;                                 // true LinDx (dynamics == LINEAR); tf nullable
  R dyn_params[5];                                          // pendulum (g, m, l, dt, max_torque); 0 -> 0.05 / 2.0
  R* x; R* u;                                               // new trajectory
  R* Ks; R* ks;                                             // [T,B,m,n], [T,B,m]
  R* u_first;                                               // alpha = 1 controls (for full_du_norm)
  R* objs;                                                  // [T,B]
  R* costs; R* old_costs; R* alphas;                        // [B]
  int* n_qp;                                                // [T,B]   1 + i per timestep
  unsigned char* free_mask;                                 // [T,B,m]
  int* n_ls; int* flags;                                    // [B]
  const int* skip;                                          // device flag (nullable): non-zero -> the launch is a no-op
  int tpe_stash;                                            // mpc_forward_tpe_kernel: candidate-trajectory stash follows K|k in smem
};

// pendulum step (env_dx/pendulum.py:65-102, `simple` model); x=(cos,sin,dth), returns x'
template <typename R>
__device__ __forceinline__ void pendulum_step(const R* par, const R* x, R u, R* xn) {
  const R g = par[0], mass = par[1], l = par[2];
  const R dt = par[3] > R(0) ? par[3] : R(0.05), maxu = par[4] > R(0) ? par[4] : R(2.0);   // PendulumDx.dt / .max_torque
  const R uc = fmin(fmax(u, -maxu), maxu);
  const R cth = x[0], sth = x[1], dth = x[2];
  const R th = atan2(sth, cth);
  // same operation order as the reference expression, every op individually rounded (no FMA)
  const R t1 = mul_rn(mul_rn(R(-3.), g) / mul_rn(R(2.), l), -sth);
  const R u3 = mul_rn(R(3.), uc);
  const R t2 = u3 == R(0) ? u3 : u3 / mul_rn(mass, mul_rn(l, l));   // (0 / x = 0 without the division's slow path)
  const R newdth = add_rn(dth, mul_rn(dt, add_rn(t1, t2)));
  const R newth = add_rn(th, mul_rn(newdth, dt));
  xn[0] = cos(newth); xn[1] = sin(newth); xn[2] = newdth;
}

// analytic Jacobian of the `simple` pendulum step at (x, u) given x' = pendulum_step(x, u): F = [R S] row-major [3][4] and
// (nullable) f = x' - R x - S u, evaluated as (x' - R x) - S u like the reference (approximate.py:111-114).  Every
// operation is individually rounded, so the linearisation does not depend on which kernel it was inlined into.
template <typename R>
__device__ __forceinline__ void pendulum_jacobian(const R* par, const R* tau, const R* xn, R* Fo, R* fo) {
  const R g = par[0], mass = par[1], l = par[2];
  const R dt = par[3] > R(0) ? par[3] : R(0.05), maxu = par[4] > R(0) ? par[4] : R(2.0);
  const R c = tau[0], sn = tau[1], uraw = tau[3];
  const R r2 = add_rn(mul_rn(c, c), mul_rn(sn, sn));
  const R dth_dc = -sn / r2, dth_ds = c / r2;
  const R a = mul_rn(R(3.), g) / mul_rn(R(2.), l), bu = R(3.) / mul_rn(mass, mul_rn(l, l));
  const R inside = (uraw >= -maxu && uraw <= maxu) ? R(1) : R(0);
  const R dnw[4] = {R(0), mul_rn(dt, a), R(1), mul_rn(mul_rn(dt, bu), inside)};
  const R dnth[4] = {dth_dc, add_rn(dth_ds, mul_rn(dt, dnw[1])), dt, mul_rn(dt, dnw[3])};
  const R cn = xn[0], snn = xn[1];
  R J[3][4];
#pragma unroll
  for (int j = 0; j < 4; ++j) { J[0][j] = mul_rn(-snn, dnth[j]); J[1][j] = mul_rn(cn, dnth[j]); J[2][j] = dnw[j]; }
#pragma unroll
  for (int i = 0; i < 3; ++i) {
#pragma unroll
    for (int j = 0; j < 4; ++j) Fo[i * 4 + j] = J[i][j];
    if (fo) {
      R rx = R(0);
#pragma unroll
      for (int j = 0; j < 3; ++j) rx = fma_rn(J[i][j], tau[j], rx);
      fo[i] = add_rn(add_rn(xn[i], -rx), -mul_rn(J[i][3], uraw));
    }
  }
}

struct MpcLayout {
  int oC, oc, oF, of_, oxn, oun, olo, ohi, oK, ok, stage, st0, st1;
  int Q, q, V, v, Mx, mv, Hf, Rhs, P, chat, kprev, lb, ub, rhs1, gb, xh, tau, dxv, xnew, piv, total, stride;
};

template <typename R>
__host__ __device__ inline MpcLayout mpc_layout(int n, int m) {
  const int W = 16 / (int)sizeof(R);
  const int s = n + m;
  MpcLayout L;
  int o = 0;
  L.oC = o; o += rup(s * s, W);
  L.oc = o; o += rup(s, W);
  L.oF = o; o += rup(n * s, W);
  L.of_ = o; o += rup(n, W);
  L.oxn = o; o += rup(n, W);
  L.oun = o; o += rup(m, W);
  L.olo = o; o += rup(m, W);
  L.ohi = o; o += rup(m, W);
  L.oK = o; o += rup(m * n, W);
  L.ok = o; o += rup(m, W);
  L.stage = o;
  o = 0;
  L.st0 = o; o += L.stage;
  L.st1 = o; o += L.stage;
  L.Q = o; o += rup(s * s, W);
  L.q = o; o += rup(s, W);
  L.V = o; o += rup(n * n, W);
  L.v = o; o += rup(n, W);
  L.Mx = o; o += rup(n * s, W);
  L.mv = o; o += rup(n, W);
  L.Hf = o; o += rup(m * m, W);
  L.Rhs = o; o += rup(m * (n + 1), W);
  L.P = o; o += rup(m * (n + 1), W);
  L.chat = o; o += rup(s, W);
  L.kprev = o; o += rup(m, W);
  L.lb = o; o += rup(m, W);
  L.ub = o; o += rup(m, W);
  L.rhs1 = o; o += rup(m, W);
  L.gb = o; o += rup(m, W);
  L.xh = o; o += rup(m, W);
  L.tau = o; o += rup(s, W);
  L.dxv = o; o += rup(n, W);
  L.xnew = o; o += rup(n, W);
  L.piv = o; o += rup((m * 4 + (int)sizeof(R) - 1) / (int)sizeof(R), W);
  L.total = o;
  const int line = 128 / (int)sizeof(R);
  L.stride = rup(o, line) + W;
  return L;
}

template <typename R, int N, int M, int G, bool BATCH>
__global__ void mpc_forward_kernel(MpcFwdParams<R> p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int n = N > 0 ? N : p.n;
  const int m = M > 0 ? M : p.m;
  const int s = n + m;
  const int T = p.T, B = p.B;
  constexpr int MMAX = M > 0 ? M : 32;
  constexpr int SG = G <= 32 ? G : 32;
  const Grp<G> g;
  const Grp<SG> sg;
  const int epb = (G <= 32) ? (blockDim.x / G) : 1;
  const int eloc = (G <= 32) ? (threadIdx.x / G) : 0;
  int e = blockIdx.x * epb + eloc;
  const bool valid = e < B;
  if (!valid) e = B - 1;
  if (p.skip && *p.skip) return;                          // device-resident BoxDDP loop already exited (uniform)
  const MpcLayout L = mpc_layout<R>(n, m);
  R* sm = reinterpret_cast<R*>(smem_raw) + (size_t)eloc * L.stride;
  R* Q = sm + L.Q; R* q = sm + L.q; R* V = sm + L.V; R* v = sm + L.v; R* Mx = sm + L.Mx; R* mv = sm + L.mv;
  R* Hf = sm + L.Hf; R* Rhs = sm + L.Rhs; R* P = sm + L.P; R* chat = sm + L.chat; R* kprev = sm + L.kprev;
  R* lb = sm + L.lb; R* ub = sm + L.ub; R* rhs1 = sm + L.rhs1; R* gb = sm + L.gb; R* xh = sm + L.xh;
  R* tau = sm + L.tau; R* dxv = sm + L.dxv; R* xnew = sm + L.xnew;
  int* piv = reinterpret_cast<int*>(sm + L.piv);
  const size_t tb = (size_t)B;
  const int ldr = n + 1;
  const bool expand = p.need_expand != 0;
  const bool have_f = (p.f != nullptr) && !expand;       // f_hat = None after the Taylor shift (:317)
  int status = 0;
  unsigned bphase = 0;                                   // batch_or flag slot (BATCH coupling over a cluster)

  // =========================== backward_rec (mpc_step.py:70-173) ===========================
  {
    auto load_tiles = [&](int t, int st) {
      R* base = sm + (st ? L.st1 : L.st0);
      const size_t idx = (size_t)t * tb + e;
      g_cp_async(g, base + L.oC, p.C + idx * s * s, s * s);
      g_cp_async(g, base + L.oc, p.c + idx * s, s);
      if (t < T - 1) {
        g_cp_async(g, base + L.oF, p.F + idx * n * s, n * s);
        if (have_f) g_cp_async(g, base + L.of_, p.f + idx * n, n);
      }
      g_cp_async(g, base + L.oxn, p.x_nom + idx * n, n);
      g_cp_async(g, base + L.oun, p.u_nom + idx * m, m);
      g_cp_async(g, base + L.olo, p.lo + idx * m, m);
      g_cp_async(g, base + L.ohi, p.hi + idx * m, m);
      cp_async_commit();
    };
    load_tiles(T - 1, 0);
    int st = 0;
    for (int t = T - 1; t >= 0; --t) {
      if (t > 0) { load_tiles(t - 1, st ^ 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
      g.sync();
      const R* base = sm + (st ? L.st1 : L.st0);
      const R* Ct = base + L.oC; const R* ct = base + L.oc; const R* Ft = base + L.oF; const R* ft = base + L.of_;
      const R* xn = base + L.oxn; const R* un = base + L.oun; const R* lot = base + L.olo; const R* hit = base + L.ohi;
      // Taylor shift: c_hat = C tau + c (:305-316)
      for (int o = g.lane; o < s; o += G) tau[o] = (o < n) ? xn[o] : un[o - n];
      for (int o = g.lane; o < m; o += G) { lb[o] = lot[o] - un[o]; ub[o] = hit[o] - un[o]; }    // :136-138
      for (int o = 0; o < m; ++o) if (lot[o] > hit[o]) status |= FLAG_BAD_BOUNDS;                 // the reference asserts (:139)
      g.sync();
      for (int o = g.lane; o < s; o += G) {
        R a = ct[o];
        if (expand) for (int j = 0; j < s; ++j) a += Ct[o * s + j] * tau[j];
        chat[o] = a;
      }
      if (t < T - 1) {
        g_gemm(g, n, s, n, Mx, s, (const R*)nullptr, 0, V, n, 1, Ft, s, 1);
        if (have_f) g_gemm(g, n, 1, n, mv, 1, v, 1, V, n, 1, ft, 1, 1);
        else for (int o = g.lane; o < n; o += G) mv[o] = v[o];
      }
      g.sync();
      if (t == T - 1) {
        for (int o = g.lane; o < s * s; o += G) Q[o] = Ct[o];
        for (int o = g.lane; o < s; o += G) q[o] = chat[o];
      } else {
        g_gemm(g, s, s, n, Q, s, Ct, s, Ft, 1, s, Mx, s, 1);
        for (int o = g.lane; o < s; o += G) {
          R a = chat[o];
          for (int k = 0; k < n; ++k) a += Ft[k * s + o] * mv[k];
          q[o] = a;
        }
      }
      g.sync();
      // ---- PNQP on (Quu, qu, lb, ub), warm start k_{t+1} (:141-146) --------------------------
      const R* Huu = Q + n * s + n;           // ld = s
      const R* quu = q + n;
      unsigned fm = 0;
      int it = 0;
      static_assert(!(BATCH && G > 32), "batch coupling needs sub-warp groups");
      if (G <= 32 || threadIdx.x < 32) {
        const bool worker = true;
        if (worker) {
          if (t == T - 1) {
            for (int o = sg.lane; o < m * m; o += SG) { const int i = o / m, j = o - i * m; Hf[o] = Huu[i * s + j]; }
            for (int o = sg.lane; o < m; o += SG) rhs1[o] = -quu[o];
            sg.sync();
            g_lu_factor<SG, MMAX>(sg, m, Hf, m, rhs1, 1, 1, (int*)nullptr);
            g_back_subst(sg, m, Hf, m, rhs1, 1, 1);
            sg.sync();
            for (int o = sg.lane; o < m; o += SG) kprev[o] = fmin(fmax(rhs1[o], lb[o]), ub[o]);
          } else {
            for (int o = sg.lane; o < m; o += SG) kprev[o] = fmin(fmax(kprev[o], lb[o]), ub[o]);
          }
          sg.sync();
        }
        if (worker)
          it = g_pnqp<SG, MMAX, BATCH>(sg, m, Huu, s, quu, lb, ub, kprev, Hf, piv, rhs1, gb, xh, p.n_qp_iter, &fm, &status, bphase);
        if (worker) {
          // K = -(LU)^-1 Qux with the rows of clamped controls zeroed (:147-157)
          for (int o = sg.lane; o < m * n; o += SG) {
            const int i = o / n, j = o - i * n;
            Rhs[i * ldr + j] = ((fm >> i) & 1u) ? -Q[(n + i) * s + j] : R(0);
          }
          for (int o = sg.lane; o < m; o += SG) Rhs[o * ldr + n] = kprev[o];
          sg.sync();
          g_lu_solve(sg, m, Hf, m, piv, Rhs, ldr, n);
          sg.sync();
        }
      }
      g.sync();
      // P = [Qux | qu] + Quu [K | k]  (unmasked, Q6)
      for (int o = g.lane; o < m * (n + 1); o += G) {
        const int i = o / (n + 1), j = o - i * (n + 1);
        R a = (j < n) ? Q[(n + i) * s + j] : q[n + i];
        for (int l = 0; l < m; ++l) a += Q[(n + i) * s + n + l] * Rhs[l * ldr + j];
        P[o] = a;
      }
      {
        const size_t idx = (size_t)t * tb + e;
        if (valid) {
          R* Kg = p.Ks + idx * m * n; R* kg = p.ks + idx * m;
          for (int o = g.lane; o < m * n; o += G) { const int i = o / n, j = o - i * n; Kg[o] = Rhs[i * ldr + j]; }
          for (int o = g.lane; o < m; o += G) {
            kg[o] = Rhs[o * ldr + n];
            if (p.free_mask) p.free_mask[idx * m + o] = (unsigned char)((fm >> o) & 1u);
          }
          if (g.lane == 0 && p.n_qp) p.n_qp[idx] = 1 + it;
        }
      }
      g.sync();
      if (t > 0) {
        for (int o = g.lane; o < n * (n + 1); o += G) {
          const int i = o / (n + 1), j = o - i * (n + 1);
          R a = (j < n) ? Q[i * s + j] : q[i];
          R b = R(0);
          for (int l = 0; l < m; ++l) {
            a += Q[i * s + n + l] * Rhs[l * ldr + j];
            b += Rhs[l * ldr + i] * P[l * (n + 1) + j];
          }
          if (j < n) V[i * n + j] = a + b; else v[i] = a + b;
        }
      }
      g.sync();
      st ^= 1;
    }
  }

  if (BATCH) batch_or_finish();      // last batch-wide decision is behind us: other CTAs of the cluster may exit
  if (p.max_ls_trials < 0) {         // backward_rec only: the caller runs the line search on the host (Python callables)
    if (valid && g.lane == 0 && p.flags) p.flags[e] = status;
    return;
  }

  // =========================== forward_rec (mpc_step.py:175-286) ===========================
  // Passes are the line-search trials with alpha = ls_decay^pass until cost <= old cost (Q5).  The cost of the nominal
  // trajectory (xpget_cost, :191) is evaluated inside the first pass, on the same C_t, c_t tiles: a separate pass for it
  // re-read every tile of the horizon (one third of this phase's DRAM traffic and barrier chain at ~1 trial per element).
  const bool linear = p.dynamics == DMPC_DYN_LINEAR;
  R alpha = R(1), old_cost = R(0), cost = R(0);
  int trial = 0;
  bool done = false;
  while (!done) {
    auto load_tiles = [&](int t, int st) {
      R* base = sm + (st ? L.st1 : L.st0);
      const size_t idx = (size_t)t * tb + e;
      g_cp_async(g, base + L.oC, p.tC + idx * s * s, s * s);
      g_cp_async(g, base + L.oc, p.tc + idx * s, s);
      if (t < T - 1 && linear) {
        g_cp_async(g, base + L.oF, p.tF + idx * n * s, n * s);
        if (p.tf) g_cp_async(g, base + L.of_, p.tf + idx * n, n);
      }
      g_cp_async(g, base + L.oxn, p.x_nom + idx * n, n);
      g_cp_async(g, base + L.oun, p.u_nom + idx * m, m);
      g_cp_async(g, base + L.olo, p.lo + idx * m, m);
      g_cp_async(g, base + L.ohi, p.hi + idx * m, m);
      g_cp_async(g, base + L.oK, p.Ks + idx * m * n, m * n);
      g_cp_async(g, base + L.ok, p.ks + idx * m, m);
      cp_async_commit();
    };
    g.sync();
    load_tiles(0, 0);
    cost = R(0);
    int st = 0;
    for (int t = 0; t < T; ++t) {
      if (t < T - 1) { load_tiles(t + 1, st ^ 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
      g.sync();
      const R* base = sm + (st ? L.st1 : L.st0);
      const R* Ct = base + L.oC; const R* ct = base + L.oc; const R* Ft = base + L.oF; const R* ft = base + L.of_;
      const R* xn = base + L.oxn; const R* un = base + L.oun; const R* lot = base + L.olo; const R* hit = base + L.ohi;
      const R* Kt = base + L.oK; const R* kt = base + L.ok;
      {
        if (t == 0) for (int o = g.lane; o < n; o += G) xnew[o] = xn[o];       // new_x[0] = states[0]
        g.sync();
        for (int o = g.lane; o < n; o += G) { tau[o] = xnew[o]; dxv[o] = (t == 0) ? R(0) : xnew[o] - xn[o]; }
        g.sync();
        for (int o = g.lane; o < m; o += G) {
          R nu = dot2(Kt + o * n, 1, dxv, n, R(0)) + un[o];                      // :209
          nu += alpha * kt[o];                                                   // :213-219
          nu = fmin(fmax(nu, lot[o]), hit[o]);                                   // :221
          tau[n + o] = nu;
        }
      }
      g.sync();
      R* tcol = chat;                                  // dead since the sweep: scratch for the column sums
      // objective 0.5 (tau^T C) tau + tau . c   (:251).  The s column sums (tau^T C)_j are split over the lanes; the two
      // length-s sums are then accumulated by every lane in the reference's order (same bits as the all-redundant loop,
      // s + 2 s instead of s^2 + 2 s multiply-adds per lane)
      const bool first = trial == 0;                   // this pass also evaluates the nominal trajectory (x_nom, u_nom)
      R* tcol0 = Rhs;                                  // dead since the sweep, m (n + 1) >= s entries
      for (int j = g.lane; j < s; j += G) {
        R tj = R(0), tj0 = R(0);
        for (int i = 0; i < s; ++i) {
          const R cij = Ct[i * s + j];
          tj += tau[i] * cij;
          if (first) tj0 += ((i < n) ? xn[i] : un[i - n]) * cij;
        }
        tcol[j] = tj;
        if (first) tcol0[j] = tj0;
      }
      g.sync();
      R quad = R(0), lin = R(0);
      for (int j = 0; j < s; ++j) {
        quad += tcol[j] * tau[j];
        lin += tau[j] * ct[j];
      }
      const R obj = R(0.5) * quad + lin;
      cost += obj;
      if (first) {
        R quad0 = R(0), lin0 = R(0);
        for (int j = 0; j < s; ++j) {
          const R tn = (j < n) ? xn[j] : un[j - n];
          quad0 += tcol0[j] * tn;
          lin0 += tn * ct[j];
        }
        old_cost += R(0.5) * quad0 + lin0;
      }
      {
        const size_t idx = (size_t)t * tb + e;
        if (valid) {
          for (int o = g.lane; o < n; o += G) p.x[idx * n + o] = tau[o];
          for (int o = g.lane; o < m; o += G) {
            p.u[idx * m + o] = tau[n + o];
            if (trial == 0 && p.u_first) p.u_first[idx * m + o] = tau[n + o];
          }
          if (g.lane == 0 && p.objs) p.objs[idx] = obj;
        }
        if (t < T - 1) {
          if (linear) {
            for (int o = g.lane; o < n; o += G) mv[o] = dot2(Ft + o * s, 1, tau, s, p.tf ? ft[o] : R(0));
          } else {
            if (g.lane == 0) pendulum_step(p.dyn_params, tau, tau[n], mv);
          }
          g.sync();
          for (int o = g.lane; o < n; o += G) xnew[o] = mv[o];
        }
      }
      g.sync();
      st ^= 1;
    }
    {
      const bool worse = cost > old_cost;             // NaN -> accepted, as in the reference
      if (!worse) done = true;
      else if (trial + 1 >= p.max_ls_trials) { status |= FLAG_LS_CAPPED; done = true; }            // alpha stays the one of the
      else { alpha *= p.ls_decay; ++trial; }                                                        // trajectory just written
    }
  }
  if (valid && g.lane == 0) {
    p.costs[e] = cost;
    if (p.old_costs) p.old_costs[e] = old_cost;
    p.alphas[e] = alpha;
    if (p.n_ls) p.n_ls[e] = trial + 1;
    if (p.flags) p.flags[e] = status;
  }
}

// ------------------------------------------------------------------------------------------
template <typename R>
__global__ void active_mask_kernel(const R* u, const R* lo, const R* hi, unsigned char* out, size_t count) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) out[i] = (fabs(u[i] - lo[i]) <= R(1e-8)) || (fabs(u[i] - hi[i]) <= R(1e-8));   // mpc_step.py:363-364
}

// util.get_traj for LinDx / pendulum: one thread per element (same dot2 order as the line search)
template <typename R>
struct TrajParams {
  int T, B, n, m, dynamics;
  const R* x0; const R* u; const R* F; const R* f;
  R dyn_params[5];
  R* x;            // [T,B,n]
  R* Fout; R* fout;  // pendulum linearisation outputs [T-1,B,3,4], [T-1,B,3] (nullable)
  const int* skip;   // device flag (nullable): non-zero -> the launch is a no-op
};

template <typename R, int NMAX>
__global__ void traj_kernel(TrajParams<R> p) {
  if (p.skip && *p.skip) return;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= p.B) return;
  const int n = p.n, m = p.m, s = n + m, T = p.T;
  const size_t tb = (size_t)p.B;
  R tau[NMAX], xn[NMAX];
  for (int i = 0; i < n; ++i) tau[i] = p.x0[(size_t)e * n + i];
  for (int t = 0; t < T; ++t) {
    const size_t idx = (size_t)t * tb + e;
    for (int i = 0; i < n; ++i) p.x[idx * n + i] = tau[i];
    if (t == T - 1) break;
    for (int j = 0; j < m; ++j) tau[n + j] = p.u[idx * m + j];
    if (p.dynamics == DMPC_DYN_LINEAR) {
      const R* Ft = p.F + idx * n * s;
      for (int i = 0; i < n; ++i) xn[i] = dot2(Ft + i * s, 1, tau, s, p.f ? p.f[idx * n + i] : R(0));
    } else {
      pendulum_step(p.dyn_params, tau, tau[n], xn);
      if (p.Fout) {
        R Fl[12], fl[3];
        pendulum_jacobian(p.dyn_params, tau, xn, Fl, fl);
        R* Fo = p.Fout + idx * 12; R* fo = p.fout + idx * 3;
        for (int i = 0; i < 12; ++i) Fo[i] = Fl[i];
        for (int i = 0; i < 3; ++i) fo[i] = fl[i];
      }
    }
    for (int i = 0; i < n; ++i) tau[i] = xn[i];
  }
}

}  // namespace dmpc
