// Batched time-varying LQR on sm_100a: Riccati recursion + rollout, and the KKT adjoint.
//
//   lqr_solve_kernel   = LqrRecursion.backward + .forward     (reference lqr/lqr_recursion.py:69-200)
//                        MASKED variant = LQR_active           (reference mpc/active_constrained_lqr.py:67-193)
//   lqr_dtau_kernel    = the second LQR solve of DiffLqr.backward re-using the forward pass's
//                        factors (reference lqr/differentiable_lqr.py:106-112)
//   adjoint_out_kernel = lambda / d-lambda recursions + dC,dc,dF,df,dx0
//                        (reference lqr/differentiable_lqr.py:87-104,114-134; mpc/mpc_step.py:383-446)
//
// One group of G lanes owns one batch element for the whole horizon (common.cuh).
#pragma once
#include "common.cuh"

namespace dmpc {

enum LqrFlags : int {
  LQR_DO_FACTOR = 1,    // run the Riccati sweep (else Ks/ks are inputs)
  LQR_DO_ROLLOUT = 2,   // run the forward rollout
  LQR_SAVE_FAC = 4,     // write Quu^-1 and Qxu per (t,b) for lqr_dtau_kernel
  LQR_MASKED = 8,       // LQR_active semantics with `active` mask
};

enum AdjFlags : int {
  ADJ_QUIRK_DC = 1,     // dC = 0.5*(dtau x tau) + (tau x dtau)      (differentiable_lqr.py:128)
  ADJ_QUIRK_DF = 2,     // df[t] = dlambda[t] instead of dlambda[t+1] (differentiable_lqr.py:133)
  ADJ_NEGATE = 4,       // MPCstep.backward sign convention (mpc_step.py:387-446)
  ADJ_NEG_RHS = 8,      // dlambda uses -d_taus_x as rhs (mpc_step.py:417)
  ADJ_REDUCE_TB = 16,   // do not materialise dC,dc,dF,df: sum them over t in shared memory and emit one partial
                        // record per element (backward of util.expand_time_batch, util.py:361-377, fused in)
};

template <typename R>
struct LqrParams {
  int T, B, n, m, flags;
  const R* x0;   // [B,n]
  const R* C;    // [T,B,s,s]
  const R* c;    // [T,B,s]   (or nullptr -> split form cx|cu below)
  const R* cx;   // [T,B,n] or nullptr (zeros)   -- used when c == nullptr
  const R* cu;   // [T,B,m] or nullptr (zeros)
  const R* F;    // [>=T-1,B,n,s]
  const R* f;    // [T-1,B,n] or nullptr
  const unsigned char* active;  // [T,B,m] (MASKED) or nullptr
  R c_scale;     // c is multiplied by this on load (MPC adjoint passes -1 with c := d_taus)
  R* x;          // [T,B,n]
  R* u;          // [T,B,m]
  R* Ks;         // [T,B,m,n]
  R* ks;         // [T,B,m]
  R* fac;        // [T,B,m*m + n*m]  (Quu^-1 | Qxu) or nullptr
  R* tau_out;    // [T,B,s] or nullptr: rollout also writes [x;u] concatenated
  R* Vsave;      // [T,B,n*n+n] or nullptr: V_t | v_t of the Riccati sweep (t >= 1) for adjoint_fused_kernel
  const int* skip;  // large-system Q / V steps only (device flag, nullable): non-zero -> the launch is a no-op
};

// shared-memory layout of one element's region for lqr_solve_kernel (offsets in reals)
struct LqrLayout {
  int oC, oc, oF, of_, stage;   // stage-relative offsets, stage size
  int st0, st1;                 // the two stages
  int Q, q, V, v, Mx, mv, H, Rhs, ldr, P, xcur, piv, total, stride;
};

// compact = rollout-only launch: the stage holds K_t (m*n) in the C slot and no Riccati work buffers
template <typename R>
__host__ __device__ inline LqrLayout lqr_layout(int n, int m, bool save_fac, bool compact = false) {
  const int W = 16 / (int)sizeof(R);
  const int s = n + m;
  LqrLayout L;
  int o = 0;
  L.oC = o; o += rup(compact ? m * n : s * s, W);
  L.oc = o; o += rup(s, W);
  L.oF = o; o += rup(n * s, W);
  L.of_ = o; o += rup(n, W);
  L.stage = o;
  o = 0;
  L.st0 = o; o += L.stage;
  L.st1 = o; o += L.stage;
  L.ldr = n + 1 + (save_fac ? m : 0);
  if (compact) {
    L.Q = L.q = L.V = L.v = L.Mx = L.H = L.Rhs = L.P = 0;
  } else {
    L.Q = o; o += rup(s * s, W);
    L.q = o; o += rup(s, W);
    L.V = o; o += rup(n * n, W);
    L.v = o; o += rup(n, W);
    L.Mx = o; o += rup(n * s, W);
    L.H = o; o += rup(m * m, W);
    L.Rhs = o; o += rup(m * L.ldr, W);
    L.P = o; o += rup(m * (n + 1), W);
  }
  L.mv = o; o += rup(n, W);
  L.xcur = o; o += rup(s, W);
  L.piv = o; o += rup((m * (int)sizeof(int) + (int)sizeof(R) - 1) / (int)sizeof(R), W);
  L.total = o;
  // stride == W (mod 128 bytes) so that same-offset accesses of neighbouring groups hit distinct banks
  const int line = 128 / (int)sizeof(R);
  L.stride = rup(o, line) + W;
  return L;
}

template <typename R, int N, int M, int G>
__global__ void lqr_solve_kernel(LqrParams<R> p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int n = N > 0 ? N : p.n;
  const int m = M > 0 ? M : p.m;
  const int s = n + m;
  const int T = p.T, B = p.B;
  constexpr int MMAX = M > 0 ? M : 32;
  const Grp<G> g;
  const int epb = (G <= 32) ? (blockDim.x / G) : 1;
  const int eloc = (G <= 32) ? (threadIdx.x / G) : 0;
  int e = blockIdx.x * epb + eloc;
  const bool valid = e < B;
  if (!valid) e = B - 1;
  const bool save_fac = (p.flags & LQR_SAVE_FAC) != 0;
  const bool masked = (p.flags & LQR_MASKED) != 0;
  const LqrLayout L = lqr_layout<R>(n, m, save_fac, !(p.flags & LQR_DO_FACTOR));
  R* sm = reinterpret_cast<R*>(smem_raw) + (size_t)eloc * L.stride;
  R* Q = sm + L.Q; R* q = sm + L.q; R* V = sm + L.V; R* v = sm + L.v;
  R* Mx = sm + L.Mx; R* mv = sm + L.mv; R* H = sm + L.H; R* Rhs = sm + L.Rhs; R* P = sm + L.P;
  R* xcur = sm + L.xcur;
  int* piv = reinterpret_cast<int*>(sm + L.piv);
  const int ldr = L.ldr;
  const size_t tb = (size_t)B;

  if (p.flags & LQR_DO_FACTOR) {
    auto load_tiles = [&](int t, int st) {
      R* base = sm + (st ? L.st1 : L.st0);
      const size_t idx = (size_t)t * tb + e;
      g_cp_async(g, base + L.oC, p.C + idx * s * s, s * s);
      if (p.c) {
        g_cp_async(g, base + L.oc, p.c + idx * s, s);
      } else {
        if (p.cx) g_cp_async(g, base + L.oc, p.cx + idx * n, n);
        else for (int o = g.lane; o < n; o += G) base[L.oc + o] = R(0);
        if (p.cu) g_cp_async(g, base + L.oc + n, p.cu + idx * m, m);
        else for (int o = g.lane; o < m; o += G) base[L.oc + n + o] = R(0);
      }
      if (t < T - 1) {
        g_cp_async(g, base + L.oF, p.F + idx * n * s, n * s);
        if (p.f) g_cp_async(g, base + L.of_, p.f + idx * n, n);
      }
      cp_async_commit();
    };
    load_tiles(T - 1, 0);
    int st = 0;
    for (int t = T - 1; t >= 0; --t) {
      if (t > 0) { load_tiles(t - 1, st ^ 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
      g.sync();
      const R* base = sm + (st ? L.st1 : L.st0);
      const R* Ct = base + L.oC; const R* ct = base + L.oc; const R* Ft = base + L.oF; const R* ft = base + L.of_;
      const R cs = p.c_scale;
      if (t == T - 1) {
        for (int o = g.lane; o < s * s; o += G) Q[o] = Ct[o];
        for (int o = g.lane; o < s; o += G) q[o] = cs * ct[o];
      } else {
        // Mx = V F ; mv = V f + v
        g_gemm(g, n, s, n, Mx, s, (const R*)nullptr, 0, V, n, 1, Ft, s, 1);
        if (p.f) g_gemm(g, n, 1, n, mv, 1, v, 1, V, n, 1, ft, 1, 1);
        else for (int o = g.lane; o < n; o += G) mv[o] = v[o];
        g.sync();
        // Q = C + F^T Mx ; q = c + F^T mv
        g_gemm(g, s, s, n, Q, s, Ct, s, Ft, 1, s, Mx, s, 1);
        for (int o = g.lane; o < s; o += G) {
          R a = cs * ct[o];
          for (int k = 0; k < n; ++k) a += Ft[k * s + o] * mv[k];
          q[o] = a;
        }
      }
      g.sync();
      // H = Quu (masked), Rhs = -[Qux | qu | (I)]
      const unsigned char* act = masked ? (p.active + ((size_t)t * tb + e) * m) : nullptr;
      for (int o = g.lane; o < m * m; o += G) {
        const int i = o / m, j = o - i * m;
        R hv = Q[(n + i) * s + n + j];
        if (masked) {
          const bool ai = act[i] != 0, aj = act[j] != 0;
          if (ai || aj) hv = R(0);
          if (ai && i == j) hv += R(1e-8);     // active_constrained_lqr.py:121-122
        }
        H[o] = hv;
      }
      for (int o = g.lane; o < m * ldr; o += G) {
        const int i = o / ldr, j = o - i * ldr;
        R rv;
        if (j < n) rv = -Q[(n + i) * s + j];
        else if (j == n) rv = -q[n + i];
        else rv = (j - n - 1 == i) ? R(1) : R(0);
        if (masked && j <= n && act[i]) rv = R(0);
        Rhs[o] = rv;
      }
      g.sync();
      g_lu_factor<G, MMAX>(g, m, H, m, Rhs, ldr, ldr, (int*)nullptr);
      g_back_subst(g, m, H, m, Rhs, ldr, ldr);
      g.sync();
      // Rhs[:, :n] = K, Rhs[:, n] = k, Rhs[:, n+1:] = Quu^-1
      // P = [Qux | qu] + Quu [K | k]      (unmasked Quu, Qux: Q6)
      for (int o = g.lane; o < m * (n + 1); o += G) {
        const int i = o / (n + 1), j = o - i * (n + 1);
        R a = (j < n) ? Q[(n + i) * s + j] : q[n + i];
        for (int l = 0; l < m; ++l) a += Q[(n + i) * s + n + l] * Rhs[l * ldr + j];
        P[o] = a;
      }
      // write gains (and factors) while P settles
      {
        const size_t idx = (size_t)t * tb + e;
        if (valid) {
          R* Kg = p.Ks + idx * m * n; R* kg = p.ks + idx * m;
          for (int o = g.lane; o < m * n; o += G) { const int i = o / n, j = o - i * n; Kg[o] = Rhs[i * ldr + j]; }
          for (int o = g.lane; o < m; o += G) kg[o] = Rhs[o * ldr + n];
          if (save_fac && p.fac) {
            R* fg = p.fac + idx * (m * m + n * m);
            for (int o = g.lane; o < m * m; o += G) { const int i = o / m, j = o - i * m; fg[o] = Rhs[i * ldr + n + 1 + j]; }
            for (int o = g.lane; o < n * m; o += G) { const int i = o / m, j = o - i * m; fg[m * m + o] = Q[i * s + n + j]; }
          }
        }
      }
      g.sync();
      // [V | v] = [Qxx | qx] + Qxu [K | k] + K^T P
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
          if (p.Vsave && valid) p.Vsave[((size_t)t * tb + e) * (n * n + n) + (j < n ? i * n + j : n * n + i)] = a + b;
        }
      }
      g.sync();
      st ^= 1;
    }
  }

  if (p.flags & LQR_DO_ROLLOUT) {
    // stage tiles re-used: K_t (m*n) -> oC slot, k_t -> oc slot, F_t, f_t
    auto load_tiles = [&](int t, int st) {
      R* base = sm + (st ? L.st1 : L.st0);
      const size_t idx = (size_t)t * tb + e;
      g_cp_async(g, base + L.oC, p.Ks + idx * m * n, m * n);
      g_cp_async(g, base + L.oc, p.ks + idx * m, m);
      if (t < T - 1) {
        g_cp_async(g, base + L.oF, p.F + idx * n * s, n * s);
        if (p.f) g_cp_async(g, base + L.of_, p.f + idx * n, n);
      }
      cp_async_commit();
    };
    g.sync();
    load_tiles(0, 0);
    for (int o = g.lane; o < n; o += G) xcur[o] = p.x0[(size_t)e * n + o];
    int st = 0;
    for (int t = 0; t < T; ++t) {
      if (t < T - 1) { load_tiles(t + 1, st ^ 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
      g.sync();
      const R* base = sm + (st ? L.st1 : L.st0);
      const R* Kt = base + L.oC; const R* kt = base + L.oc; const R* Ft = base + L.oF; const R* ft = base + L.of_;
      const unsigned char* act = masked ? (p.active + ((size_t)t * tb + e) * m) : nullptr;
      for (int o = g.lane; o < m; o += G) {
        R uv = dot_rot(Kt + o * n, xcur, n, o, kt[o]);
        if (masked && act[o]) uv = R(0);      // active_constrained_lqr.py:175
        xcur[n + o] = uv;
      }
      g.sync();
      {
        const size_t idx = (size_t)t * tb + e;
        if (valid) {
          if (p.x) for (int o = g.lane; o < n; o += G) p.x[idx * n + o] = xcur[o];
          if (p.u) for (int o = g.lane; o < m; o += G) p.u[idx * m + o] = xcur[n + o];
          if (p.tau_out) for (int o = g.lane; o < s; o += G) p.tau_out[idx * s + o] = xcur[o];
        }
      }
      if (t < T - 1) {
        // x' = F [x;u] + f  -> into mv then copy
        for (int o = g.lane; o < n; o += G) mv[o] = dot_rot(Ft + o * s, xcur, s, o, p.f ? ft[o] : R(0));
        g.sync();
        for (int o = g.lane; o < n; o += G) xcur[o] = mv[o];
      }
      g.sync();
      st ^= 1;
    }
  }
}

// ------------------------------------------------------------------------------------------
// Second LQR solve of DiffLqr.backward with saved factors:
//   backward in t:  q = drl_t + F_t^T v'_{t+1};  k'_t = -Quu^-1 q_u;  v'_t = q_x + Qxu k'_t
//   forward  in t:  du_t = K_t dx_t + k'_t;  dx_{t+1} = F_t [dx_t; du_t]
// (K^T(q_u + Quu k') vanishes identically for the exact Newton gain, see DESIGN.md §4.2.)
// dtau is written to `dc` ([T,B,s]); k'_t is parked in dc[t,b,n:] between the sweeps.
template <typename R>
struct DtauParams {
  int T, B, n, m;
  const R* F;    // [>=T-1,B,n,s]
  const R* gx;   // [T,B,n]
  const R* gu;   // [T,B,m]
  const R* Ks;   // [T,B,m,n]
  const R* fac;  // [T,B,m*m+n*m]
  R* dc;         // [T,B,s]  out: dtau
  R* vp;         // FUSED: [T-1,B,n] out: v'_t for t >= 1 at row t-1 (the caller parks it in the df output buffer);
                 //        nullptr -> v'_t goes to dc[t,b,:n] instead (the fused-reduction adjoint, where dc is a workspace)
  R* dx0;        // FUSED: [B,n] out: v'_0 = dlambda_0
};

struct DtauLayout { int oF, oA, oB, og, stage, st0, st1, q, vp, kp, dx, tmp, total, stride; };

template <typename R>
__host__ __device__ inline DtauLayout dtau_layout(int n, int m) {
  const int W = 16 / (int)sizeof(R);
  const int s = n + m;
  DtauLayout L;
  int o = 0;
  L.oF = o; o += rup(n * s, W);
  L.oA = o; o += rup(m * m + n * m, W);     // sweep1: fac ; sweep2: K (m*n <= m*m+n*m)
  L.oB = o; o += rup(s, W);                  // sweep1: gx|gu staged separately (n, then m)
  L.og = o; o += rup(s, W);
  L.stage = o;
  o = 0;
  L.st0 = o; o += L.stage;
  L.st1 = o; o += L.stage;
  L.q = o; o += rup(s, W);
  L.vp = o; o += rup(n, W);
  L.kp = o; o += rup(m, W);
  L.dx = o; o += rup(s, W);
  L.tmp = o; o += rup(n, W);
  L.total = o;
  const int line = 128 / (int)sizeof(R);
  L.stride = rup(o, line) + W;
  return L;
}

// FUSED = sweep 1 only, for adjoint_fused_kernel (lqr_adjoint_fused.cuh): also emits v'_t.
template <typename R, int N, int M, int G, bool FUSED = false>
__global__ void lqr_dtau_kernel(DtauParams<R> p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int n = N > 0 ? N : p.n;
  const int m = M > 0 ? M : p.m;
  const int s = n + m;
  const int T = p.T, B = p.B;
  const Grp<G> g;
  const int epb = (G <= 32) ? (blockDim.x / G) : 1;
  const int eloc = (G <= 32) ? (threadIdx.x / G) : 0;
  int e = blockIdx.x * epb + eloc;
  const bool valid = e < B;
  if (!valid) e = B - 1;
  const DtauLayout L = dtau_layout<R>(n, m);
  R* sm = reinterpret_cast<R*>(smem_raw) + (size_t)eloc * L.stride;
  R* q = sm + L.q; R* vp = sm + L.vp; R* kp = sm + L.kp; R* dx = sm + L.dx; R* tmp = sm + L.tmp;
  const size_t tb = (size_t)B;
  const int fsz = m * m + n * m;

  // ---- sweep 1 (t = T-1 .. 0)
  {
    auto load_tiles = [&](int t, int st) {
      R* base = sm + (st ? L.st1 : L.st0);
      const size_t idx = (size_t)t * tb + e;
      if (t < T - 1) g_cp_async(g, base + L.oF, p.F + idx * n * s, n * s);
      g_cp_async(g, base + L.oA, p.fac + idx * fsz, fsz);
      g_cp_async(g, base + L.oB, p.gx + idx * n, n);
      g_cp_async(g, base + L.og, p.gu + idx * m, m);
      cp_async_commit();
    };
    load_tiles(T - 1, 0);
    int st = 0;
    for (int t = T - 1; t >= 0; --t) {
      if (t > 0) { load_tiles(t - 1, st ^ 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
      g.sync();
      const R* base = sm + (st ? L.st1 : L.st0);
      const R* Ft = base + L.oF; const R* Qi = base + L.oA; const R* Qxu = base + L.oA + m * m;
      const R* gxt = base + L.oB; const R* gut = base + L.og;
      for (int o = g.lane; o < s; o += G) {
        R a0 = (o < n) ? gxt[o] : gut[o - n], a1 = R(0);
        if (t < T - 1) {
          int k = 0;
          for (; k + 1 < n; k += 2) { a0 += Ft[k * s + o] * vp[k]; a1 += Ft[(k + 1) * s + o] * vp[k + 1]; }
          if (k < n) a0 += Ft[k * s + o] * vp[k];
        }
        q[o] = a0 + a1;
      }
      g.sync();
      for (int o = g.lane; o < m; o += G) {
        kp[o] = -dot_rot(Qi + o * m, q + n, m, o, R(0));
      }
      g.sync();
      for (int o = g.lane; o < n; o += G) {
        vp[o] = dot_rot(Qxu + o * m, kp, m, o, q[o]);
      }
      if (valid) for (int o = g.lane; o < m; o += G) p.dc[((size_t)t * tb + e) * s + n + o] = kp[o];
      g.sync();
      if (FUSED && valid) {
        R* dst = t == 0 ? p.dx0 + (size_t)e * n : (p.vp ? p.vp + ((size_t)(t - 1) * tb + e) * n : p.dc + ((size_t)t * tb + e) * s);
        for (int o = g.lane; o < n; o += G) dst[o] = vp[o];
      }
      st ^= 1;
    }
  }
  if (FUSED) return;
  // ---- sweep 2 (t = 0 .. T-1)
  {
    auto load_tiles = [&](int t, int st) {
      R* base = sm + (st ? L.st1 : L.st0);
      const size_t idx = (size_t)t * tb + e;
      if (t < T - 1) g_cp_async(g, base + L.oF, p.F + idx * n * s, n * s);
      g_cp_async(g, base + L.oA, p.Ks + idx * m * n, m * n);
      g_cp_async(g, base + L.og, p.dc + idx * s + n, m);
      cp_async_commit();
    };
    g.sync();
    load_tiles(0, 0);
    for (int o = g.lane; o < n; o += G) dx[o] = R(0);
    int st = 0;
    for (int t = 0; t < T; ++t) {
      if (t < T - 1) { load_tiles(t + 1, st ^ 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
      g.sync();
      const R* base = sm + (st ? L.st1 : L.st0);
      const R* Ft = base + L.oF; const R* Kt = base + L.oA; const R* kpt = base + L.og;
      for (int o = g.lane; o < m; o += G) dx[n + o] = dot_rot(Kt + o * n, dx, n, o, kpt[o]);
      g.sync();
      if (valid) for (int o = g.lane; o < s; o += G) p.dc[((size_t)t * tb + e) * s + o] = dx[o];
      if (t < T - 1) {
        for (int o = g.lane; o < n; o += G) tmp[o] = dot_rot(Ft + o * s, dx, s, o, R(0));
        g.sync();
        for (int o = g.lane; o < n; o += G) dx[o] = tmp[o];
      }
      g.sync();
      st ^= 1;
    }
  }
}

// ------------------------------------------------------------------------------------------
// lambda / d-lambda recursions and the gradient outer products.
template <typename R>
struct AdjOutParams {
  int T, B, n, m, F_T, flags;
  const R* C; const R* c; const R* F;
  const R* x; const R* u;      // tau
  const R* dtau;               // [T,B,s] (may alias dc when !ADJ_NEGATE)
  const R* gx; const R* gu;    // upstream grads (nullable -> zeros)
  R* dx0; R* dC; R* dc; R* dF; R* df;   // df nullable
  R* red;                      // ADJ_REDUCE_TB: [B][s*s + s + n*s + n] per-element sums over t (dC | dc | dF | df)
};

struct AdjLayout { int oC, oc, oF, otau, odtau, og, stage, st0, st1, lam, dlam, lamn, dlamn, red, total, stride; };

__host__ __device__ inline int adj_red_elems(int n, int m) { const int s = n + m; return s * s + s + n * s + n; }

template <typename R>
__host__ __device__ inline AdjLayout adj_layout(int n, int m, bool reduce = false) {
  const int W = 16 / (int)sizeof(R);
  const int s = n + m;
  AdjLayout L;
  int o = 0;
  L.oC = o; o += rup(n * s, W);
  L.oc = o; o += rup(s, W);
  L.oF = o; o += rup(n * s, W);
  L.otau = o; o += rup(n, W) + rup(m, W);
  L.odtau = o; o += rup(s, W);
  L.og = o; o += rup(n, W);
  L.stage = o;
  o = 0;
  L.st0 = o; o += L.stage;
  L.st1 = o; o += L.stage;
  L.lam = o; o += rup(n, W);
  L.dlam = o; o += rup(n, W);
  L.lamn = o; o += rup(n, W);
  L.dlamn = o; o += rup(n, W);
  L.red = o; if (reduce) o += rup(adj_red_elems(n, m), W);
  L.total = o;
  const int line = 128 / (int)sizeof(R);
  L.stride = rup(o, line) + W;
  return L;
}

template <typename R, int N, int M, int G, bool RED = false>
__global__ void adjoint_out_kernel(AdjOutParams<R> p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int n = N > 0 ? N : p.n;
  const int m = M > 0 ? M : p.m;
  const int s = n + m;
  const int T = p.T, B = p.B;
  const Grp<G> g;
  const int epb = (G <= 32) ? (blockDim.x / G) : 1;
  const int eloc = (G <= 32) ? (threadIdx.x / G) : 0;
  int e = blockIdx.x * epb + eloc;
  const bool valid = e < B;
  if (!valid) e = B - 1;
  constexpr bool reduce = RED;                 // ADJ_REDUCE_TB is a separate instantiation (register budget)
  const AdjLayout L = adj_layout<R>(n, m, reduce && N == 0);
  R* sm = reinterpret_cast<R*>(smem_raw) + (size_t)eloc * L.stride;
  R* lam = sm + L.lam; R* dlam = sm + L.dlam; R* lamn = sm + L.lamn; R* dlamn = sm + L.dlamn;
  // ADJ_REDUCE_TB accumulators: every output (i,j) is owned by one lane for the whole horizon, so compile-time
  // shapes keep the running sums in registers (acc*[k] <-> o = lane + k G); runtime shapes keep them in shared memory
  constexpr bool REG = RED && N > 0;
  constexpr int S_ = N + M;
  // outer products in the REG path: lane = (row group ti, column tj); the lane keeps tau_j, dtau_j in registers and
  // walks the rows ti, ti + NR, ... whose tau_i / dtau_i / lambda_i loads are warp broadcasts - two shared-memory
  // loads per output instead of four and no index arithmetic
  constexpr int NR = REG ? (G / S_ > 0 ? G / S_ : 1) : 1;
  constexpr int KC = REG ? (S_ + NR - 1) / NR : 1, KF = REG ? (N + NR - 1) / NR : 1,
                Kc = REG ? (S_ + G - 1) / G : 1, Kf = REG ? (N + G - 1) / G : 1;
  static_assert(!REG || G >= S_, "REG path: one column per lane");
  const int tj = REG ? g.lane % S_ : 0, ti = REG ? g.lane / S_ : 0;
  const bool tile_lane = ti < NR;
  R accC[KC], accF[KF], accc[Kc], accf[Kf];
#pragma unroll
  for (int k = 0; k < KC; ++k) accC[k] = R(0);
#pragma unroll
  for (int k = 0; k < KF; ++k) accF[k] = R(0);
#pragma unroll
  for (int k = 0; k < Kc; ++k) accc[k] = R(0);
#pragma unroll
  for (int k = 0; k < Kf; ++k) accf[k] = R(0);
  R* rC = sm + L.red; R* rc = rC + s * s; R* rF = rc + s; R* rf = rF + n * s;     // per-element sums over t
  if (reduce && !REG) for (int o = g.lane; o < adj_red_elems(n, m); o += G) rC[o] = R(0);
  const size_t tb = (size_t)B;
  const int nxoff = rup(n, 16 / (int)sizeof(R));
  const bool neg = (p.flags & ADJ_NEGATE) != 0;
  const R sgn = neg ? R(-1) : R(1);
  const R rsgn = (p.flags & ADJ_NEG_RHS) ? R(-1) : R(1);

  auto load_tiles = [&](int t, int st) {
    R* base = sm + (st ? L.st1 : L.st0);
    const size_t idx = (size_t)t * tb + e;
    g_cp_async(g, base + L.oC, p.C + idx * s * s, n * s);        // top n rows of C_t
    g_cp_async(g, base + L.oc, p.c + idx * s, n);
    if (t < T - 1) g_cp_async(g, base + L.oF, p.F + idx * n * s, n * s);
    g_cp_async(g, base + L.otau, p.x + idx * n, n);
    g_cp_async(g, base + L.otau + nxoff, p.u + idx * m, m);
    g_cp_async(g, base + L.odtau, p.dtau + idx * s, s);
    if (p.gx) g_cp_async(g, base + L.og, p.gx + idx * n, n);
    cp_async_commit();
  };
  load_tiles(T - 1, 0);
  int st = 0;
  for (int t = T - 1; t >= 0; --t) {
    if (t > 0) { load_tiles(t - 1, st ^ 1); cp_async_wait<1>(); } else { cp_async_wait<0>(); }
    g.sync();
    const R* base = sm + (st ? L.st1 : L.st0);
    const R* Ct = base + L.oC; const R* ct = base + L.oc; const R* Ft = base + L.oF;
    const R* xt = base + L.otau; const R* ut = base + L.otau + nxoff;
    const R* dt = base + L.odtau; const R* gxt = base + L.og;
    auto tau = [&](int j) -> R { return j < n ? xt[j] : ut[j - n]; };
    const size_t idx = (size_t)t * tb + e;
    // dF_t = dlam_{t+1} (x) tau_t + lam_{t+1} (x) dtau_t      (t < T-1)
    if (t < T - 1 && valid) {
      R* dFg = p.dF + idx * n * s;
      auto dF_val = [&](int o) -> R { const int i = o / s, j = o - i * s; return sgn * (dlam[i] * tau(j) + lam[i] * dt[j]); };
      if (reduce && REG) {
        if (tile_lane) {
          const R tau_j = tau(tj), dt_j = dt[tj];
#pragma unroll
          for (int k = 0; k < KF; ++k) { const int i = ti + k * NR; if (i < n) accF[k] += sgn * (dlam[i] * tau_j + lam[i] * dt_j); }
        }
      } else {
        for (int o = g.lane; o < n * s; o += G) { const R v = dF_val(o); if (reduce) rF[o] += v; else dFg[o] = v; }
      }
      if (!(p.flags & ADJ_QUIRK_DF)) {
        if (reduce && REG) {
#pragma unroll
          for (int k = 0; k < Kf; ++k) { const int o = g.lane + k * G; if (o < n) accf[k] += sgn * dlam[o]; }
        } else if (reduce) { for (int o = g.lane; o < n; o += G) rf[o] += sgn * dlam[o]; }
        else if (p.df) { for (int o = g.lane; o < n; o += G) p.df[idx * n + o] = sgn * dlam[o]; }
      }
    }
    // lam_t, dlam_t
    for (int o = g.lane; o < 2 * n; o += G) {
      const bool isd = o >= n;
      const int i = isd ? o - n : o;
      R a0, a1 = R(0);
      if (isd) a0 = p.gx ? rsgn * gxt[i] : R(0); else a0 = ct[i];
      const R* ln = isd ? dlam : lam;
      if (isd) { a0 = dot_rot(Ct + i * s, dt, s, i, a0); }
      else     { int j = i % s; for (int c = 0; c < s; ++c) { a0 += Ct[i * s + j] * tau(j); if (++j == s) j = 0; } }
      if (t < T - 1) for (int k = 0; k < n; ++k) a1 += Ft[k * s + i] * ln[k];
      (isd ? dlamn : lamn)[i] = a0 + a1;
    }
    // dC_t, dc_t
    if (valid) {
      R* dCg = p.dC + idx * s * s;
      const bool quirk = (p.flags & ADJ_QUIRK_DC) != 0;
      auto dC_val = [&](int o) -> R {
        const int i = o / s, j = o - i * s;
        const R a = dt[i] * tau(j), b = tau(i) * dt[j];
        return quirk ? (R(0.5) * a + b) : (sgn * R(0.5) * (a + b));
      };
      if (reduce && REG) {
        if (tile_lane) {
          const R tau_j = tau(tj), dt_j = dt[tj];
#pragma unroll
          for (int k = 0; k < KC; ++k) {
            const int i = ti + k * NR;
            if (i < s) { const R a = dt[i] * tau_j, b = tau(i) * dt_j; accC[k] += quirk ? (R(0.5) * a + b) : (sgn * R(0.5) * (a + b)); }
          }
        }
#pragma unroll
        for (int k = 0; k < Kc; ++k) { const int o = g.lane + k * G; if (o < s) accc[k] += sgn * dt[o]; }
      } else {
        for (int o = g.lane; o < s * s; o += G) { const R v = dC_val(o); if (reduce) rC[o] += v; else dCg[o] = v; }
      }
      if (reduce) { if (!REG) for (int o = g.lane; o < s; o += G) rc[o] += sgn * dt[o]; }
      else if (neg || p.dc != p.dtau) for (int o = g.lane; o < s; o += G) p.dc[idx * s + o] = sgn * dt[o];
    }
    g.sync();
    for (int o = g.lane; o < n; o += G) { lam[o] = lamn[o]; dlam[o] = dlamn[o]; }
    if (valid) {
      if ((p.flags & ADJ_QUIRK_DF) && t < T - 1) {
        if (reduce && REG) {
#pragma unroll
          for (int k = 0; k < Kf; ++k) { const int o = g.lane + k * G; if (o < n) accf[k] += sgn * dlamn[o]; }
        } else if (reduce) { for (int o = g.lane; o < n; o += G) rf[o] += sgn * dlamn[o]; }
        else if (p.df) { for (int o = g.lane; o < n; o += G) p.df[idx * n + o] = sgn * dlamn[o]; }
      }
      if (t == 0) for (int o = g.lane; o < n; o += G) p.dx0[(size_t)e * n + o] = sgn * dlamn[o];
    }
    g.sync();
    st ^= 1;
  }
  if (reduce) {   // every (i,j) is owned by one lane for the whole horizon: no barrier needed before the write-out
    if (valid) {
      const int rsz = adj_red_elems(n, m);
      R* out = p.red + (size_t)e * rsz;
      if (REG) {
        if (tile_lane) {
#pragma unroll
          for (int k = 0; k < KC; ++k) { const int i = ti + k * NR; if (i < s) out[i * s + tj] = accC[k]; }
#pragma unroll
          for (int k = 0; k < KF; ++k) { const int i = ti + k * NR; if (i < n) out[s * s + s + i * s + tj] = accF[k]; }
        }
#pragma unroll
        for (int k = 0; k < Kc; ++k) { const int o = g.lane + k * G; if (o < s) out[s * s + o] = accc[k]; }
#pragma unroll
        for (int k = 0; k < Kf; ++k) { const int o = g.lane + k * G; if (o < n) out[s * s + s + n * s + o] = accf[k]; }
      } else {
        for (int o = g.lane; o < rsz; o += G) out[o] = rC[o];
      }
    }
    return;
  }
  // zero-fill the T-th row of dF when F was given with T rows (Q8, mpc_step.py:428)
  if (p.F_T == T && valid) {
    R* dFg = p.dF + ((size_t)(T - 1) * tb + e) * n * s;
    for (int o = g.lane; o < n * s; o += G) dFg[o] = R(0);
  }
}

// util.expand_time_batch on the device (reference util.py:361-377): dst[t][b][:] = src[:] for a parameter block shared
// by every (t, b) - the forward half of the shared-parameter entry (LqrNet, MpcNet_dx, IL_Env.mpc broadcast n*s or 2*n_sc
// doubles over [T,B]); its backward is the fused (T,B)-sum of ADJ_REDUCE_TB.
template <typename R>
__global__ void expand_time_batch_kernel(const R* __restrict__ src, R* __restrict__ dst, int count, size_t total) {
  for (size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x; o < total; o += (size_t)gridDim.x * blockDim.x)
    dst[o] = src[o % count];
}

// Second stage of ADJ_REDUCE_TB: out[o] = sum_e red[e][o] in a fixed order (lane-strided partial sums, then a
// shuffle tree) - deterministic, unlike atomics.  One warp per output element: the lanes' loads are rsz elements apart,
// but neighbouring warps (outputs o, o+1, ...) read the same sectors at the same time and the L2 serves them - a variant
// with one warp per four consecutive outputs (whole-sector loads, a quarter of the warps) measured 2.4x SLOWER at
// rsz = 2952, B = 8192 (79 vs 33 us) and 3.6x slower at rsz = 35: the loop is latency bound and wants the warps.
template <typename R>
__global__ void reduce_partials_kernel(const R* red, int B, int rsz, R* out) {
  const int o = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (o >= rsz) return;
  const int lane = threadIdx.x & 31;
  R a0 = R(0), a1 = R(0);
  int e = lane;
  for (; e + 32 < B; e += 64) { a0 += red[(size_t)e * rsz + o]; a1 += red[(size_t)(e + 32) * rsz + o]; }
  if (e < B) a0 += red[(size_t)e * rsz + o];
  R a = a0 + a1;
  for (int d = 16; d > 0; d >>= 1) a += __shfl_xor_sync(0xffffffffu, a, d);
  if (lane == 0) out[o] = a;
}

}  // namespace dmpc
