// LqrRecursion.backward + .forward (reference lqr/lqr_recursion.py:69-200) and LQR_active (reference
// mpc/active_constrained_lqr.py:67-193) for SMALL systems - s = n + m <= 6: the pendulum / Boyd / LQRnet shape (3,1), the
// one-variable example (2,1) and BASELINE config 2 (4,2) - with ONE THREAD per batch element and the whole recursion in
// registers.
//
// Why: lqr_solve_kernel gives such an element a group of 4-8 lanes that exchange every intermediate through shared
// memory, with seven group barriers and a generic LU per time step; at s = 6 a Riccati step is ~700 flops, and the group
// kernel spends ~7900 cycles on it (profiles/r2/r2y_bench_c2.json: 0.201 ms for T = 50) - dependent-chain latency, not
// bandwidth (7 % of HBM).  A thread that owns the element needs no barrier and its m <= 2 elimination is a handful of
// FMAs; shared memory only stages the operands (below).  Same contract as lqr_solve_kernel (LqrParams, every flag); pivoting as there (first maximum
// wins), the pivots enter through their reciprocals.
#pragma once
#include "lqr_kernels.cuh"

namespace dmpc {

// in-register pivoted Gaussian elimination H X = Rhs (H: M x M, Rhs: M x NC), M <= 2; X overwrites Rhs
template <typename R, int M, int NC>
__device__ __forceinline__ void tpe_solve(R (&H)[M][M], R (&X)[M][NC]) {
  if constexpr (M == 2) {
    if (fabs(H[1][0]) > fabs(H[0][0])) {                     // first maximum wins (LAPACK idamax)
#pragma unroll
      for (int j = 0; j < 2; ++j) { const R t = H[0][j]; H[0][j] = H[1][j]; H[1][j] = t; }
#pragma unroll
      for (int j = 0; j < NC; ++j) { const R t = X[0][j]; X[0][j] = X[1][j]; X[1][j] = t; }
    }
    // two reciprocals per step instead of a guarded division per column and row (fourteen at n = 4, m = 2, each with a
    // branch around its slow path that keeps the compiler from interleaving them)
    const R r0 = R(1) / H[0][0];
    const R l = H[1][0] * r0;
    const R r1 = R(1) / (H[1][1] - l * H[0][1]);
#pragma unroll
    for (int j = 0; j < NC; ++j) {
      X[1][j] = (X[1][j] - l * X[0][j]) * r1;
      X[0][j] = (X[0][j] - H[0][1] * X[1][j]) * r0;
    }
  } else {
    static_assert(M == 1, "tpe_solve: m <= 2");
    const R r0 = R(1) / H[0][0];                             // lqr_recursion.py:112-115 takes the scalar reciprocal too
#pragma unroll
    for (int j = 0; j < NC; ++j) X[0][j] *= r0;
  }
}

// Operand staging.  Elements e0 .. e0+31 of one time step are CONTIGUOUS in the reference layout ([T][B][...]), but a
// thread that loads its own element directly touches a different 128-byte line than its neighbour: every LDG is 32
// separate L1 requests (measured: the first version of this kernel, direct loads + L2 prefetch, 0.247 ms against the group
// kernel's 0.259 ms at config 2).  So the WARP copies the step's operands of its elements with coalesced cp.async into a
// ring of shared-memory stages (one slot per element, odd stride: conflict-free reads), one step ahead in the Riccati
// sweep and two in the rollout.
//
// Elements per warp (epw, a launch argument; 32 by default).  At config 2 the kernel's duration is ONE warp's serial
// instruction stream (ncu, profiles/r2/r2an_c2_tpe.summary.txt: 1670 instructions per Riccati step at one issue every
// 3.2 cycles, `wait` the top stall, DRAM at 15 %, 1.6 % of the warp slots in use), and ~30 % of that stream is this
// staging.  A batch that leaves most of the GPU's 592 warp schedulers idle anyway can be spread thinner - 16 or 8 elements
// per warp, the other lanes shadow the last element - so that each warp stages half or a quarter as much; the recursion's
// own instructions do not shrink, so the gain is bounded by ~1.3x.  Opt-in (DMPC_LQR_TPE_EPW, lqr_launch.cu): checked
// against the oracle by tests/test_gpu_dispatch_matrix.py, not yet timed.
template <typename R>
__device__ __forceinline__ void tpe_cp(R* sdst, const R* g) {
  if (sizeof(R) == 8) cp_async8(sdst, g); else cp_async4(sdst, g);
}
// CNT reals per element for `nv` consecutive elements -> slot[le * stride + off + j].  Full warps (nv == 32) take the
// unrolled path: the (element, item) pair of a lane's i-th copy advances by compile-time constants, no division.
template <int CNT, typename R>
__device__ __forceinline__ void tpe_stage(R* dst, int stride, int off, const R* src, int nv, int lane) {
  if (nv == 32) {
    constexpr int Q32 = 32 / CNT, R32 = 32 % CNT;
    int j = lane % CNT;
    int d = (lane / CNT) * stride + off + j;
#pragma unroll
    for (int it = 0; it < CNT; ++it) {
      tpe_cp(dst + d, src + lane + 32 * it);
      j += R32; d += Q32 * stride + R32;
      if (j >= CNT) { j -= CNT; d += stride - CNT; }
    }
  } else {
    const int total = nv * CNT;
    for (int i = lane; i < total; i += 32) { const int le = i / CNT, j = i - le * CNT; tpe_cp(dst + le * stride + off + j, src + i); }
  }
}
// the same for element records that are GSTRIDE reals apart in global memory, of which the first CNT are wanted
template <int CNT, int GSTRIDE, typename R>
__device__ __forceinline__ void tpe_stage_rows(R* dst, int stride, int off, const R* src, int nv, int lane) {
  if (nv == 32) {
    constexpr int Q32 = 32 / CNT, R32 = 32 % CNT;
    int j = lane % CNT;
    int d = (lane / CNT) * stride + off + j;
    int g = (lane / CNT) * GSTRIDE + j;
#pragma unroll
    for (int it = 0; it < CNT; ++it) {
      tpe_cp(dst + d, src + g);
      j += R32; d += Q32 * stride + R32; g += Q32 * GSTRIDE + R32;
      if (j >= CNT) { j -= CNT; d += stride - CNT; g += GSTRIDE - CNT; }
    }
  } else {
    const int total = nv * CNT;
    for (int i = lane; i < total; i += 32) { const int le = i / CNT, j = i - le * CNT; tpe_cp(dst + le * stride + off + j, src + le * GSTRIDE + j); }
  }
}
template <typename R>
__device__ __forceinline__ void tpe_zero(R* dst, int stride, int off, int cnt, int nv, int lane) {
  const int total = nv * cnt;
  for (int i = lane; i < total; i += 32) { const int le = i / cnt, j = i - le * cnt; dst[le * stride + off + j] = R(0); }
}
__host__ __device__ constexpr int tpe_lqr_stride_f(int n, int m) { return ((n + m) * (n + m) + (n + m) + n * (n + m) + n) | 1; }
__host__ __device__ constexpr int tpe_lqr_stride_r(int n, int m) { return (m * n + m + n * (n + m) + n) | 1; }
// reals of shared memory per warp
// ring depths: DS stages in the Riccati sweep (DS - 1 steps ahead), DR in the rollout; shipped: 2 / 3, and 3 for the
// adjoint's solve below.  Deeper rings (4 / 8 / 8, for batches that leave each SM a single warp) were measured at config 2
// and are slower: forward 0.165 against 0.143 ms, adjoint solve 0.096 against 0.079 ms (gpurun_out r2al vs r2ak) - the
// longer prologue and the extra address arithmetic cost more than the exposed latency they remove.
__host__ __device__ constexpr int tpe_lqr_warp_reals(int n, int m, int ds, int dr) {
  return 32 * (ds * tpe_lqr_stride_f(n, m) > dr * tpe_lqr_stride_r(n, m) ? ds * tpe_lqr_stride_f(n, m) : dr * tpe_lqr_stride_r(n, m));
}

template <typename R, int N, int M, int TPB, int DS, int DR>
__global__ void __launch_bounds__(TPB) lqr_tpe_kernel(LqrParams<R> p, int epw) {
  constexpr int n = N, m = M, s = N + M, NC = N + 1 + M;
  constexpr int SF = tpe_lqr_stride_f(N, M), SR = tpe_lqr_stride_r(N, M);
  constexpr int oC = 0, oc = s * s, oF = s * s + s, of = s * s + s + n * s;      // sweep slot: C | c | F | f
  constexpr int rK = 0, rk = m * n, rF = m * n + m, rf = m * n + m + n * s;      // rollout slot: K | k | F | f
  static_assert(DS >= 2 && DR >= 2, "ring depths");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int T = p.T;
  const int lane = threadIdx.x & 31;
  const int e0 = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * epw;      // first element of this warp
  if (e0 >= p.B) return;                                                          // whole warp (only __syncwarp below)
  const int nv = p.B - e0 < epw ? p.B - e0 : epw;                                   // elements of this warp
  const bool valid = lane < nv;
  const int ls = valid ? lane : nv - 1;                                           // padding lanes shadow the last element
  const int e = e0 + ls;
  const size_t tb = (size_t)p.B;
  const bool masked = (p.flags & LQR_MASKED) != 0;
  const bool save_fac = (p.flags & LQR_SAVE_FAC) != 0 && p.fac != nullptr;
  const bool have_f = p.f != nullptr;
  R* wsm = reinterpret_cast<R*>(smem_raw) + (size_t)(threadIdx.x >> 5) * tpe_lqr_warp_reals(N, M, DS, DR);

  if (p.flags & LQR_DO_FACTOR) {
    const R cs = p.c_scale;
    auto issue = [&](int t, int slot) {
      R* st = wsm + slot * 32 * SF;
      const size_t i0 = (size_t)t * tb + e0;
      tpe_stage<s * s>(st, SF, oC, p.C + i0 * s * s, nv, lane);
      if (p.c) {
        tpe_stage<s>(st, SF, oc, p.c + i0 * s, nv, lane);
      } else {
        if (p.cx) tpe_stage<n>(st, SF, oc, p.cx + i0 * n, nv, lane); else tpe_zero(st, SF, oc, n, nv, lane);
        if (p.cu) tpe_stage<m>(st, SF, oc + n, p.cu + i0 * m, nv, lane); else tpe_zero(st, SF, oc + n, m, nv, lane);
      }
      if (t < T - 1) {
        tpe_stage<n * s>(st, SF, oF, p.F + i0 * n * s, nv, lane);
        if (have_f) tpe_stage<n>(st, SF, of, p.f + i0 * n, nv, lane);
      }
    };
#pragma unroll
    for (int k = 0; k < DS - 1; ++k) {                       // stage of step t lives in slot (T - 1 - t) % DS
      if (T - 1 - k >= 0) issue(T - 1 - k, k);
      cp_async_commit();
    }
    int slot = 0;
    R V[n][n], v[n];
    for (int t = T - 1; t >= 0; --t) {
      const size_t idx = (size_t)t * tb + e;
      if (t - (DS - 1) >= 0) issue(t - (DS - 1), slot == 0 ? DS - 1 : slot - 1);
      cp_async_commit();
      cp_async_wait<DS - 1>();
      __syncwarp();
      const R* my = wsm + slot * 32 * SF + ls * SF;
      // Q starts as C_t, q as c_scale * c_t
      R Q[s][s], q[s];
#pragma unroll
      for (int i = 0; i < s; ++i) {
#pragma unroll
        for (int j = 0; j < s; ++j) Q[i][j] = my[oC + i * s + j];
        q[i] = cs * my[oc + i];
      }
      if (t < T - 1) {
        R F[n][s];
#pragma unroll
        for (int i = 0; i < n; ++i)
#pragma unroll
          for (int j = 0; j < s; ++j) F[i][j] = my[oF + i * s + j];
        // Q += F^T (V F), q += F^T (V f + v): one row of V F at a time (lqr_recursion.py:79-95)
#pragma unroll
        for (int k = 0; k < n; ++k) {
          R Mk[s];
#pragma unroll
          for (int j = 0; j < s; ++j) {
            R acc = R(0);
#pragma unroll
            for (int i = 0; i < n; ++i) acc += V[k][i] * F[i][j];
            Mk[j] = acc;
          }
          R mvk = v[k];
          if (have_f) {
#pragma unroll
            for (int i = 0; i < n; ++i) mvk += V[k][i] * my[of + i];
          }
#pragma unroll
          for (int i = 0; i < s; ++i) {
#pragma unroll
            for (int j = 0; j < s; ++j) Q[i][j] += F[k][i] * Mk[j];
            q[i] += F[k][i] * mvk;
          }
        }
      }
      // H = Quu (masked: active rows / columns zeroed, +1e-8 on an active diagonal, active_constrained_lqr.py:112-126);
      // X = [-Qux | -qu | I] -> after the solve [K | k | Quu^-1]
      bool act[m];
#pragma unroll
      for (int i = 0; i < m; ++i) act[i] = masked && p.active[idx * m + i] != 0;
      R H[m][m], X[m][NC];
#pragma unroll
      for (int i = 0; i < m; ++i) {
#pragma unroll
        for (int j = 0; j < m; ++j) {
          R hv = Q[n + i][n + j];
          if (act[i] || act[j]) hv = R(0);
          if (act[i] && i == j) hv += R(1e-8);
          H[i][j] = hv;
        }
#pragma unroll
        for (int j = 0; j < n; ++j) X[i][j] = act[i] ? R(0) : -Q[n + i][j];
        X[i][n] = act[i] ? R(0) : -q[n + i];
#pragma unroll
        for (int j = 0; j < m; ++j) X[i][n + 1 + j] = (i == j) ? R(1) : R(0);
      }
      tpe_solve<R, M, NC>(H, X);
      if (valid) {
        R* Kg = p.Ks + idx * m * n; R* kg = p.ks + idx * m;
#pragma unroll
        for (int i = 0; i < m; ++i) {
#pragma unroll
          for (int j = 0; j < n; ++j) Kg[i * n + j] = X[i][j];
          kg[i] = X[i][n];
        }
        if (save_fac) {
          R* fg = p.fac + idx * (m * m + n * m);
#pragma unroll
          for (int i = 0; i < m; ++i)
#pragma unroll
            for (int j = 0; j < m; ++j) fg[i * m + j] = X[i][n + 1 + j];
#pragma unroll
          for (int i = 0; i < n; ++i)
#pragma unroll
            for (int j = 0; j < m; ++j) fg[m * m + i * m + j] = Q[i][n + j];
        }
      }
      if (t > 0) {
        // P = [Qux | qu] + Quu [K | k] (unmasked Quu, Qux: Q6);  [V | v] = [Qxx | qx] + Qxu [K | k] + K^T P
        R P[m][n + 1];
#pragma unroll
        for (int i = 0; i < m; ++i)
#pragma unroll
          for (int j = 0; j <= n; ++j) {
            R a = (j < n) ? Q[n + i][j] : q[n + i];
#pragma unroll
            for (int l = 0; l < m; ++l) a += Q[n + i][n + l] * X[l][j];
            P[i][j] = a;
          }
#pragma unroll
        for (int i = 0; i < n; ++i)
#pragma unroll
          for (int j = 0; j <= n; ++j) {
            R a = (j < n) ? Q[i][j] : q[i];
            R b = R(0);
#pragma unroll
            for (int l = 0; l < m; ++l) { a += Q[i][n + l] * X[l][j]; b += X[l][i] * P[l][j]; }
            if (j < n) V[i][j] = a + b; else v[i] = a + b;
          }
        if (p.Vsave && valid) {
          R* Vg = p.Vsave + idx * (n * n + n);
#pragma unroll
          for (int i = 0; i < n; ++i) {
#pragma unroll
            for (int j = 0; j < n; ++j) Vg[i * n + j] = V[i][j];
            Vg[n * n + i] = v[i];
          }
        }
      }
      __syncwarp();                                          // every lane is done with this stage before it is refilled
      slot = slot == DS - 1 ? 0 : slot + 1;
    }
  }

  if (p.flags & LQR_DO_ROLLOUT) {                            // lqr_recursion.py:160-200
    // K_t, k_t were written by this warp's own lanes above (or by an earlier launch): make them visible to the copies
    __threadfence_block();
    __syncwarp();
    auto issue = [&](int t, int slot) {
      R* st = wsm + slot * 32 * SR;
      const size_t i0 = (size_t)t * tb + e0;
      tpe_stage<m * n>(st, SR, rK, p.Ks + i0 * m * n, nv, lane);
      tpe_stage<m>(st, SR, rk, p.ks + i0 * m, nv, lane);
      if (t < T - 1) {
        tpe_stage<n * s>(st, SR, rF, p.F + i0 * n * s, nv, lane);
        if (have_f) tpe_stage<n>(st, SR, rf, p.f + i0 * n, nv, lane);
      }
    };
#pragma unroll
    for (int k = 0; k < DR - 1; ++k) {                       // stage of step t lives in slot t % DR
      if (k < T) issue(k, k);
      cp_async_commit();
    }
    int slot = 0;
    R x[s];
#pragma unroll
    for (int i = 0; i < n; ++i) x[i] = p.x0[(size_t)e * n + i];
    for (int t = 0; t < T; ++t) {
      const size_t idx = (size_t)t * tb + e;
      if (t + DR - 1 < T) issue(t + DR - 1, slot == 0 ? DR - 1 : slot - 1);
      cp_async_commit();
      cp_async_wait<DR - 1>();
      __syncwarp();
      const R* my = wsm + slot * 32 * SR + ls * SR;
#pragma unroll
      for (int o = 0; o < m; ++o) {
        R a0 = my[rk + o], a1 = R(0);                        // two interleaved accumulators
#pragma unroll
        for (int k = 0; k < n; ++k) { if (k & 1) a1 += my[rK + o * n + k] * x[k]; else a0 += my[rK + o * n + k] * x[k]; }
        R uv = a0 + a1;
        if (masked && p.active[idx * m + o]) uv = R(0);      // active_constrained_lqr.py:175
        x[n + o] = uv;
      }
      if (valid) {
        if (p.x) {
#pragma unroll
          for (int i = 0; i < n; ++i) p.x[idx * n + i] = x[i];
        }
        if (p.u) {
#pragma unroll
          for (int i = 0; i < m; ++i) p.u[idx * m + i] = x[n + i];
        }
        if (p.tau_out) {
#pragma unroll
          for (int i = 0; i < s; ++i) p.tau_out[idx * s + i] = x[i];
        }
      }
      if (t < T - 1) {
        R xn[n];
#pragma unroll
        for (int o = 0; o < n; ++o) {
          R a0 = have_f ? my[rf + o] : R(0), a1 = R(0);
#pragma unroll
          for (int k = 0; k < s; ++k) { if (k & 1) a1 += my[rF + o * s + k] * x[k]; else a0 += my[rF + o * s + k] * x[k]; }
          xn[o] = a0 + a1;
        }
#pragma unroll
        for (int o = 0; o < n; ++o) x[o] = xn[o];
      }
      __syncwarp();
      slot = slot == DR - 1 ? 0 : slot + 1;
    }
  }
}

// dot_rot (common.cuh) on compile-time sizes: same rotated start, same two interleaved accumulators, fully unrolled so
// that register arrays stay in registers
template <int K, int ROT, typename R, typename A, typename B>
__device__ __forceinline__ R tpe_dot_rot(const A& row, const B& vec, R init) {
  R a0 = init, a1 = R(0);
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const int k = (ROT % K + i) % K;
    if (i & 1) a1 += row(k) * vec(k); else a0 += row(k) * vec(k);
  }
  return a0 + a1;
}

// The second LQR solve of DiffLqr.backward with the saved factors (lqr_dtau_kernel, non-fused form; reference
// lqr/differentiable_lqr.py:106-112) for s <= 6, one thread per element.  The work per step is two tiny mat-vecs: the
// group kernel's 1 us per step (config 2: 0.100 ms for 2 x 50 steps) is its two-stage operand pipeline against DRAM
// latency, so the ring here is at least three stages deep (DD - 1 steps ahead) in both sweeps.  dc carries k'_t in its control rows
// between the sweeps exactly as in lqr_dtau_kernel.
__host__ __device__ constexpr int tpe_dtau_stride(int n, int m) { return (n * (n + m) + m * m + n * m + n + m) | 1; }
__host__ __device__ constexpr int tpe_dtau_warp_reals(int n, int m, int dd) { return dd * 32 * tpe_dtau_stride(n, m); }

template <int O, int M, typename R, typename QV>
__device__ __forceinline__ void tpe_dtau_kp(const R* fac, const QV& qu, R (&kp)[M]) {
  if constexpr (O < M) {
    kp[O] = -tpe_dot_rot<M, O, R>([&](int k) { return fac[O * M + k]; }, qu, R(0));
    tpe_dtau_kp<O + 1, M, R>(fac, qu, kp);
  }
}
template <int O, int N, int M, typename R>
__device__ __forceinline__ void tpe_dtau_vp(const R* qxu, const R (&kp)[M], const R (&q)[N + M], R (&vp)[N]) {
  if constexpr (O < N) {
    vp[O] = tpe_dot_rot<M, O, R>([&](int k) { return qxu[O * M + k]; }, [&](int k) { return kp[k]; }, q[O]);
    tpe_dtau_vp<O + 1, N, M, R>(qxu, kp, q, vp);
  }
}
template <int O, int N, int M, typename R>
__device__ __forceinline__ void tpe_dtau_du(const R* Kt, const R (&kn)[M], R (&dx)[N + M]) {
  if constexpr (O < M) {
    dx[N + O] = tpe_dot_rot<N, O, R>([&](int k) { return Kt[O * N + k]; }, [&](int k) { return dx[k]; }, kn[O]);
    tpe_dtau_du<O + 1, N, M, R>(Kt, kn, dx);
  }
}
template <int O, int N, int M, typename R>
__device__ __forceinline__ void tpe_dtau_dx(const R* Ft, const R (&dx)[N + M], R (&xn)[N]) {
  if constexpr (O < N) {
    xn[O] = tpe_dot_rot<N + M, O, R>([&](int k) { return Ft[O * (N + M) + k]; }, [&](int k) { return dx[k]; }, R(0));
    tpe_dtau_dx<O + 1, N, M, R>(Ft, dx, xn);
  }
}

template <typename R, int N, int M, int TPB, int DD>
__global__ void __launch_bounds__(TPB) lqr_dtau_tpe_kernel(DtauParams<R> p, int epw) {
  constexpr int n = N, m = M, s = N + M, fsz = M * M + N * M;
  constexpr int SD = tpe_dtau_stride(N, M);
  constexpr int oF = 0, oA = n * s, ogx = n * s + fsz, ogu = n * s + fsz + n;      // sweep 1 slot: F | Quu^-1 | Qxu | gx | gu
  constexpr int oK = n * s;                                                        // sweep 2 slot: F | K
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int T = p.T;
  const int lane = threadIdx.x & 31;
  const int e0 = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * epw;
  if (e0 >= p.B) return;
  const int nv = p.B - e0 < epw ? p.B - e0 : epw;
  const bool valid = lane < nv;
  const int ls = valid ? lane : nv - 1;
  const int e = e0 + ls;
  const size_t tb = (size_t)p.B;
  R* wsm = reinterpret_cast<R*>(smem_raw) + (size_t)(threadIdx.x >> 5) * tpe_dtau_warp_reals(N, M, DD);

  // ---- sweep 1 (t = T-1 .. 0): q = g_t + F_t^T v'_{t+1};  k'_t = -Quu^-1 q_u;  v'_t = q_x + Qxu k'_t
  {
    auto issue = [&](int t, int slot) {
      R* st = wsm + slot * 32 * SD;
      const size_t i0 = (size_t)t * tb + e0;
      if (t < T - 1) tpe_stage<n * s>(st, SD, oF, p.F + i0 * n * s, nv, lane);
      tpe_stage<fsz>(st, SD, oA, p.fac + i0 * fsz, nv, lane);
      tpe_stage<n>(st, SD, ogx, p.gx + i0 * n, nv, lane);
      tpe_stage<m>(st, SD, ogu, p.gu + i0 * m, nv, lane);
    };
#pragma unroll
    for (int k = 0; k < DD - 1; ++k) {
      if (T - 1 - k >= 0) issue(T - 1 - k, k);
      cp_async_commit();
    }
    int slot = 0;
    R vp[n];
    for (int t = T - 1; t >= 0; --t) {
      if (t - (DD - 1) >= 0) issue(t - (DD - 1), slot == 0 ? DD - 1 : slot - 1);
      cp_async_commit();
      cp_async_wait<DD - 1>();
      __syncwarp();
      const R* my = wsm + slot * 32 * SD + ls * SD;
      R q[s];
#pragma unroll
      for (int o = 0; o < s; ++o) {
        R a0 = (o < n) ? my[ogx + o] : my[ogu + o - n], a1 = R(0);
        if (t < T - 1) {
#pragma unroll
          for (int k = 0; k < n; ++k) { if (k & 1) a1 += my[oF + k * s + o] * vp[k]; else a0 += my[oF + k * s + o] * vp[k]; }
        }
        q[o] = a0 + a1;
      }
      R kp[m];
      tpe_dtau_kp<0, M, R>(my + oA, [&](int k) { return q[n + k]; }, kp);
      tpe_dtau_vp<0, N, M, R>(my + oA + m * m, kp, q, vp);
      if (valid) {
#pragma unroll
        for (int o = 0; o < m; ++o) p.dc[((size_t)t * tb + e) * s + n + o] = kp[o];
      }
      __syncwarp();
      slot = slot == DD - 1 ? 0 : slot + 1;
    }
  }
  // ---- sweep 2 (t = 0 .. T-1): du_t = K_t dx_t + k'_t;  dx_{t+1} = F_t [dx_t; du_t];  dc[t] <- [dx_t; du_t]
  {
    auto issue = [&](int t, int slot) {
      R* st = wsm + slot * 32 * SD;
      const size_t i0 = (size_t)t * tb + e0;
      if (t < T - 1) tpe_stage<n * s>(st, SD, oF, p.F + i0 * n * s, nv, lane);
      tpe_stage<m * n>(st, SD, oK, p.Ks + i0 * m * n, nv, lane);
    };
#pragma unroll
    for (int k = 0; k < DD - 1; ++k) {
      if (k < T) issue(k, k);
      cp_async_commit();
    }
    int slot = 0;
    R dx[s], kn[m];
#pragma unroll
    for (int o = 0; o < n; ++o) dx[o] = R(0);
#pragma unroll
    for (int o = 0; o < m; ++o) kn[o] = p.dc[(size_t)e * s + n + o];               // this thread's own k'_0 (written above)
    for (int t = 0; t < T; ++t) {
      const size_t idx = (size_t)t * tb + e;
      if (t + DD - 1 < T) issue(t + DD - 1, slot == 0 ? DD - 1 : slot - 1);
      cp_async_commit();
      cp_async_wait<DD - 1>();
      __syncwarp();
      const R* my = wsm + slot * 32 * SD + ls * SD;
      tpe_dtau_du<0, N, M, R>(my + oK, kn, dx);
      if (t + 1 < T) {                                                             // k'_{t+1}: requested a step ahead
#pragma unroll
        for (int o = 0; o < m; ++o) kn[o] = p.dc[(idx + tb) * s + n + o];
      }
      if (valid) {
#pragma unroll
        for (int o = 0; o < s; ++o) p.dc[idx * s + o] = dx[o];
      }
      if (t < T - 1) {
        R xn[n];
        tpe_dtau_dx<0, N, M, R>(my + oF, dx, xn);
#pragma unroll
        for (int o = 0; o < n; ++o) dx[o] = xn[o];
      }
      __syncwarp();
      slot = slot == DD - 1 ? 0 : slot + 1;
    }
  }
}

// shared memory -> global mirror of tpe_stage: the warp writes CNT reals per element for nv consecutive elements as one
// contiguous, coalesced run
template <int CNT, typename R>
__device__ __forceinline__ void tpe_unstage(R* gdst, const R* src, int stride, int off, int nv, int lane) {
  if (nv == 32) {
    constexpr int Q32 = 32 / CNT, R32 = 32 % CNT;
    int j = lane % CNT;
    int d = (lane / CNT) * stride + off + j;
#pragma unroll
    for (int it = 0; it < CNT; ++it) {
      gdst[lane + 32 * it] = src[d];
      j += R32; d += Q32 * stride + R32;
      if (j >= CNT) { j -= CNT; d += stride - CNT; }
    }
  } else {
    const int total = nv * CNT;
    for (int i = lane; i < total; i += 32) { const int le = i / CNT, j = i - le * CNT; gdst[i] = src[le * stride + off + j]; }
  }
}

// lambda / d-lambda recursions + dC, dc, dF, df, dx0 (adjoint_out_kernel without ADJ_REDUCE_TB; reference
// lqr/differentiable_lqr.py:87-104, 114-134 and mpc/mpc_step.py:383-446) for s <= 6, one thread per element.  Inputs come
// through the same warp-staged ring as above; the outputs of a step (s*s + s + n*s + n reals per element, 560 bytes at
// config 2) go back through shared memory too, so that the warp stores them as contiguous runs instead of 32 scattered
// 8-byte pieces per instruction.
__host__ __device__ constexpr int tpe_adj_stride_in(int n, int m) { return (2 * n * (n + m) + 3 * n + m + (n + m)) | 1; }
__host__ __device__ constexpr int tpe_adj_stride_out(int n, int m) { return ((n + m) * (n + m) + (n + m) + n * (n + m) + n) | 1; }
__host__ __device__ constexpr int tpe_adj_warp_reals(int n, int m) { return 32 * (2 * tpe_adj_stride_in(n, m) + tpe_adj_stride_out(n, m)); }

template <int I, int N, int M, typename R>
__device__ __forceinline__ void tpe_adj_lam(const R* my, int oC, int oc, int oF, int og, const R (&tau)[N + M], const R (&dt)[N + M],
                                            const R (&lam)[N], const R (&dlam)[N], bool have_next, bool have_g, R rsgn,
                                            R (&lamn)[N], R (&dlamn)[N]) {
  if constexpr (I < N) {
    constexpr int s = N + M;
    R a0 = my[oc + I];                                       // lam: c_i + C_i tau, rotated start (as adjoint_out_kernel)
#pragma unroll
    for (int c = 0; c < s; ++c) { const int j = (I % s + c) % s; a0 += my[oC + I * s + j] * tau[j]; }
    R a1 = R(0), b1 = R(0);
    if (have_next) {
#pragma unroll
      for (int k = 0; k < N; ++k) { a1 += my[oF + k * s + I] * lam[k]; b1 += my[oF + k * s + I] * dlam[k]; }
    }
    lamn[I] = a0 + a1;
    const R b0 = tpe_dot_rot<s, I, R>([&](int k) { return my[oC + I * s + k]; }, [&](int k) { return dt[k]; },
                                      have_g ? rsgn * my[og + I] : R(0));
    dlamn[I] = b0 + b1;
    tpe_adj_lam<I + 1, N, M, R>(my, oC, oc, oF, og, tau, dt, lam, dlam, have_next, have_g, rsgn, lamn, dlamn);
  }
}

template <typename R, int N, int M, int TPB>
__global__ void __launch_bounds__(TPB) adjoint_out_tpe_kernel(AdjOutParams<R> p, int epw) {
  constexpr int n = N, m = M, s = N + M;
  constexpr int SI = tpe_adj_stride_in(N, M), SO = tpe_adj_stride_out(N, M);
  constexpr int oC = 0, oc = n * s, oF = n * s + n, ox = 2 * n * s + n, ou = ox + n, od = ou + m, og = od + s;   // in slot
  constexpr int qC = 0, qc = s * s, qF = s * s + s, qf = s * s + s + n * s;                                     // out slot
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int T = p.T;
  const int lane = threadIdx.x & 31;
  const int e0 = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * epw;
  if (e0 >= p.B) return;
  const int nv = p.B - e0 < epw ? p.B - e0 : epw;
  const bool valid = lane < nv;
  const int ls = valid ? lane : nv - 1;
  const int e = e0 + ls;
  const size_t tb = (size_t)p.B;
  R* wsm = reinterpret_cast<R*>(smem_raw) + (size_t)(threadIdx.x >> 5) * tpe_adj_warp_reals(N, M);
  R* outs = wsm + 2 * 32 * SI;
  const bool neg = (p.flags & ADJ_NEGATE) != 0;
  const R sgn = neg ? R(-1) : R(1);
  const R rsgn = (p.flags & ADJ_NEG_RHS) ? R(-1) : R(1);
  const bool quirk_dC = (p.flags & ADJ_QUIRK_DC) != 0, quirk_df = (p.flags & ADJ_QUIRK_DF) != 0;
  const bool have_g = p.gx != nullptr;
  const bool write_dc = neg || p.dc != p.dtau;

  // top n rows of C_t and the first n entries of c_t: prefixes of the elements' records (tpe_stage_rows)
  auto issue_in = [&](int t, int slot) {
    R* st = wsm + slot * 32 * SI;
    const size_t i0 = (size_t)t * tb + e0;
    tpe_stage_rows<n * s, s * s>(st, SI, oC, p.C + i0 * s * s, nv, lane);
    tpe_stage_rows<n, s>(st, SI, oc, p.c + i0 * s, nv, lane);
    if (t < T - 1) tpe_stage<n * s>(st, SI, oF, p.F + i0 * n * s, nv, lane);
    tpe_stage<n>(st, SI, ox, p.x + i0 * n, nv, lane);
    tpe_stage<m>(st, SI, ou, p.u + i0 * m, nv, lane);
    tpe_stage<s>(st, SI, od, p.dtau + i0 * s, nv, lane);
    if (have_g) tpe_stage<n>(st, SI, og, p.gx + i0 * n, nv, lane);
  };
  issue_in(T - 1, 0);
  cp_async_commit();
  int slot = 0;
  R lam[n], dlam[n];
#pragma unroll
  for (int i = 0; i < n; ++i) { lam[i] = R(0); dlam[i] = R(0); }
  for (int t = T - 1; t >= 0; --t) {
    const size_t i0 = (size_t)t * tb + e0;
    if (t > 0) issue_in(t - 1, slot ^ 1);
    cp_async_commit();
    cp_async_wait<1>();
    __syncwarp();
    const R* my = wsm + slot * 32 * SI + ls * SI;
    R* mo = outs + ls * SO;
    R tau[s], dt[s];
#pragma unroll
    for (int j = 0; j < s; ++j) { tau[j] = my[ox + j]; dt[j] = my[od + j]; }      // x | u are adjacent in the slot
    const bool have_next = t < T - 1;
    // dF_t = dlam_{t+1} (x) tau_t + lam_{t+1} (x) dtau_t   (t < T-1)
    if (have_next && valid) {
#pragma unroll
      for (int i = 0; i < n; ++i)
#pragma unroll
        for (int j = 0; j < s; ++j) mo[qF + i * s + j] = sgn * (dlam[i] * tau[j] + lam[i] * dt[j]);
      if (!quirk_df) {
#pragma unroll
        for (int i = 0; i < n; ++i) mo[qf + i] = sgn * dlam[i];
      }
    }
    R lamn[n], dlamn[n];
    tpe_adj_lam<0, N, M, R>(my, oC, oc, oF, og, tau, dt, lam, dlam, have_next, have_g, rsgn, lamn, dlamn);
    if (valid) {
#pragma unroll
      for (int i = 0; i < s; ++i)
#pragma unroll
        for (int j = 0; j < s; ++j) {
          const R a = dt[i] * tau[j], b = tau[i] * dt[j];
          mo[qC + i * s + j] = quirk_dC ? (R(0.5) * a + b) : (sgn * R(0.5) * (a + b));
        }
#pragma unroll
      for (int i = 0; i < s; ++i) mo[qc + i] = sgn * dt[i];
      if (quirk_df && have_next) {
#pragma unroll
        for (int i = 0; i < n; ++i) mo[qf + i] = sgn * dlamn[i];
      }
      if (t == 0) {
#pragma unroll
        for (int i = 0; i < n; ++i) p.dx0[(size_t)e * n + i] = sgn * dlamn[i];
      }
    }
#pragma unroll
    for (int i = 0; i < n; ++i) { lam[i] = lamn[i]; dlam[i] = dlamn[i]; }
    __syncwarp();                                            // the step's outputs are in the out slots
    tpe_unstage<s * s>(p.dC + i0 * s * s, outs, SO, qC, nv, lane);
    if (write_dc) tpe_unstage<s>(p.dc + i0 * s, outs, SO, qc, nv, lane);
    if (have_next) {
      tpe_unstage<n * s>(p.dF + i0 * n * s, outs, SO, qF, nv, lane);
      if (p.df) tpe_unstage<n>(p.df + i0 * n, outs, SO, qf, nv, lane);
    }
    __syncwarp();                                            // out slots and this input stage may be overwritten
    slot ^= 1;
  }
  // zero-fill the T-th row of dF when F was given with T rows (Q8, mpc_step.py:428)
  if (p.F_T == T && valid) {
    R* dFg = p.dF + ((size_t)(T - 1) * tb + e) * n * s;
#pragma unroll
    for (int o = 0; o < n * s; ++o) dFg[o] = R(0);
  }
}

}  // namespace dmpc
