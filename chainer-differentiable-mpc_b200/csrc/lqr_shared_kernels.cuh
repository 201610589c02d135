// LQR batches whose C_t and F_t are shared by every element (DESIGN.md §4.7).
//
// With C_t, F_t the same for all b, every matrix of the recursion is too: Q_t, Quu_t^-1, Qxu_t, K_t, V_t.  One Riccati
// sweep at B = 1 (launch_lqr_solve with FACTOR | SAVE_FAC, a zero c and Vsave) produces them; what is left per element is
// a set of linear vector recursions with shared matrices.  A CTA owns a chunk of NB consecutive elements and keeps their
// vectors as [NB][len] blocks in shared memory (the reference's [T][B][len] layout, so every per-t tile is one
// contiguous run); each step is a handful of products (shared matrix) x [len x NB].
//
//   lqr_shared_fwd_kernel    vector sweep  (t down)  mv = V_{t+1} f_t + v_{t+1};  q = c_t + F_t^T mv;
//                                                    k_t = -Quu^-1 q_u;  v_t = q_x + Qxu k_t   (= q_x - G_t q_u,
//                                                    G_t = Qxu Quu^-1: no symmetry of C is assumed)
//                            rollout       (t up)    u_t = K_t x_t + k_t;  x_{t+1} = F_t [x_t; u_t] + f_t
//   lqr_shared_adj_kernel    d-tau sweep   (t down)  the same with c := [gx; gu], f = 0     (differentiable_lqr.py:106-112)
//                            d-tau rollout (t up)    from d-x_0 = 0
//                            lambda sweep  (t down)  reference form (:87-104, :114-125):
//                                                    lambda_t = A_t^T lambda_{t+1} + C_t[:n,:] tau_t + c_t[:n],
//                                                    d-lambda likewise with d-tau and gx; per chunk and t the partial
//                                                    sums P_t = sum_b dtau tau^T and R_t = sum_b (dlambda_{t+1} tau_t^T +
//                                                    lambda_{t+1} dtau_t^T)
//   lqr_shared_reduce_kernel dC_t, dF_t from the partials, summed over the chunks in a fixed order (no atomics)
//
// Batch-shared c (c_shared: c is [T,s], the model's one learned block).  c_t is staged once per step and read with a
// column stride of 0.  With f == nullptr as well, every element has the same k_t, and the B = 1 sweep (run on the real c)
// already holds it in ks: lqr_shared_rollout_kernel runs only the rollout, reading x0 and writing x, u.  With f given,
// lqr_shared_fwd_kernel runs its vector sweep on the stride-0 c.  The adjoint then returns dc[T,s] = sum_b dtau_{t,b}
// (the reference's dc = dtau, summed as the backward of the broadcast would): sweep 3 appends the chunk's sum_b dtau_t to
// its partial record and the reduce kernel sums those over the chunks in the same fixed order; sweeps 1-2 park k' and
// dtau in a [T,B,s] region of the workspace instead of in dc.
//
// Products: fp64 runs them on the FP64 tensor cores (mma.sync.m8n8k4.f64, 8x8 output tiles spread over the warps);
// fp32 on FMA.  Both sum in a fixed order, so results are deterministic.
#pragma once
#include "common.cuh"
#include "lqr_kernels.cuh"

namespace dmpc {

constexpr int kSharedThreads = 256;

template <typename R>
struct LqrSharedParams {
  int T, B, n, m, F_T, NB, flags;   // flags: ADJ_QUIRK_DC | ADJ_QUIRK_DF
  int c_shared;     // 1: c is [T,s] and dc is [T,s], summed over the batch
  const R* x0;      // [B,n]
  const R* C;       // [T,s,s]    shared
  const R* c;       // [T,B,s], or [T,s] when c_shared
  const R* F;       // [F_T,n,s]  shared
  const R* f;       // [T-1,B,n] or nullptr
  const R* Ks;      // [T,m,n]            K_t of the B = 1 sweep
  const R* ks;      // [T,m]              k_t of the B = 1 sweep (the batch's k_t when it ran on a shared c, f == nullptr)
  const R* fac;     // [T,m*m+n*m]        Quu_t^-1 | Qxu_t
  const R* Vsave;   // [T,n*n+n]          V_t | (unused) for t >= 1
  R* x;             // [T,B,n]  forward output / adjoint input
  R* u;             // [T,B,m]
  const R* gx;      // [T,B,n] or nullptr (zeros)
  const R* gu;      // [T,B,m] or nullptr (zeros)
  R* dx0;           // [B,n]
  R* dc;            // [T,B,s]; c_shared: [T,s] or nullptr
  R* df;            // [T-1,B,n] or nullptr
  R* park;          // [T,B,s]  k'_t, then d-tau_t, between the adjoint's sweeps (dc itself unless c_shared)
  R* part;          // [nchunk][T][shared_rec_elems]: P_t | R_t (| sum_b dtau_t when c_shared) per chunk
  R* dC;            // [T,s,s]
  R* dF;            // [F_T,n,s] or nullptr
};

// Reals of one partial record (one chunk, one step) of the adjoint.
__host__ __device__ __forceinline__ int shared_rec_elems(int n, int m, bool c_shared) {
  const int s = n + m;
  return s * s + n * s + (c_shared ? s : 0);
}

// Outputs of lqr_shared_reduce_kernel: dC, then dF (when given), then dc (c_shared, when given).
template <typename R>
__host__ __device__ __forceinline__ size_t shared_reduce_outputs(const LqrSharedParams<R>& p) {
  const size_t s = (size_t)(p.n + p.m);
  return (size_t)p.T * s * s + (p.dF ? (size_t)p.F_T * p.n * s : 0) + (p.c_shared && p.dc ? (size_t)p.T * s : 0);
}

// Shared-memory layouts (offsets in reals).  Each kernel has two staging slots (step t and the prefetched next step) and
// its state blocks.  Every offset is a multiple of 2 reals so 16-byte cp.async stays possible.
struct SharedFwdLayout {
  int oc, of, oF, oV, oQi, oK, slot;    // slot-relative
  int q, v, mv, kb, tau0, tau1, total;
  __host__ __device__ SharedFwdLayout(int n, int m, int NB) {
    const int s = n + m;
    auto r2 = [](int v) { return (v + 1) & ~1; };
    int o = 0;
    oc = o; o += r2(NB * s); of = o; o += r2(NB * n); oF = o; o += r2(n * s); oV = o; o += r2(n * n);
    oQi = o; o += r2(m * m + n * m);                     // Quu^-1 | Qxu, one run
    oK = o; o += r2(m * n);
    slot = o;
    o = 2 * slot;
    q = o; o += r2(NB * s); v = o; o += r2(NB * n); mv = o; o += r2(NB * n); kb = o; o += r2(NB * m);
    tau0 = o; o += r2(NB * s); tau1 = o; o += r2(NB * s);
    total = o;
  }
};

struct SharedAdjLayout {
  // sweep 1 slot: F | Qi | Qxu | g[NB][s];  sweep 2 slot: K | F;  sweep 3 slot: Cx[n][s] | F | tau[NB][s] | cx | gx
  int oF, oQi, og, oK, oCx, otau, ocx, ogx, slot;
  int q, v, kb, dtau, l0, l1, dl0, dl1, total;
  __host__ __device__ SharedAdjLayout(int n, int m, int NB) {
    const int s = n + m;
    auto r2 = [](int v) { return (v + 1) & ~1; };
    oF = 0;
    const int o1 = r2(n * s);                            // after F (common to all three sweeps)
    oQi = o1; og = oQi + r2(m * m + n * m);               // Quu^-1 | Qxu, one run
    const int end1 = og + r2(NB * s);
    oK = o1;
    const int end2 = oK + r2(m * n);
    oCx = o1; otau = oCx + r2(n * s); ocx = otau + r2(NB * s); ogx = ocx + r2(NB * n);
    const int end3 = ogx + r2(NB * n);
    slot = end1 > end2 ? end1 : end2;
    if (end3 > slot) slot = end3;
    int o = 2 * slot;
    // state: sweep 1 (q, v, kb) and sweep 3 (dtau, lambda, d-lambda pairs) are never live together
    q = o; v = q + r2(NB * s); kb = v + r2(NB * n);
    const int e1 = kb + r2(NB * m);
    dtau = o; l0 = dtau + r2(NB * s); l1 = l0 + r2(NB * n); dl0 = l1 + r2(NB * n); dl1 = dl0 + r2(NB * n);
    const int e3 = dl1 + r2(NB * n);
    total = e1 > e3 ? e1 : e3;
  }
};

__device__ __forceinline__ void dmma_f64(double (&c)[2], double a, double b) {
  asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
      : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}

// CTA-wide product: out(i,j) = base(i,j) + sgn * sum_{k<K} A(i,k) Bm(k,j) for i < I, j < J, with X(i,j) at
// X[i*xr + j*xc]; base may be nullptr (zero), K may be 0 (out = base).  out may alias base (the same thread reads and
// writes an entry) but not A or Bm.  Callers synchronise afterwards.
template <typename R>
__device__ __forceinline__ void cta_gemm(int I, int J, int K, R* out, int orr, int oc, const R* base, int br, int bc,
                                         const R* A, int ar, int ac, const R* Bm, int bkr, int bjc, bool neg) {
  if constexpr (sizeof(R) == 8) {
    // 8x8 output tiles over the warps; fragments of mma.m8n8k4.f64: lane (g, q) holds A(g, q), B(q, g), D(g, 2q..2q+1).
    // Out-of-range rows / columns / k load as zero, so no operand needs padding.
    const int warp = threadIdx.x >> 5, nw = blockDim.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, q = lane & 3;
    const int ti = (I + 7) >> 3, tj = (J + 7) >> 3;
    for (int tile = warp; tile < ti * tj; tile += nw) {
      const int i0 = (tile / tj) * 8, j0 = (tile % tj) * 8;
      const int i = i0 + g, ja = j0 + 2 * q, jb = ja + 1, jB = j0 + g;
      double acc[2];
      acc[0] = (base && i < I && ja < J) ? (double)base[i * br + ja * bc] : 0.0;
      acc[1] = (base && i < I && jb < J) ? (double)base[i * br + jb * bc] : 0.0;
      for (int k0 = 0; k0 < K; k0 += 4) {
        const int k = k0 + q;
        double a = (i < I && k < K) ? (double)A[i * ar + k * ac] : 0.0;
        const double b = (k < K && jB < J) ? (double)Bm[k * bkr + jB * bjc] : 0.0;
        if (neg) a = -a;
        dmma_f64(acc, a, b);
      }
      if (i < I && ja < J) out[i * orr + ja * oc] = (R)acc[0];
      if (i < I && jb < J) out[i * orr + jb * oc] = (R)acc[1];
    }
  } else {
    for (int o = threadIdx.x; o < I * J; o += blockDim.x) {
      const int i = o / J, j = o - i * J;
      R a0 = R(0), a1 = R(0);
      int k = 0;
      for (; k + 1 < K; k += 2) {
        a0 = fmaf(A[i * ar + k * ac], Bm[k * bkr + j * bjc], a0);
        a1 = fmaf(A[i * ar + (k + 1) * ac], Bm[(k + 1) * bkr + j * bjc], a1);
      }
      if (k < K) a0 = fmaf(A[i * ar + k * ac], Bm[k * bkr + j * bjc], a0);
      const R a = neg ? -(a0 + a1) : a0 + a1;
      out[i * orr + j * oc] = base ? base[i * br + j * bc] + a : a;
    }
  }
}

using CtaGrp = Grp<kSharedThreads>;

// cnt rows of w reals, src row stride sld -> [cnt][ld] shared block (cp.async, any alignment)
template <typename R>
__device__ __forceinline__ void stage_rows(R* dst, int ld, const R* src, int sld, int w, int cnt) {
  const CtaGrp g;
  if (w == ld && w == sld) { g_cp_async(g, dst, src, cnt * w); return; }
  for (int o = threadIdx.x; o < cnt * w; o += blockDim.x) {
    const int e = o / w, j = o - e * w;
    if (sizeof(R) == 8) cp_async8(dst + e * ld + j, src + e * sld + j); else cp_async4(dst + e * ld + j, src + e * sld + j);
  }
}
template <typename R>
__device__ __forceinline__ void zero_rows(R* dst, int ld, int w, int cnt) {
  for (int o = threadIdx.x; o < cnt * w; o += blockDim.x) { const int e = o / w; dst[e * ld + o - e * w] = R(0); }
}

// kRollOnly: c shared and f == nullptr, so k_t is the B = 1 sweep's ks and the vector sweep is skipped.
template <typename R, bool kRollOnly>
__device__ __forceinline__ void lqr_shared_fwd_body(const LqrSharedParams<R>& p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  R* sm = reinterpret_cast<R*>(smem_raw);
  const int n = p.n, m = p.m, s = n + m, T = p.T, NB = p.NB;
  const size_t B = (size_t)p.B;
  const int b0 = blockIdx.x * NB;
  const int ne = (p.B - b0) < NB ? (p.B - b0) : NB;
  const SharedFwdLayout L(n, m, NB);
  const CtaGrp g;
  const int fsz = m * m + n * m;
  int sl = 0;

  // ---- vector sweep, t = T-1 .. 0.  Slot of step t: c_t, f_t, F_t, V_{t+1}, Quu_t^-1, Qxu_t.
  if constexpr (!kRollOnly) {
    R *q = sm + L.q, *v = sm + L.v, *mv = sm + L.mv, *kb = sm + L.kb;
    const int cbs = p.c_shared ? 0 : s;                                   // column (element) stride of the staged c_t
    auto stage_bw = [&](int t, int sl) {
      R* S = sm + sl * L.slot;
      if (p.c_shared) g_cp_async(g, S + L.oc, p.c + (size_t)t * s, s);
      else g_cp_async(g, S + L.oc, p.c + ((size_t)t * B + b0) * s, ne * s);
      g_cp_async(g, S + L.oQi, p.fac + (size_t)t * fsz, fsz);
      if (t < T - 1) {
        g_cp_async(g, S + L.oF, p.F + (size_t)t * n * s, n * s);
        if (p.f) {
          g_cp_async(g, S + L.of, p.f + ((size_t)t * B + b0) * n, ne * n);
          g_cp_async(g, S + L.oV, p.Vsave + (size_t)(t + 1) * (n * n + n), n * n);
        }
      }
      cp_async_commit();
    };
    stage_bw(T - 1, 0);
    for (int t = T - 1; t >= 0; --t) {
      if (t > 0) { stage_bw(t - 1, sl ^ 1); cp_async_wait<1>(); } else cp_async_wait<0>();
      __syncthreads();
      R* S = sm + sl * L.slot;
      const R* vin = v;
      if (t < T - 1 && p.f) {                                                // mv = V_{t+1} f_t + v_{t+1}
        cta_gemm<R>(n, ne, n, mv, 1, n, v, 1, n, S + L.oV, n, 1, S + L.of, 1, n, false);
        __syncthreads();
        vin = mv;
      }
      // q = c_t + F_t^T mv     (t = T-1: q = c_t)
      cta_gemm<R>(s, ne, t < T - 1 ? n : 0, q, 1, s, S + L.oc, 1, cbs, S + L.oF, 1, s, vin, 1, n, false);
      __syncthreads();
      // k_t = -Quu^-1 q_u
      cta_gemm<R>(m, ne, m, kb, 1, m, nullptr, 0, 0, S + L.oQi, m, 1, q + n, 1, s, true);
      __syncthreads();
      // v_t = q_x + Qxu k_t; k_t is parked in the u output until the rollout reads it back
      if (t > 0) cta_gemm<R>(n, ne, m, v, 1, n, q, 1, s, S + L.oQi + m * m, m, 1, kb, 1, m, false);
      R* ug = p.u + ((size_t)t * B + b0) * m;
      for (int o = threadIdx.x; o < ne * m; o += blockDim.x) ug[o] = kb[o];
      __syncthreads();
      sl ^= 1;
    }
  }

  // ---- rollout, t = 0 .. T-1.  Slot of step t: K_t, F_t, f_t.
  auto stage_fw = [&](int t, int sl2) {
    R* S = sm + sl2 * L.slot;
    g_cp_async(g, S + L.oK, p.Ks + (size_t)t * m * n, m * n);
    if (t < T - 1) {
      g_cp_async(g, S + L.oF, p.F + (size_t)t * n * s, n * s);
      if (p.f) g_cp_async(g, S + L.of, p.f + ((size_t)t * B + b0) * n, ne * n);
    }
    cp_async_commit();
  };
  R* tc = sm + L.tau0; R* tn = sm + L.tau1;
  for (int o = threadIdx.x; o < ne * n; o += blockDim.x) { const int e = o / n; tc[e * s + o - e * n] = p.x0[(size_t)b0 * n + o]; }
  stage_fw(0, 0);
  sl = 0;
  for (int t = 0; t < T; ++t) {
    if (t < T - 1) { stage_fw(t + 1, sl ^ 1); cp_async_wait<1>(); } else cp_async_wait<0>();
    if constexpr (kRollOnly) {                                            // k_t of the B = 1 sweep, the same for all
      const R* kg = p.ks + (size_t)t * m;
      for (int o = threadIdx.x; o < ne * m; o += blockDim.x) { const int e = o / m; tc[e * s + n + o - e * m] = kg[o - e * m]; }
    } else {
      const R* ug = p.u + ((size_t)t * B + b0) * m;                       // k_t from the sweep (this CTA wrote it)
      for (int o = threadIdx.x; o < ne * m; o += blockDim.x) { const int e = o / m; tc[e * s + n + o - e * m] = ug[o]; }
    }
    __syncthreads();
    R* S = sm + sl * L.slot;
    cta_gemm<R>(m, ne, n, tc + n, 1, s, tc + n, 1, s, S + L.oK, n, 1, tc, 1, s, false);   // u = K x + k
    __syncthreads();
    R* xg = p.x + ((size_t)t * B + b0) * n; R* ug2 = p.u + ((size_t)t * B + b0) * m;
    for (int o = threadIdx.x; o < ne * n; o += blockDim.x) { const int e = o / n; xg[o] = tc[e * s + o - e * n]; }
    for (int o = threadIdx.x; o < ne * m; o += blockDim.x) { const int e = o / m; ug2[o] = tc[e * s + n + o - e * m]; }
    if (t < T - 1)                                                        // x_{t+1} = F_t tau_t + f_t
      cta_gemm<R>(n, ne, s, tn, 1, s, p.f ? S + L.of : nullptr, 1, n, S + L.oF, s, 1, tc, 1, s, false);
    __syncthreads();
    R* tmp = tc; tc = tn; tn = tmp;
    sl ^= 1;
  }
}

// Vector sweep + rollout (c per element, or c shared with f given).
template <typename R>
__global__ void __launch_bounds__(kSharedThreads) lqr_shared_fwd_kernel(const LqrSharedParams<R> p) {
  lqr_shared_fwd_body<R, false>(p);
}

// Rollout only (c shared, f == nullptr): k_t comes from the B = 1 sweep.
template <typename R>
__global__ void __launch_bounds__(kSharedThreads) lqr_shared_rollout_kernel(const LqrSharedParams<R> p) {
  lqr_shared_fwd_body<R, true>(p);
}

template <typename R>
__global__ void __launch_bounds__(kSharedThreads) lqr_shared_adj_kernel(const LqrSharedParams<R> p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  R* sm = reinterpret_cast<R*>(smem_raw);
  const int n = p.n, m = p.m, s = n + m, T = p.T, NB = p.NB;
  const size_t B = (size_t)p.B;
  const int b0 = blockIdx.x * NB;
  const int ne = (p.B - b0) < NB ? (p.B - b0) : NB;
  const SharedAdjLayout L(n, m, NB);
  const CtaGrp g;
  const int fsz = m * m + n * m;

  // ---- sweep 1, t = T-1 .. 0: q = g_t + F_t^T v'_{t+1};  k'_t = -Quu^-1 q_u;  v'_t = q_x + Qxu k'_t.  k'_t -> park[t][:, n:]
  {
    R *q = sm + L.q, *v = sm + L.v, *kb = sm + L.kb;
    auto stage1 = [&](int t, int sl) {
      R* S = sm + sl * L.slot;
      g_cp_async(g, S + L.oQi, p.fac + (size_t)t * fsz, fsz);
      if (t < T - 1) g_cp_async(g, S + L.oF, p.F + (size_t)t * n * s, n * s);
      if (p.gx) stage_rows(S + L.og, s, p.gx + ((size_t)t * B + b0) * n, n, n, ne); else zero_rows(S + L.og, s, n, ne);
      if (p.gu) stage_rows(S + L.og + n, s, p.gu + ((size_t)t * B + b0) * m, m, m, ne); else zero_rows(S + L.og + n, s, m, ne);
      cp_async_commit();
    };
    stage1(T - 1, 0);
    int sl = 0;
    for (int t = T - 1; t >= 0; --t) {
      if (t > 0) { stage1(t - 1, sl ^ 1); cp_async_wait<1>(); } else cp_async_wait<0>();
      __syncthreads();
      R* S = sm + sl * L.slot;
      cta_gemm<R>(s, ne, t < T - 1 ? n : 0, q, 1, s, S + L.og, 1, s, S + L.oF, 1, s, v, 1, n, false);
      __syncthreads();
      cta_gemm<R>(m, ne, m, kb, 1, m, nullptr, 0, 0, S + L.oQi, m, 1, q + n, 1, s, true);
      __syncthreads();
      if (t > 0) cta_gemm<R>(n, ne, m, v, 1, n, q, 1, s, S + L.oQi + m * m, m, 1, kb, 1, m, false);
      R* dg = p.park + ((size_t)t * B + b0) * s;
      for (int o = threadIdx.x; o < ne * m; o += blockDim.x) { const int e = o / m; dg[e * s + n + o - e * m] = kb[o]; }
      __syncthreads();
      sl ^= 1;
    }
  }

  // ---- sweep 2, t = 0 .. T-1: d-u_t = K_t d-x_t + k'_t;  d-x_{t+1} = F_t d-tau_t  (d-x_0 = 0).  d-tau_t -> park[t]
  {
    R* tc = sm + L.q; R* tn = sm + L.v;                                   // two [NB][s] blocks (q and v|kb of sweep 1)
    auto stage2 = [&](int t, int sl) {
      R* S = sm + sl * L.slot;
      g_cp_async(g, S + L.oK, p.Ks + (size_t)t * m * n, m * n);
      if (t < T - 1) g_cp_async(g, S + L.oF, p.F + (size_t)t * n * s, n * s);
      cp_async_commit();
    };
    zero_rows(tc, s, n, ne);
    stage2(0, 0);
    int sl = 0;
    for (int t = 0; t < T; ++t) {
      if (t < T - 1) { stage2(t + 1, sl ^ 1); cp_async_wait<1>(); } else cp_async_wait<0>();
      R* dg = p.park + ((size_t)t * B + b0) * s;
      for (int o = threadIdx.x; o < ne * m; o += blockDim.x) { const int e = o / m; const int j = n + o - e * m; tc[e * s + j] = dg[e * s + j]; }
      __syncthreads();
      R* S = sm + sl * L.slot;
      cta_gemm<R>(m, ne, n, tc + n, 1, s, tc + n, 1, s, S + L.oK, n, 1, tc, 1, s, false);
      __syncthreads();
      for (int o = threadIdx.x; o < ne * s; o += blockDim.x) dg[o] = tc[o];
      if (t < T - 1) cta_gemm<R>(n, ne, s, tn, 1, s, nullptr, 0, 0, S + L.oF, s, 1, tc, 1, s, false);
      __syncthreads();
      R* tmp = tc; tc = tn; tn = tmp;
      sl ^= 1;
    }
  }

  // ---- sweep 3, t = T-1 .. 0: lambda / d-lambda (reference form) and the chunk's P_t, R_t
  {
    R* dt = sm + L.dtau;
    R *lo = sm + L.l0, *ln = sm + L.l1, *dlo = sm + L.dl0, *dln = sm + L.dl1;   // lambda_{t+1} (old), lambda_t (new)
    const bool strict_df = (p.flags & ADJ_QUIRK_DF) != 0;
    const int rsz = shared_rec_elems(n, m, p.c_shared);
    const int cbs = p.c_shared ? 0 : n;                                   // column (element) stride of the staged c_x
    auto stage3 = [&](int t, int sl) {
      R* S = sm + sl * L.slot;
      g_cp_async(g, S + L.oCx, p.C + (size_t)t * s * s, n * s);          // rows 0..n-1 of C_t
      if (t < T - 1) g_cp_async(g, S + L.oF, p.F + (size_t)t * n * s, n * s);
      stage_rows(S + L.otau, s, p.x + ((size_t)t * B + b0) * n, n, n, ne);
      stage_rows(S + L.otau + n, s, p.u + ((size_t)t * B + b0) * m, m, m, ne);
      if (p.c_shared) g_cp_async(g, S + L.ocx, p.c + (size_t)t * s, n);   // c_t[:n], once
      else stage_rows(S + L.ocx, n, p.c + ((size_t)t * B + b0) * s, s, n, ne);   // c_t[:, :n]: rows of length n, stride s
      if (p.gx) g_cp_async(g, S + L.ogx, p.gx + ((size_t)t * B + b0) * n, ne * n); else zero_rows(S + L.ogx, n, n, ne);
      cp_async_commit();
    };
    stage3(T - 1, 0);
    int sl = 0;
    for (int t = T - 1; t >= 0; --t) {
      if (t > 0) { stage3(t - 1, sl ^ 1); cp_async_wait<1>(); } else cp_async_wait<0>();
      const R* dg = p.park + ((size_t)t * B + b0) * s;
      for (int o = threadIdx.x; o < ne * s; o += blockDim.x) dt[o] = dg[o];
      __syncthreads();
      R* S = sm + sl * L.slot;
      const R* tau = S + L.otau;
      R* pt = p.part + ((size_t)blockIdx.x * T + t) * rsz;
      if (p.c_shared)                                                     // sum_b dtau_t over the chunk, in element order
        for (int j = threadIdx.x; j < s; j += blockDim.x) {
          R a = R(0);
          for (int e = 0; e < ne; ++e) a += dt[e * s + j];
          pt[s * s + n * s + j] = a;
        }
      cta_gemm<R>(s, s, ne, pt, s, 1, nullptr, 0, 0, dt, 1, s, tau, s, 1, false);               // P_t = sum dtau tau^T
      if (t < T - 1) {                                                    // R_t = sum dlambda_{t+1} tau^T + lambda_{t+1} dtau^T
        cta_gemm<R>(n, s, ne, pt + s * s, s, 1, nullptr, 0, 0, dlo, 1, n, tau, s, 1, false);
        cta_gemm<R>(n, s, ne, pt + s * s, s, 1, pt + s * s, s, 1, lo, 1, n, dt, s, 1, false);
        if (!strict_df && p.df) {                                         // df[t] = dlambda_{t+1}
          R* fg = p.df + ((size_t)t * B + b0) * n;
          for (int o = threadIdx.x; o < ne * n; o += blockDim.x) fg[o] = dlo[o];
        }
      }
      // lambda_t = c_x + C_x tau_t (+ A_t^T lambda_{t+1}),  d-lambda_t = gx + C_x dtau_t (+ A_t^T dlambda_{t+1})
      cta_gemm<R>(n, ne, s, ln, 1, n, S + L.ocx, 1, cbs, S + L.oCx, s, 1, tau, 1, s, false);
      cta_gemm<R>(n, ne, s, dln, 1, n, S + L.ogx, 1, n, S + L.oCx, s, 1, dt, 1, s, false);
      __syncthreads();
      if (t < T - 1) {
        cta_gemm<R>(n, ne, n, ln, 1, n, ln, 1, n, S + L.oF, 1, s, lo, 1, n, false);
        cta_gemm<R>(n, ne, n, dln, 1, n, dln, 1, n, S + L.oF, 1, s, dlo, 1, n, false);
        __syncthreads();
      }
      if (strict_df && p.df && t < T - 1) {                               // df[t] = dlambda_t (reference :133)
        R* fg = p.df + ((size_t)t * B + b0) * n;
        for (int o = threadIdx.x; o < ne * n; o += blockDim.x) fg[o] = dln[o];
      }
      if (t == 0) {
        R* xg = p.dx0 + (size_t)b0 * n;
        for (int o = threadIdx.x; o < ne * n; o += blockDim.x) xg[o] = dln[o];
      }
      __syncthreads();
      R* tmp = lo; lo = ln; ln = tmp; tmp = dlo; dlo = dln; dln = tmp;
      sl ^= 1;
    }
  }
}

// dC_t = 0.5 P_t + P_t^T (ADJ_QUIRK_DC, reference :128) or 0.5 (P_t + P_t^T);  dF_t = R_t (t < T-1), 0 for row T-1;
// c_shared: dc_t = sum_b dtau_t.  One thread per output, chunks summed in index order: deterministic.
template <typename R>
__global__ void lqr_shared_reduce_kernel(const LqrSharedParams<R> p, int nchunk) {
  const int n = p.n, s = n + p.m, T = p.T, rsz = shared_rec_elems(n, p.m, p.c_shared);
  const size_t nC = (size_t)T * s * s, nCF = nC + (p.dF ? (size_t)p.F_T * n * s : 0), total = shared_reduce_outputs(p);
  const size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= total) return;
  if (o < nC) {
    const int t = (int)(o / (s * s)), ij = (int)(o - (size_t)t * s * s), i = ij / s, j = ij - i * s;
    R a = R(0), b = R(0);
    for (int k = 0; k < nchunk; ++k) {
      const R* pt = p.part + ((size_t)k * T + t) * rsz;
      a += pt[i * s + j];
      b += pt[j * s + i];
    }
    p.dC[o] = (p.flags & ADJ_QUIRK_DC) ? R(0.5) * a + b : R(0.5) * (a + b);
  } else if (o < nCF) {
    const size_t r = o - nC;
    const int t = (int)(r / (n * s)), ij = (int)(r - (size_t)t * n * s);
    R a = R(0);
    if (t < T - 1)
      for (int k = 0; k < nchunk; ++k) a += p.part[((size_t)k * T + t) * rsz + s * s + ij];
    p.dF[r] = a;
  } else {
    const size_t r = o - nCF;
    const int t = (int)(r / s), j = (int)(r - (size_t)t * s);
    R a = R(0);
    for (int k = 0; k < nchunk; ++k) a += p.part[((size_t)k * T + t) * rsz + s * s + n * s + j];
    p.dc[r] = a;
  }
}

// Elements per CTA: the largest of 64, 32, 16, 8 whose shared memory fits and that still gives every SM a CTA (down to 8).
// 0: no chunk fits (the shape is unsupported).  The workspace size depends on it (one partial record per chunk and t).
inline int lqr_shared_chunk(size_t real_bytes, int B, int n, int m, size_t max_smem) {
  for (int NB = 64; NB >= 8; NB /= 2) {
    const size_t a = (size_t)SharedFwdLayout(n, m, NB).total, b = (size_t)SharedAdjLayout(n, m, NB).total;
    if ((a > b ? a : b) * real_bytes > max_smem) continue;
    if (NB > 8 && (B + NB - 1) / NB < 148) continue;
    return NB;
  }
  return 0;
}

}  // namespace dmpc
