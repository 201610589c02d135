/*
 * diffmpc_b200 - C ABI of the B200-native batched LQR / box-DDP solver.
 *
 * Drop-in boundary for the hot path of pfnet-research/chainer-differentiable-mpc.
 * Every entry point states the reference interface it replaces (file:line in the
 * reference tree).  The reference is pure Python/NumPy, so "the FFI a maintainer
 * would bind" is ctypes: see INTEGRATION.md for the stubs.
 *
 * Conventions
 *   - All tensors use the reference's layout: time-major, batch-second, C-contiguous
 *     (lqr_recursion.py:51-66):  x_init[B,n] C[T,B,s,s] c[T,B,s] F[F_T,B,n,s] f[T-1,B,n]
 *     x[T,B,n] u[T,B,m]   with s = n + m and F_T in {T-1, T} (mpc_step.py:83-89).
 *   - dtype: DMPC_F64 (the reference is float64 end to end) or DMPC_F32.  dtype is the element type of
 *     every tensor argument; kernels compute in that type, except dmpc_lqr_solve at n=32, m=8 with
 *     DMPC_F32, which widens the float tiles and runs the fp64 tensor-core (DMMA) recursion.
 *   - Pointers named d_* are DEVICE pointers; the call is asynchronous on `stream`
 *     (a cudaStream_t passed as void*; NULL = the handle's stream).
 *   - Pointers named h_* are HOST pointers; those entry points copy in/out and
 *     synchronise before returning (they are what the Python facade uses).
 *   - Return value: 0 on success, else a dmpc_status; dmpc_last_error() has detail.
 *   - The library never falls back to a CPU path: without a CUDA device
 *     dmpc_create() returns DMPC_ERR_NO_DEVICE.
 *   - Inputs are never modified (pnqp.py:86, util.py:496,514 make copies);
 *     the caller owns every buffer.
 *   - Threads: the library keeps no global state; a handle carries a stream, a launch counter, the last error text and
 *     (dmpc_boxddp_solve) a small pinned record, so ONE thread at a time may use a given handle.  Different handles - also
 *     on the same device - may be used concurrently (bench.py's e2e feeders hold one each).
 */
#ifndef DIFFMPC_B200_H
#define DIFFMPC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dmpc_ctx* dmpc_handle;

enum dmpc_dtype { DMPC_F64 = 0, DMPC_F32 = 1 };

enum dmpc_status {
  DMPC_OK = 0,
  DMPC_ERR_BAD_SHAPE = 1,   /* the reference's shape asserts (lqr_recursion.py:51-66, mpc_step.py:79-92) */
  DMPC_ERR_BAD_BOUNDS = 2,  /* lower > upper (pnqp.py:64, mpc_step.py:139): returned by dmpc_boxddp_solve (which reads its
                               loop record anyway); the stream-ordered calls dmpc_pnqp / dmpc_mpc_step_forward do not
                               synchronise and report it per element instead (DMPC_FLAG_BAD_BOUNDS in d_flags) */
  DMPC_ERR_NONFINITE = 3,   /* NaN / inf asserts (mpc_step.py:133-135,161-162,284-285): returned by dmpc_boxddp_solve;
                               per element DMPC_FLAG_NONFINITE elsewhere */
  DMPC_ERR_CUDA = 4,
  DMPC_ERR_UNSUPPORTED = 5,
  DMPC_ERR_NULL = 6,
  DMPC_ERR_NO_DEVICE = 7
};

/* per-element flag bits reported in `d_flags[B]` (int32) */
enum dmpc_elem_flag {
  DMPC_FLAG_QP_NOT_CONVERGED = 1, /* pnqp.py:192 "Did not converge" warning */
  DMPC_FLAG_NONFINITE = 2,
  DMPC_FLAG_LS_CAPPED = 4,        /* line search hit the safety cap (mpc_step.py:196 would not terminate); d_alphas is
                                     the alpha of the trajectory that was written */
  DMPC_FLAG_BAD_BOUNDS = 8        /* lower > upper for this element at some timestep (the reference asserts) */
};

/* lqr_solve flags */
enum {
  DMPC_LQR_FACTOR = 1,   /* LqrRecursion.backward (lqr_recursion.py:69-158): Riccati sweep -> Ks, ks */
  DMPC_LQR_ROLLOUT = 2,  /* LqrRecursion.forward  (lqr_recursion.py:160-200): x, u from Ks, ks */
  DMPC_LQR_SAVE_FAC = 4  /* also store Quu^-1 and Qxu per (t,b) for dmpc_lqr_adjoint */
};

/* adjoint flags */
enum {
  DMPC_ADJ_STRICT_REFERENCE = 1, /* reproduce differentiable_lqr.py:128 (dC precedence) and :133 (df shift) */
  /* profiling aids: run one of the two kernels of dmpc_lqr_adjoint.  STAGE_OUT alone re-uses the d-tau that a
   * previous full (or STAGE_DTAU) call left in d_dc, so the pair can be timed kernel by kernel. */
  DMPC_ADJ_STAGE_DTAU_ONLY = 2,
  DMPC_ADJ_STAGE_OUT_ONLY = 4
};

/* coupling of the batch-global control flow of PNQP (SURVEY.md H2) */
enum dmpc_coupling { DMPC_COUPLING_ELEMENT = 0, DMPC_COUPLING_BATCH = 1 };

/* true-dynamics selector for the line-search rollout (mpc_step.py:229-240) */
enum dmpc_dynamics { DMPC_DYN_LINEAR = 0, DMPC_DYN_PENDULUM = 1 };

/* ---- library / context ------------------------------------------------------------- */
int dmpc_version(void);
const char* dmpc_status_string(int status);
int dmpc_create(int device, dmpc_handle* out);
int dmpc_destroy(dmpc_handle h);
const char* dmpc_last_error(dmpc_handle h);
int dmpc_device_count(void);

/* ---- memory / stream helpers (so a ctypes host needs no other CUDA binding) ---------- */
int dmpc_malloc(dmpc_handle h, size_t bytes, void** d_ptr);
int dmpc_free(dmpc_handle h, void* d_ptr);
int dmpc_host_alloc(dmpc_handle h, size_t bytes, void** h_ptr); /* pinned */
int dmpc_host_free(dmpc_handle h, void* h_ptr);
int dmpc_memcpy_h2d(dmpc_handle h, void* d_dst, const void* h_src, size_t bytes, void* stream);
int dmpc_memcpy_d2h(dmpc_handle h, void* h_dst, const void* d_src, size_t bytes, void* stream);
int dmpc_memset(dmpc_handle h, void* d_dst, int value, size_t bytes, void* stream);
int dmpc_sync(dmpc_handle h, void* stream);
/* number of kernels this handle has launched (bench.py's gpu_launches) */
long long dmpc_launch_count(dmpc_handle h);

/* ---- LQR (replaces LqrRecursion, lqr/lqr_recursion.py:18-209) ------------------------ */
/* elements (not bytes) of the factor cache written with DMPC_LQR_SAVE_FAC: Quu_t^-1 | Qxu_t per (t,b) [T,B,m*m+n*m], then
 * the value function V_t | v_t per (t,b) [T,B,n*n+n] (written for the shapes whose adjoint runs as two sweeps on
 * lambda_t = V_t x_t + v_t, today n=32/m=8, and by the large-system kernels; reserved otherwise).  Opaque to the caller: allocate, pass to lqr_solve, pass
 * on to lqr_adjoint. */
size_t dmpc_lqr_fac_elems(int T, int B, int n, int m);

/*
 * LqrRecursion.solve_recursion / .backward / .forward (lqr_recursion.py:202, :69, :160).
 *   flags = FACTOR|ROLLOUT  -> solve_recursion: writes d_Ks, d_ks, d_x, d_u
 *   flags = FACTOR          -> backward(): writes d_Ks[T,B,m,n], d_ks[T,B,m]
 *   flags = ROLLOUT         -> forward(Ks, ks): reads d_Ks, d_ks, writes d_x, d_u
 * d_f may be NULL (f is None).  d_fac may be NULL unless SAVE_FAC.
 * Alignment: any alignment of the element type is accepted.  The n=32/m=8 tensor-core kernel moves C, c, F, f, Ks, ks and
 * the factor cache with 16-byte asynchronous copies; when one of those pointers is not 16-byte aligned the call is served
 * by the generic kernel instead (same results, slower) - cudaMalloc'ed buffers and torch tensors are always aligned.
 * Shapes: any T, B >= 1 and 1 <= m <= 32, 1 <= n <= 128 in both dtypes.  Systems whose per-element layout does not fit one
 * CTA's shared memory (fp64 with SAVE_FAC from n = 64 / 58 / 52 / 38 at m = 1 / 8 / 16 / 32; fp32 from n = 90 / 85 / 78 / 65)
 * run the tile-parallel kernels of DESIGN.md 4.8, which allocate fp64 scratch stream-ordered on `stream` (up to
 * 8*(n(n+1) + s(s+1) + 2m(n+1)) bytes per element).  m > 32, or n > 128 where the per-element kernels do not fit:
 * DMPC_ERR_UNSUPPORTED, nothing launched.
 */
int dmpc_lqr_solve(dmpc_handle h, int dtype, int T, int B, int n, int m,
                   const void* d_x0, const void* d_C, const void* d_c,
                   const void* d_F, int F_T, const void* d_f,
                   void* d_x, void* d_u, void* d_Ks, void* d_ks, void* d_fac,
                   int flags, void* stream);

/*
 * DiffLqr.backward (lqr/differentiable_lqr.py:78-142).  Needs d_Ks and d_fac from a
 * dmpc_lqr_solve(... FACTOR|SAVE_FAC) on the same C, F.  Outputs have the shapes of
 * the inputs: d_dx0[B,n] d_dC[T,B,s,s] d_dc[T,B,s] d_dF[T-1,B,n,s] d_df[T-1,B,n] (nullable).
 * With DMPC_ADJ_STRICT_REFERENCE the reference's dC / df quirks (Q1, Q2) are reproduced;
 * without it the mathematically correct gradients are returned.
 * Shapes: as dmpc_lqr_solve; the factor cache of either kernel family is accepted.  Where the per-element adjoint kernels
 * do not fit shared memory the large-system kernels run (fp64 scratch of 16*T*B*n bytes, stream-ordered); outside
 * n <= 128, m <= 32 at such shapes: DMPC_ERR_UNSUPPORTED, nothing launched.
 */
int dmpc_lqr_adjoint(dmpc_handle h, int dtype, int T, int B, int n, int m,
                     const void* d_C, const void* d_c, const void* d_F,
                     const void* d_x, const void* d_u,
                     const void* d_gx, const void* d_gu,
                     const void* d_Ks, const void* d_fac,
                     void* d_dx0, void* d_dC, void* d_dc, void* d_dF, void* d_df,
                     int flags, void* stream);


/* ---- LQR with C and F shared by the batch (DiffLqr, lqr/differentiable_lqr.py:65-142, on a batch whose C_t, F_t are the
 *      same for every element: LqrNet / LqrNet_cost_dx, differentiable_lqr.py:186-198, 237-248) --------------------- */
/*
 * Shapes: d_C[T,s,s] and d_F[F_T,n,s] (F_T in {T-1, T}; row T-1 is not read) are ONE block per time step, shared by all B
 * elements; everything per element keeps the reference layout: d_x0[B,n] d_c[T,B,s] d_f[T-1,B,n] (NULL = None)
 * d_x[T,B,n] d_u[T,B,m].  Results equal dmpc_lqr_solve / dmpc_lqr_adjoint on the broadcast tensors, with the shared
 * gradients summed over the batch.  C need not be symmetric.
 * The workspace (dmpc_lqr_shared_workspace_bytes, any alignment) holds the matrices of the one Riccati sweep the whole
 * batch needs (K_t, Quu_t^-1, Qxu_t, V_t: a few KB to ~100 KB) and the per-chunk partial sums of the adjoint; its size
 * depends on (dtype, T, B, n, m).  m > 32 and shapes too large for the chunk kernels: DMPC_ERR_UNSUPPORTED (at NB = 8 the
 * chunk kernels hold fp64 n <= 74 / 70 / 64 / 53 and fp32 n <= 109 / 105 / 100 / 88 at m = 1 / 8 / 16 / 32); the one
 * Riccati sweep runs at any shape dmpc_lqr_solve runs.  The MPC step, its backward, dmpc_lqr_active_solve, dmpc_get_traj
 * (LinDx) and BoxDDP (LinDx) run every n <= 128, m <= 32 as well (DESIGN.md §4.9); dmpc_pnqp stays at m <= 32.
 */
int dmpc_lqr_shared_workspace_bytes(int dtype, int T, int B, int n, int m, size_t* bytes);

/*
 * LqrRecursion.solve_recursion (lqr_recursion.py:202-209) for the shared batch: the Riccati sweep (:69-158) runs once, at
 * B = 1, and leaves its matrices in d_ws; the per-element vector sweep (k_t, v_t: :85-120, :152) and the rollout
 * (:160-200) run for the whole batch.  Writes d_x, d_u (and d_ws, which dmpc_lqr_adjoint_shared reads).
 */
int dmpc_lqr_solve_shared(dmpc_handle h, int dtype, int T, int B, int n, int m,
                          const void* d_x0, const void* d_C, const void* d_c, const void* d_F, int F_T, const void* d_f,
                          void* d_x, void* d_u, void* d_ws, size_t ws_bytes, void* stream);

/*
 * DiffLqr.backward (differentiable_lqr.py:78-142) for the shared batch.  Needs d_ws of a dmpc_lqr_solve_shared call on the
 * same C, F, and its d_x, d_u.  d_gx[T,B,n], d_gu[T,B,m] may be NULL (zeros).
 * Outputs: per element d_dx0[B,n] d_dc[T,B,s] d_df[T-1,B,n] (nullable); shared d_dC[T,s,s] = sum_b dC_b (:128) and
 * d_dF[F_T,n,s] = sum_b dF_b (:130-131; row T-1 zero when F_T == T), summed in a fixed order (deterministic).
 * DMPC_ADJ_STRICT_REFERENCE reproduces quirks Q1 and Q2 as dmpc_lqr_adjoint does.
 */
int dmpc_lqr_adjoint_shared(dmpc_handle h, int dtype, int T, int B, int n, int m,
                            const void* d_C, const void* d_c, const void* d_F, int F_T,
                            const void* d_x, const void* d_u, const void* d_gx, const void* d_gu,
                            void* d_ws, size_t ws_bytes,
                            void* d_dx0, void* d_dC, void* d_dc, void* d_dF, void* d_df, int flags, void* stream);

/* ---- the same with c shared by the batch as well (LqrNet_cost_dx, differentiable_lqr.py:237-248, and LqrNet on a batch
 *      whose c does not vary, :186-198: one learned c broadcast over [T, B] with util.expand_time_batch) ----------------- */
/* bits of `share` */
enum { DMPC_SHARE_C = 1 };  /* d_c is [T,s], one block per step for every element; d_dc is [T,s] = sum_b dc_b */

/*
 * The three calls above with one more argument, `share`; share = 0 is exactly the call above.  With DMPC_SHARE_C:
 *   - d_c[T,s] replaces the [T,B,s] tensor the reference builds with expand_time_batch (the host never broadcasts it);
 *   - dmpc_lqr_adjoint_shared_ex writes d_dc[T,s] = sum_b dtau_{t,b} (the reference's dc = dtau, :140, summed as the
 *     backward of the broadcast does), in a fixed order (deterministic).  d_dc may be NULL; no per-element dc is written;
 *   - with d_f == NULL as well, every element has the same k_t: the one Riccati sweep computes it and the forward only
 *     rolls the batch out (no per-element vector sweep).  With d_f given, the vector sweep runs on the shared c.
 * f stays per element (d_f[T-1,B,n]) or NULL.  The workspace size depends on `share` (it holds a [T,B,s] staging region
 * for the adjoint with DMPC_SHARE_C): size it with dmpc_lqr_shared_workspace_bytes_ex and the same `share`.
 * Unknown bits in `share`: DMPC_ERR_UNSUPPORTED.
 */
int dmpc_lqr_shared_workspace_bytes_ex(int dtype, int T, int B, int n, int m, int share, size_t* bytes);

int dmpc_lqr_solve_shared_ex(dmpc_handle h, int dtype, int T, int B, int n, int m,
                             const void* d_x0, const void* d_C, const void* d_c, const void* d_F, int F_T, const void* d_f,
                             void* d_x, void* d_u, void* d_ws, size_t ws_bytes, int share, void* stream);

int dmpc_lqr_adjoint_shared_ex(dmpc_handle h, int dtype, int T, int B, int n, int m,
                               const void* d_C, const void* d_c, const void* d_F, int F_T,
                               const void* d_x, const void* d_u, const void* d_gx, const void* d_gu,
                               void* d_ws, size_t ws_bytes,
                               void* d_dx0, void* d_dC, void* d_dc, void* d_dF, void* d_df, int flags, int share,
                               void* stream);

/* ---- PNQP (replaces PNQP, mpc/pnqp.py:37-201) ---------------------------------------------- */
/*
 * Batched projected-Newton box QP: min 0.5 x^T H x + q^T x  s.t. lower <= x <= upper.
 *   d_H[B,m,m] d_q,d_lower,d_upper[B,m]; d_x_init[B,m] or NULL (pnqp.py:75-93).
 * Outputs: d_x[B,m]; d_LU[B,m,m] + d_piv[B,m] (int32, 1-based LAPACK pivots) = factorisation of the
 * last masked Hessian (+1e-11 I) (for m == 1, d_LU is the scalar H_f the reference returns);
 * d_free[B,m] (1.0 = free, 0.0 = clamped, the reference's Index_f); d_iters[B] (int32, the
 * reference's `i`; identical for all elements under DMPC_COUPLING_BATCH); d_flags[B] (nullable).
 * lower <= upper is the caller's contract (the facade asserts it, pnqp.py:64).
 */
int dmpc_pnqp(dmpc_handle h, int dtype, int B, int m,
              const void* d_H, const void* d_q, const void* d_lower, const void* d_upper, const void* d_x_init,
              int n_iter, int coupling,
              void* d_x, void* d_LU, void* d_piv, void* d_free, void* d_iters, void* d_flags, void* stream);

/* ---- MPC step (replaces MPCstep, mpc/mpc_step.py:33-460) ------------------------------------ */
/*
 * MPCstep.forward (mpc_step.py:288-328): Taylor shift of c (need_expand), backward_rec with one
 * PNQP per timestep (:70-173), forward_rec line search through the TRUE dynamics and cost (:175-286),
 * fused in one launch.
 *   model:      d_C[T,B,s,s] d_c[T,B,s] d_F[F_T,B,n,s] d_f[T-1,B,n] (NULL = None; ignored when need_expand)
 *   nominal:    d_x_nom[T,B,n] (current_states)  d_u_nom[T,B,m] (controls)
 *   bounds:     d_lower, d_upper [T,B,m]   (scalar bounds are broadcast by the caller, box_ddp.py:68-90)
 *   true cost:  QuadCost d_tC[T,B,s,s], d_tc[T,B,s]  (may alias d_C, d_c)
 *   true dyn:   DMPC_DYN_LINEAR with d_tF[>=T-1,B,n,s], d_tf (nullable)  or
 *               DMPC_DYN_PENDULUM with h_dyn_params = {g, m, l, dt, max_torque} (env_dx/pendulum.py:31-102; dt and
 *               max_torque <= 0 mean the reference's 0.05 and 2.0); five doubles are read
 * max_ls_trials: cap of the per-element line search (0: 64); < 0: backward_rec ONLY - the call writes d_Ks, d_ks, d_n_qp,
 *   d_free and d_flags and returns, so that a host whose true cost / dynamics are Python callables (reference
 *   mpc_step.py:237-251 calls them inside forward_rec) can run the line search itself; the true-cost / true-dynamics /
 *   trajectory arguments may then be NULL.
 * Outputs: d_x[T,B,n] d_u[T,B,m]; gains d_Ks[T,B,m,n] d_ks[T,B,m]; d_u_first[T,B,m] = controls of the
 * alpha=1 pass (for full_du_norm, :260-263); d_objs[T,B]; d_costs[B]; d_old_costs[B] (nullable);
 * d_alphas[B]; d_n_qp[T,B] int32 (1 + PNQP iterations); d_free[T,B,m] uint8; d_n_ls[B] int32
 * (line-search passes run: the accepted pass, or max_ls_trials on an element whose line search hit the cap - that one
 * carries DMPC_FLAG_LS_CAPPED and its alpha is the one of the last pass); d_flags[B] int32 (dmpc_elem_flag bits).
 * max_ls_trials caps the per-element line search (the reference's loop has no effective cap, Q5).
 * Shapes: any T, B >= 1 and 1 <= m <= 32, 1 <= n <= 128 in both dtypes.  Systems whose per-element layout does not fit one
 * CTA's shared memory (fp64 from n = 57 at m = 8) run on host-stepped large-system kernels (DESIGN.md §4.9): element
 * coupling and DMPC_DYN_LINEAR only (DMPC_COUPLING_BATCH there returns DMPC_ERR_UNSUPPORTED), every product in fp64, fp32
 * tensors widened on load and rounded once on store; outside the range DMPC_ERR_UNSUPPORTED, nothing launched.
 */
int dmpc_mpc_step_forward(dmpc_handle h, int dtype, int T, int B, int n, int m,
                          const void* d_C, const void* d_c, const void* d_F, int F_T, const void* d_f,
                          const void* d_x_nom, const void* d_u_nom, const void* d_lower, const void* d_upper,
                          const void* d_tC, const void* d_tc, int dynamics, const void* d_tF, const void* d_tf,
                          const double* h_dyn_params, double ls_decay, int max_ls_trials, int need_expand,
                          int coupling,
                          void* d_x, void* d_u, void* d_Ks, void* d_ks, void* d_u_first, void* d_objs,
                          void* d_costs, void* d_old_costs, void* d_alphas, void* d_n_qp, void* d_free,
                          void* d_n_ls, void* d_flags, void* stream);

/*
 * MPCstep.backward (mpc_step.py:330-460) incl. LQR_active (mpc/active_constrained_lqr.py:67-193).
 *   d_x, d_u = the step's outputs (retained); d_gx[T,B,n], d_gu[T,B,m] = upstream grads (NULL = zeros).
 * Workspaces (caller-owned): d_ws_Ks[T,B,m,n] d_ws_ks[T,B,m] d_ws_dtau[T,B,s] d_active[T,B,m] uint8
 * (d_active doubles as an output: the active set used).
 * Outputs: d_dx0[B,n] d_dC[T,B,s,s] d_dc[T,B,s] d_dF[F_T,B,n,s] (row T-1 zero-filled when F_T == T, Q8)
 * d_df[T-1,B,n] (NULL when f_hat is None).
 * Shapes: as dmpc_mpc_step_forward.  The masked solve and the adjoint each take the large-system kernels where their own
 * per-element kernel does not fit (DESIGN.md §4.9); outside n <= 128, m <= 32 DMPC_ERR_UNSUPPORTED, nothing launched.
 */
int dmpc_mpc_step_backward(dmpc_handle h, int dtype, int T, int B, int n, int m,
                           const void* d_C, const void* d_c, const void* d_F, int F_T,
                           const void* d_x, const void* d_u, const void* d_lower, const void* d_upper,
                           const void* d_gx, const void* d_gu,
                           void* d_ws_Ks, void* d_ws_ks, void* d_ws_dtau, void* d_active,
                           void* d_dx0, void* d_dC, void* d_dc, void* d_dF, void* d_df, void* stream);

/*
 * LQR_active.solve_recursion (mpc/active_constrained_lqr.py:195-202) on its own:
 * d_active[T,B,m] uint8 = u_zero_Index.  Same tensors as dmpc_lqr_solve.
 * Shapes: as dmpc_lqr_solve (the large-system kernels apply the masks where the per-element layout does not fit).
 */
int dmpc_lqr_active_solve(dmpc_handle h, int dtype, int T, int B, int n, int m,
                          const void* d_x0, const void* d_C, const void* d_c, const void* d_F, int F_T,
                          const void* d_f, const void* d_active,
                          void* d_x, void* d_u, void* d_Ks, void* d_ks, void* stream);

/* ---- trajectory helpers (util.get_traj util.py:201-236; PendulumDx env_dx/pendulum.py:65-102;
 *      linearize_dynamics mpc/approximate.py:77-119 for the pendulum) -------------------------- */
/*
 * Roll x_{t+1} = dyn(x_t, u_t) from d_x0 under d_u[T,B,m] -> d_x[T,B,n].  For DMPC_DYN_PENDULUM
 * (n=3, m=1) d_Fout[T-1,B,3,4] / d_fout[T-1,B,3] (nullable) receive the analytic linearisation.
 * Shapes: DMPC_DYN_LINEAR at any n <= 128, m <= 32 (past n + m = 64 one CTA per element, with the row-dot order and
 * rounding of the large-system line search, so get_traj of its accepted controls reproduces its trajectory bit for bit).
 */
int dmpc_get_traj(dmpc_handle h, int dtype, int T, int B, int n, int m, int dynamics,
                  const void* d_x0, const void* d_u, const void* d_F, const void* d_f,
                  const double* h_dyn_params, void* d_x, void* d_Fout, void* d_fout, void* stream);

/*
 * BoxDDP.forward (mpc/box_ddp.py:93-291): the box-constrained iLQR outer loop, device resident.
 * Per iteration: rollout of the nominal controls + linearisation (util.get_traj :123,
 * approximate.linearize_dynamics :126-131 - analytic for the pendulum), one MPCstep.forward (:173-193),
 * per-element best trajectory (:195-209, costs <= best + best_cost_eps), then the reference's batch-global exits:
 * max(full_du_norm) < eps -> converged (:223); the shared n_not_improved counter > not_improved_lim (:227).
 * full_du_norm keeps the reference's batch-mixing reshape (mpc_step.py:261-263) with numpy's summation order.
 * The host reads one 32-byte status record per iteration; all tensors stay in HBM.
 *   inputs : d_x_init[B,n], d_C[T,B,s,s], d_c[T,B,s] (the QuadCost, also the true cost), d_lower/d_upper[T,B,m],
 *            dynamics selector (+ d_F[F_T,B,n,s], d_f[T-1,B,n] or NULL for DMPC_DYN_LINEAR; h_dyn_params (g,m,l)
 *            for DMPC_DYN_PENDULUM), d_u_init[T,B,m] (not modified)
 *   outputs: d_x_best[T,B,n], d_u_best[T,B,m], d_costs_best[B], d_du_best[B] (full_du_norm at the best step),
 *            d_du_last[B] (of the last step; may be NULL), d_F_lin[T-1,B,n,s], d_f_lin[T-1,B,n] = linearisation
 *            at the returned point (pendulum only, :235-242; NULL for linear dynamics),
 *            *h_n_iter, *h_status (DMPC_BOXDDP_*), *h_flags (OR of the per-element DMPC_FLAG_* over all steps)
 *   d_ws   : caller-owned workspace of dmpc_boxddp_workspace_bytes() bytes
 * Returns DMPC_ERR_NONFINITE where the reference's NaN asserts would fire (mpc_step.py:284-285).
 * Shapes: those of dmpc_mpc_step_forward; with DMPC_DYN_LINEAR every n <= 128, m <= 32 (element coupling past the
 * per-element kernels, DESIGN.md §4.9).
 */
typedef struct {
  double eps;               /* box_ddp.py:27 eps */
  double best_cost_eps;
  double ls_decay;          /* line_search_decay */
  int not_improved_lim;
  int max_iter;
  int max_ls_trials;        /* safety cap of the per-element line search (<= 0: 64) */
  int coupling;             /* DMPC_COUPLING_* */
  int poll_every;           /* iterations enqueued between two reads of the device-side loop record (<= 0: 8); the exit
                               tests themselves run on the device after every iteration, so the result does not depend on it */
} dmpc_boxddp_opts;

enum { DMPC_BOXDDP_MAX_ITER = 0, DMPC_BOXDDP_CONVERGED = 1, DMPC_BOXDDP_NOT_IMPROVED = 2 };

int dmpc_boxddp_workspace_bytes(int dtype, int T, int B, int n, int m, size_t* bytes);
int dmpc_boxddp_solve(dmpc_handle h, int dtype, int T, int B, int n, int m,
                      const void* d_x_init, const void* d_C, const void* d_c,
                      const void* d_lower, const void* d_upper,
                      int dynamics, const void* d_F, int F_T, const void* d_f, const double* h_dyn_params,
                      const void* d_u_init, const dmpc_boxddp_opts* opts, void* d_ws, size_t ws_bytes,
                      void* d_x_best, void* d_u_best, void* d_costs_best, void* d_du_best, void* d_du_last,
                      void* d_F_lin, void* d_f_lin, int* h_n_iter, int* h_status, int* h_flags, void* stream);

/*
 * Fused parameter-gradient reduction (SURVEY 8f-2): the backward of util.expand_time_batch (util.py:361-377 - the
 * sum over T and B that every shared-parameter model applies to dC, dc, dF, df: LqrNet differentiable_lqr.py:186-198,
 * MpcNet mpc_net.py:78-86, IL_Env.mpc il_env.py:120-129) is done inside the adjoint kernel, so the [T,B,s,s] /
 * [T,B,n,s] gradient tensors are never written.  Same arguments as dmpc_lqr_adjoint / dmpc_mpc_step_backward except:
 *   d_ws_dtau[T,B,s] and d_ws_partials[B * dmpc_reduced_grad_elems(n,m)] are caller-owned workspaces;
 *   d_sums[dmpc_reduced_grad_elems(n,m)] = (sum dC [s,s] | sum dc [s] | sum dF [n,s] | sum df [n]) over (t,b),
 *   summed in a fixed order (deterministic); d_dx0[B,n] stays per element.
 * The result feeds the NCCL all-reduce of the training step directly (a few hundred doubles per rank).
 * dmpc_lqr_adjoint_reduced covers the shapes of dmpc_lqr_adjoint (its per-element sums need more shared memory, so it moves
 * to the large-system kernels first: fp64 (64, 8) already does).  dmpc_mpc_step_backward_reduced covers the shapes of
 * dmpc_mpc_step_backward the same way.
 */
/* util.expand_time_batch on the device (reference util.py:361-377; callers differentiable_lqr.py:186-198,
 * mpc_net.py:78-80, il_env.py:120-129): d_dst[t][b][0..count) = d_src[0..count) for t < T, b < B.  The forward half of the
 * shared-parameter path; its backward is the fused (T,B)-sum of dmpc_*_reduced below. */
int dmpc_expand_time_batch(dmpc_handle h, int dtype, int T, int B, int count, const void* d_src, void* d_dst, void* stream);

/* Warm-start cache of controls in HBM (reference env_dx/il_exp.py:215-257: train_warmstart[n_samples][T][m] indexed by the
 * sample ids of the minibatch; IL_Env.mpc transposes the gathered rows to [T][B][m], il_env.py:113).
 *   take: d_u[t][b][:] = d_cache[d_idx[b]][t][:]      put: d_cache[d_idx[b]][t][:] = d_u[t][b][:]
 * d_idx[B] int32 sample ids; ids outside [0, n_samples) read as zeros / are not written.  With dmpc_boxddp_solve taking
 * d_u_init and returning d_u_best on the device, a training loop keeps its warm starts resident (no PCIe round trip). */
int dmpc_warmstart_take(dmpc_handle h, int dtype, int T, int B, int m, int n_samples, const void* d_cache,
                        const int32_t* d_idx, void* d_u, void* stream);
int dmpc_warmstart_put(dmpc_handle h, int dtype, int T, int B, int m, int n_samples, void* d_cache,
                       const int32_t* d_idx, const void* d_u, void* stream);

size_t dmpc_reduced_grad_elems(int n, int m);
int dmpc_lqr_adjoint_reduced(dmpc_handle h, int dtype, int T, int B, int n, int m,
                             const void* d_C, const void* d_c, const void* d_F, const void* d_x, const void* d_u,
                             const void* d_gx, const void* d_gu, const void* d_Ks, const void* d_fac,
                             void* d_ws_dtau, void* d_ws_partials, void* d_dx0, void* d_sums, int flags, void* stream);
int dmpc_mpc_step_backward_reduced(dmpc_handle h, int dtype, int T, int B, int n, int m,
                                   const void* d_C, const void* d_c, const void* d_F, int F_T,
                                   const void* d_x, const void* d_u, const void* d_lower, const void* d_upper,
                                   const void* d_gx, const void* d_gu,
                                   void* d_ws_Ks, void* d_ws_ks, void* d_ws_dtau, void* d_active,
                                   void* d_ws_partials, void* d_dx0, void* d_sums, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DIFFMPC_B200_H */
