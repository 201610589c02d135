// extern "C" boundary of libdiffmpc_b200.so (declared in include/diffmpc_b200.h).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include "../../include/diffmpc_b200.h"
#include "launch.h"
#include "mpc_launch.h"
#include "boxddp_kernels.cuh"

struct dmpc_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  long long launches = 0;
  std::string err;
  void* pinned = nullptr;        // small page-locked scratch (BoxDDP control records), allocated on first use
  cudaEvent_t ev[2] = {nullptr, nullptr};
};

using namespace dmpc;

namespace {
inline cudaStream_t pick(dmpc_handle h, void* s) { return s ? (cudaStream_t)s : h->stream; }
inline int fail(dmpc_handle h, int code, const char* what) {
  if (h) h->err = what;
  return code;
}
inline int cuda_fail(dmpc_handle h, cudaError_t e, const char* where) {
  if (h) h->err = std::string(where) + ": " + cudaGetErrorString(e);
  return DMPC_ERR_CUDA;
}
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return cuda_fail(h, e_, #call); } while (0)
inline int set_dev(dmpc_handle h) { return cudaSetDevice(h->device) == cudaSuccess ? 0 : DMPC_ERR_CUDA; }
// fn(double{}) or fn(float{}): the typed implementation of an entry point
template <class Fn>
int by_dtype(dmpc_handle h, int dtype, Fn fn) {
  if (dtype == DMPC_F64) return fn(double{});
  if (dtype == DMPC_F32) return fn(float{});
  return fail(h, DMPC_ERR_UNSUPPORTED, "dtype");
}
inline size_t fac_elems_per_step(int n, int m) { return (size_t)(m * m + n * m); }
const char* kLargeUnsupported = "shape beyond the per-element kernels' shared memory and the large-system kernels' range (n <= 128, m <= 32)";
}  // namespace

template <typename R>
static int lqr_solve_impl(dmpc_handle h, int T, int B, int n, int m, const void* x0, const void* C, const void* c,
                          const void* F, const void* f, void* x, void* u, void* Ks, void* ks, void* fac, int flags,
                          cudaStream_t st) {
  LqrParams<R> p;
  memset(&p, 0, sizeof(p));
  p.T = T; p.B = B; p.n = n; p.m = m;
  p.flags = 0;
  if (flags & DMPC_LQR_FACTOR) p.flags |= LQR_DO_FACTOR;
  if (flags & DMPC_LQR_ROLLOUT) p.flags |= LQR_DO_ROLLOUT;
  if ((flags & DMPC_LQR_SAVE_FAC) && fac) p.flags |= LQR_SAVE_FAC;
  p.x0 = (const R*)x0; p.C = (const R*)C; p.c = (const R*)c; p.F = (const R*)F; p.f = (const R*)f;
  p.c_scale = R(1);
  p.x = (R*)x; p.u = (R*)u; p.Ks = (R*)Ks; p.ks = (R*)ks; p.fac = (R*)fac;
  if ((p.flags & LQR_SAVE_FAC) && adjoint_fused_available<R>(n, m)) p.Vsave = (R*)fac + (size_t)T * B * fac_elems_per_step(n, m);
  int rc = launch_lqr_solve<R>(p, st, &h->launches);
  if (rc) h->err = rc == DMPC_ERR_UNSUPPORTED ? std::string("lqr_solve: ") + kLargeUnsupported : "lqr_solve launch failed";
  return rc;
}

template <typename R>
static int lqr_adjoint_impl(dmpc_handle h, int T, int B, int n, int m, const void* C, const void* c, const void* F,
                            const void* x, const void* u, const void* gx, const void* gu, const void* Ks,
                            const void* fac, void* dx0, void* dC, void* dc, void* dF, void* df, int flags,
                            cudaStream_t st, void* partials = nullptr, void* sums = nullptr) {
  DtauParams<R> d;
  memset(&d, 0, sizeof(d));
  d.T = T; d.B = B; d.n = n; d.m = m;
  d.F = (const R*)F; d.gx = (const R*)gx; d.gu = (const R*)gu; d.Ks = (const R*)Ks; d.fac = (const R*)fac;
  d.dc = (R*)dc;
  // two-sweep adjoint only.  Full gradients: v'_t is parked in the df output buffer (row t-1) and in dx0 (t = 0) between
  // the sweeps.  Fused (T,B)-reduction: dc is a workspace, v'_t travels in its first n entries, nothing but dx0 and the
  // per-element partial sums is written.
  d.vp = partials ? nullptr : (R*)df; d.dx0 = (R*)dx0;
  const int qflags = (flags & DMPC_ADJ_STRICT_REFERENCE) ? (ADJ_QUIRK_DC | ADJ_QUIRK_DF) : 0;
  AdjFusedParams<R> f;
  memset(&f, 0, sizeof(f));
  f.T = T; f.B = B; f.n = n; f.m = m; f.flags = qflags;
  f.F = (const R*)F; f.Ks = (const R*)Ks; f.Vv = (const R*)fac + (size_t)T * B * fac_elems_per_step(n, m);
  f.x = (const R*)x; f.u = (const R*)u; f.vp = (const R*)df; f.dx0 = (const R*)dx0;
  f.dc = (R*)dc; f.dC = (R*)dC; f.dF = (R*)dF; f.df = (R*)df; f.red = (R*)partials;
  AdjOutParams<R> a;
  memset(&a, 0, sizeof(a));
  a.T = T; a.B = B; a.n = n; a.m = m; a.F_T = T - 1; a.flags = qflags;
  a.C = (const R*)C; a.c = (const R*)c; a.F = (const R*)F; a.x = (const R*)x; a.u = (const R*)u;
  a.dtau = (const R*)dc; a.gx = (const R*)gx; a.gu = (const R*)gu;
  a.dx0 = (R*)dx0; a.dC = (R*)dC; a.dc = (R*)dc; a.dF = (R*)dF; a.df = (R*)df;
  if (partials) { a.flags |= ADJ_REDUCE_TB; a.red = (R*)partials; }
  const int stage = (flags & DMPC_ADJ_STAGE_OUT_ONLY) ? 2 : ((flags & DMPC_ADJ_STAGE_DTAU_ONLY) ? 1 : 0);
  const char* failed = nullptr;
  const int rc = launch_lqr_adjoint<R>(d, f, a, stage, (R*)sums, st, &h->launches, &failed);
  if (rc) h->err = failed ? failed : std::string("lqr_adjoint: ") + kLargeUnsupported;
  return rc;
}

template <typename R>
static int mpc_forward_impl(dmpc_handle h, int T, int B, int n, int m, const void* C, const void* c, const void* F,
                            int F_T, const void* f, const void* x_nom, const void* u_nom, const void* lo,
                            const void* hi, const void* tC, const void* tc, int dynamics, const void* tF,
                            const void* tf, const double* dynp, double ls_decay, int max_ls_trials, int need_expand,
                            int coupling, void* x, void* u, void* Ks, void* ks, void* u_first, void* objs,
                            void* costs, void* old_costs, void* alphas, void* n_qp, void* free_m, void* n_ls,
                            void* flags, cudaStream_t st, const int* skip = nullptr) {
  MpcFwdParams<R> p;
  memset(&p, 0, sizeof(p));
  p.T = T; p.B = B; p.n = n; p.m = m; p.F_T = F_T; p.need_expand = need_expand; p.dynamics = dynamics;
  p.coupling = coupling; p.max_ls_trials = max_ls_trials > 0 ? max_ls_trials : (max_ls_trials < 0 ? -1 : 64); p.n_qp_iter = 20;
  p.ls_decay = (R)ls_decay;
  p.C = (const R*)C; p.c = (const R*)c; p.F = (const R*)F; p.f = (const R*)f;
  p.x_nom = (const R*)x_nom; p.u_nom = (const R*)u_nom; p.lo = (const R*)lo; p.hi = (const R*)hi;
  p.tC = (const R*)tC; p.tc = (const R*)tc; p.tF = (const R*)tF; p.tf = (const R*)tf;
  for (int i = 0; i < 5; ++i) p.dyn_params[i] = dynp ? (R)dynp[i] : R(0);
  p.x = (R*)x; p.u = (R*)u; p.Ks = (R*)Ks; p.ks = (R*)ks; p.u_first = (R*)u_first; p.objs = (R*)objs;
  p.costs = (R*)costs; p.old_costs = (R*)old_costs; p.alphas = (R*)alphas; p.n_qp = (int*)n_qp;
  p.free_mask = (unsigned char*)free_m; p.n_ls = (int*)n_ls; p.flags = (int*)flags; p.skip = skip;
  int rc = launch_mpc_forward<R>(p, st, &h->launches);
  if (rc) h->err = rc == DMPC_ERR_UNSUPPORTED ? "mpc_step_forward: unsupported shape (n <= 128, m <= 32) or batch coupling (the batch must fit one CTA or cluster, and past the per-element kernels' shared memory only element coupling runs)" : "mpc_step_forward launch failed";
  return rc;
}

template <typename R>
static int mpc_backward_impl(dmpc_handle h, int T, int B, int n, int m, const void* C, const void* c, const void* F,
                             int F_T, const void* x, const void* u, const void* lo, const void* hi, const void* gx,
                             const void* gu, void* wsK, void* wsk, void* wsd, void* act, void* dx0, void* dC,
                             void* dc, void* dF, void* df, cudaStream_t st, void* partials = nullptr,
                             void* sums = nullptr) {
  // The masked solve and the adjoint each take the large-system kernels where their own per-element kernel does not fit.
  // Outside the large-system range (n <= 128, m <= 32) at least the masked solve would not run: at m > 32 it is sent to
  // the large-system kernels, and at n > 128 one element's lqr_layout exceeds kMaxSmem in either dtype (at (129, 1):
  // 465 KiB in fp32, 929 KiB in fp64, against 227 KiB).  Refusing those shapes here launches nothing, not even
  // active_mask_kernel.
  if (!lqr_large_shape_ok(n, m)) return fail(h, DMPC_ERR_UNSUPPORTED, (std::string("mpc_step_backward: ") + kLargeUnsupported).c_str());
  int rc = launch_active_mask<R>((const R*)u, (const R*)lo, (const R*)hi, (unsigned char*)act, (size_t)T * B * m, st, &h->launches);
  if (rc) { h->err = "active_mask launch failed"; return rc; }
  if (cudaMemsetAsync(dx0, 0, (size_t)B * n * sizeof(R), st) != cudaSuccess) return DMPC_ERR_CUDA;
  LqrParams<R> p;
  memset(&p, 0, sizeof(p));
  p.T = T; p.B = B; p.n = n; p.m = m;
  p.flags = LQR_DO_FACTOR | LQR_DO_ROLLOUT | LQR_MASKED;
  p.x0 = (const R*)dx0;                       // zeros (mpc_step.py:365)
  p.C = (const R*)C; p.c = nullptr; p.cx = (const R*)gx; p.cu = (const R*)gu; p.c_scale = R(-1);   // c := -d_taus (:374)
  p.F = (const R*)F; p.f = nullptr; p.active = (const unsigned char*)act;
  p.Ks = (R*)wsK; p.ks = (R*)wsk; p.tau_out = (R*)wsd;
  rc = launch_lqr_solve<R>(p, st, &h->launches);
  if (rc) { h->err = "lqr_active launch failed"; return rc; }
  AdjOutParams<R> a;
  memset(&a, 0, sizeof(a));
  a.T = T; a.B = B; a.n = n; a.m = m; a.F_T = F_T;
  a.flags = ADJ_NEGATE | ADJ_NEG_RHS;
  a.C = (const R*)C; a.c = (const R*)c; a.F = (const R*)F; a.x = (const R*)x; a.u = (const R*)u;
  a.dtau = (const R*)wsd; a.gx = (const R*)gx; a.gu = (const R*)gu;
  a.dx0 = (R*)dx0; a.dC = (R*)dC; a.dc = (R*)dc; a.dF = (R*)dF; a.df = (R*)df;
  if (partials) { a.flags |= ADJ_REDUCE_TB; a.red = (R*)partials; }
  const char* failed = nullptr;
  rc = launch_adjoint_out<R>(a, (R*)sums, st, &h->launches, &failed);
  if (rc) h->err = failed;
  return rc;
}

template <typename R>
static int lqr_active_impl(dmpc_handle h, int T, int B, int n, int m, const void* x0, const void* C, const void* c,
                           const void* F, const void* f, const void* act, void* x, void* u, void* Ks, void* ks,
                           cudaStream_t st) {
  LqrParams<R> p;
  memset(&p, 0, sizeof(p));
  p.T = T; p.B = B; p.n = n; p.m = m;
  p.flags = LQR_DO_FACTOR | LQR_DO_ROLLOUT | LQR_MASKED;
  p.x0 = (const R*)x0; p.C = (const R*)C; p.c = (const R*)c; p.c_scale = R(1); p.F = (const R*)F; p.f = (const R*)f;
  p.active = (const unsigned char*)act; p.x = (R*)x; p.u = (R*)u; p.Ks = (R*)Ks; p.ks = (R*)ks;
  int rc = launch_lqr_solve<R>(p, st, &h->launches);
  if (rc) h->err = rc == DMPC_ERR_UNSUPPORTED ? std::string("lqr_active: ") + kLargeUnsupported : "lqr_active launch failed";
  return rc;
}

template <typename R>
static int pnqp_impl(dmpc_handle h, int B, int m, const void* H, const void* q, const void* lo, const void* hi,
                     const void* xi, int n_iter, int coupling, void* x, void* LU, void* piv, void* fr, void* it,
                     void* fl, cudaStream_t st) {
  PnqpParams<R> p;
  memset(&p, 0, sizeof(p));
  p.B = B; p.m = m; p.n_iter = n_iter; p.coupling = coupling;
  p.H = (const R*)H; p.q = (const R*)q; p.lo = (const R*)lo; p.hi = (const R*)hi; p.x_init = (const R*)xi;
  p.x = (R*)x; p.LU = (R*)LU; p.piv = (int*)piv; p.free_out = (R*)fr; p.iters = (int*)it; p.flags = (int*)fl;
  int rc = launch_pnqp<R>(p, st, &h->launches);
  if (rc) h->err = rc == DMPC_ERR_UNSUPPORTED ? "pnqp: unsupported (m > 32, or batch coupling with the batch not in one CTA)" : "pnqp launch failed";
  return rc;
}

template <typename R>
static int traj_impl(dmpc_handle h, int T, int B, int n, int m, int dynamics, const void* x0, const void* u,
                     const void* F, const void* f, const double* dynp, void* x, void* Fo, void* fo, cudaStream_t st,
                     const int* skip = nullptr) {
  TrajParams<R> p;
  memset(&p, 0, sizeof(p));
  p.T = T; p.B = B; p.n = n; p.m = m; p.dynamics = dynamics;
  p.x0 = (const R*)x0; p.u = (const R*)u; p.F = (const R*)F; p.f = (const R*)f;
  for (int i = 0; i < 5; ++i) p.dyn_params[i] = dynp ? (R)dynp[i] : R(0);
  p.x = (R*)x; p.Fout = (R*)Fo; p.fout = (R*)fo; p.skip = skip;
  int rc = launch_traj<R>(p, st, &h->launches);
  if (rc) h->err = rc == DMPC_ERR_UNSUPPORTED ? std::string("get_traj: ") + kLargeUnsupported : "get_traj launch failed";
  return rc;
}

extern "C" int dmpc_get_traj(dmpc_handle, int, int, int, int, int, int, const void*, const void*, const void*, const void*, const double*, void*, void*, void*, void*);

// ------------------------------------------------------------------------------------------------
// Device-resident BoxDDP outer loop (reference mpc/box_ddp.py:121-230).  Everything stays in HBM; per iteration the
// host reads one 32-byte status record to apply the reference's (batch-global) exit tests.
namespace {
struct BoxWs {
  size_t x_nom, u_a, u_b, x_new, Ks, ks, u_first, objs, costs, old, alphas, du, n_qp, free_m, n_ls, flags, mask, dynp, status, ctl, total;
};
inline BoxWs box_ws(size_t w, int T, int B, int n, int m) {
  BoxWs L; size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o = al256(o + bytes); return at; };
  L.x_nom = take(w * T * B * n); L.u_a = take(w * T * B * m); L.u_b = take(w * T * B * m); L.x_new = take(w * T * B * n);
  L.Ks = take(w * T * B * m * n); L.ks = take(w * T * B * m); L.u_first = take(w * T * B * m); L.objs = take(w * T * B);
  L.costs = take(w * B); L.old = take(w * B); L.alphas = take(w * B); L.du = take(w * B);
  L.n_qp = take(sizeof(int) * (size_t)T * B); L.free_m = take((size_t)T * B * m); L.n_ls = take(sizeof(int) * (size_t)B);
  L.flags = take(sizeof(int) * (size_t)B); L.mask = take((size_t)B); L.dynp = take(w * 5); L.status = take(sizeof(BoxDdpStatus)); L.ctl = take(sizeof(BoxDdpCtl));
  L.total = o;
  return L;
}
}  // namespace

template <typename R>
static int boxddp_impl(dmpc_handle h, int dtype, int T, int B, int n, int m, const void* x_init, const void* C, const void* c,
                       const void* lo, const void* hi, int dynamics, const void* F, int F_T, const void* f,
                       const double* dynp, const void* u_init, const dmpc_boxddp_opts* o, void* ws, void* x_best,
                       void* u_best, void* costs_best, void* du_best, void* du_last, void* F_lin, void* f_lin,
                       int* h_n_iter, int* h_status, int* h_flags, cudaStream_t st) {
  const BoxWs L = box_ws(sizeof(R), T, B, n, m);
  char* w = (char*)ws;
  R* x_nom = (R*)(w + L.x_nom); R* u_cur = (R*)(w + L.u_a); R* u_new = (R*)(w + L.u_b); R* x_new = (R*)(w + L.x_new);
  R* Ks = (R*)(w + L.Ks); R* ks = (R*)(w + L.ks); R* u_first = (R*)(w + L.u_first); R* objs = (R*)(w + L.objs);
  R* costs = (R*)(w + L.costs); R* old = (R*)(w + L.old); R* alphas = (R*)(w + L.alphas); R* du = (R*)(w + L.du);
  int* n_qp = (int*)(w + L.n_qp); unsigned char* free_m = (unsigned char*)(w + L.free_m); int* n_ls = (int*)(w + L.n_ls);
  int* flags = (int*)(w + L.flags); BoxDdpStatus* dst = (BoxDdpStatus*)(w + L.status);
  BoxDdpCtl* dctl = (BoxDdpCtl*)(w + L.ctl);
  const bool pend = dynamics == DMPC_DYN_PENDULUM;
  const size_t ub = sizeof(R) * (size_t)T * B * m;
  CK(cudaMemcpyAsync(u_cur, u_init, ub, cudaMemcpyDeviceToDevice, st));
  CK(cudaMemsetAsync(dst, 0, sizeof(BoxDdpStatus), st));
  CK(cudaMemsetAsync(dctl, 0, sizeof(BoxDdpCtl), st));
  // The loop runs on the device: the exit tests run in the last CTA of boxddp_post_kernel, later iterations see ctl->done and return at
  // once, and the host only reads the control record once per block of `poll` enqueued iterations (no per-iteration sync).
  const int poll = o->poll_every > 0 ? o->poll_every : 8;
  const int tpb = 64, grid = (B + tpb - 1) / tpb;                   // one thread per element: many small CTAs
  const int pgrid = (int)(((size_t)T * B + kPostThreads - 1) / kPostThreads);   // one thread per (t, b)
  unsigned char* mask = (unsigned char*)(w + L.mask);
  R* d_dynp = (R*)(w + L.dynp);
  if (pend) {
    R hp[5];
    for (int i = 0; i < 5; ++i) hp[i] = (R)dynp[i];
    CK(cudaMemcpyAsync(d_dynp, hp, sizeof(hp), cudaMemcpyHostToDevice, st));   // pageable: staged before the call returns
  }
  const int* skip = &dctl->done;
  // Control records come back through page-locked memory and the NEXT block of iterations is enqueued before the host
  // waits for the record of the current one, so the GPU never idles on the host; if the current block raised `done`, the
  // kernels of the block already enqueued see the flag and return at once.
  if (!h->pinned) CK(cudaHostAlloc(&h->pinned, 2 * sizeof(BoxDdpCtl), cudaHostAllocDefault));
  for (int k = 0; k < 2; ++k) if (!h->ev[k]) CK(cudaEventCreateWithFlags(&h->ev[k], cudaEventDisableTiming));
  BoxDdpCtl* hrec = (BoxDdpCtl*)h->pinned;
  BoxDdpCtl hc;
  memset(&hc, 0, sizeof(hc));
  auto enqueue_block = [&](int i0, int slot) -> int {
    const int i1 = i0 + poll < o->max_iter ? i0 + poll : o->max_iter;
    for (int i = i0; i < i1; ++i) {
      // nominal trajectory and linearisation (box_ddp.py:123-131).  Pendulum: after iteration 0 the step's accepted
      // rollout x_new IS get_traj(u_new) and boxddp_post_kernel has linearised it, so no launch is needed here.
      int rc = DMPC_OK;
      if (!pend || i == 0)
        rc = traj_impl<R>(h, T, B, n, m, dynamics, x_init, u_cur, F, f, dynp, x_nom, pend ? F_lin : nullptr,
                          pend ? f_lin : nullptr, st, skip);
      if (rc) return rc;
      rc = mpc_forward_impl<R>(h, T, B, n, m, C, c, pend ? F_lin : F, pend ? T - 1 : F_T, nullptr, x_nom, u_cur, lo, hi, C, c,
                               dynamics, pend ? nullptr : F, pend ? nullptr : f, dynp, o->ls_decay, o->max_ls_trials, 1,
                               o->coupling, x_new, u_new, Ks, ks, u_first, objs, costs, old, alphas, n_qp, free_m, n_ls, flags,
                               st, skip);
      if (rc) return rc;
      boxddp_norm_better_kernel<R><<<grid, tpb, 0, st>>>(T, B, m, i == 0, (R)o->best_cost_eps, u_cur, u_first, costs, flags, du,
                                                         (R*)costs_best, (R*)du_best, mask, dst, skip);
      boxddp_post_kernel<R><<<pgrid, kPostThreads, 0, st>>>(T, B, n, m, x_new, u_new, mask, (R*)x_best, (R*)u_best, d_dynp,
                                                            pend ? (R*)F_lin : nullptr, dst, dctl, i, o->eps, o->not_improved_lim);
      h->launches += 2;
      R* t_ = u_cur; u_cur = u_new; u_new = t_;                     // next nominal controls = this step's controls
      if (pend) { t_ = x_nom; x_nom = x_new; x_new = t_; }          // ... and its rollout is the next nominal trajectory
    }
    if (cudaMemcpyAsync(&hrec[slot], dctl, sizeof(BoxDdpCtl), cudaMemcpyDeviceToHost, st) != cudaSuccess) return DMPC_ERR_CUDA;
    if (cudaEventRecord(h->ev[slot], st) != cudaSuccess) return DMPC_ERR_CUDA;
    return DMPC_OK;
  };
  if (o->max_iter > 0) {
    int rc = enqueue_block(0, 0);
    if (rc) return rc;
    int slot = 0;
    for (int i0 = 0; i0 < o->max_iter; i0 += poll) {
      const bool more = i0 + poll < o->max_iter;
      if (more) { rc = enqueue_block(i0 + poll, slot ^ 1); if (rc) return rc; }
      CK(cudaEventSynchronize(h->ev[slot]));
      hc = hrec[slot];
      if (hc.done) break;
      slot ^= 1;
    }
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
  }
  const int n_iter = hc.n_iter, status = hc.done ? hc.status : DMPC_BOXDDP_MAX_ITER, flags_or = hc.flags_or;
  if (hc.nonfinite) { if (h_n_iter) *h_n_iter = n_iter; return fail(h, DMPC_ERR_NONFINITE, "boxddp: non-finite trajectory, cost or step norm"); }
  if (flags_or & DMPC_FLAG_BAD_BOUNDS) { if (h_n_iter) *h_n_iter = n_iter; return fail(h, DMPC_ERR_BAD_BOUNDS, "boxddp: lower is larger than upper"); }
  if (du_last) CK(cudaMemcpyAsync(du_last, du, sizeof(R) * (size_t)B, cudaMemcpyDeviceToDevice, st));
  if (pend) {   // linearise at the returned point (box_ddp.py:235-242); the rollout itself is scratch
    int rc = dmpc_get_traj(h, dtype, T, B, n, m, dynamics, x_best, u_best, nullptr, nullptr, dynp, x_nom, F_lin, f_lin, st);
    if (rc) return rc;
  }
  CK(cudaStreamSynchronize(st));
  if (h_n_iter) *h_n_iter = n_iter;
  if (h_status) *h_status = status;
  if (h_flags) *h_flags = flags_or;
  return DMPC_OK;
}

// ------------------------------------------------------------------------------------------------
// C and F shared by the batch (lqr_shared_kernels.cuh).  Workspace: the zero c block and outputs of the B = 1 Riccati
// sweep (K_t, k_t, Quu_t^-1 | Qxu_t, V_t | v_t), then one partial record [T][s*s + n*s] per chunk of elements; with
// DMPC_SHARE_C the records carry sum_b dtau_t as well ([T][s*s + n*s + s]) and a [T,B,s] region follows, where the adjoint
// parks k' and dtau between its sweeps (dc being [T,s]).  The caller's pointer is rounded up to 256 bytes first, so the
// sweep's 16-byte copies never depend on the caller's alignment.
namespace {
struct SharedWs { size_t c0, Ks, ks, fac, V, part, park, total; int NB, nchunk; };
inline SharedWs shared_ws(size_t w, int T, int B, int n, int m, int share) {
  SharedWs L; size_t o = 0;
  const size_t s = (size_t)(n + m);
  const bool c_shared = (share & DMPC_SHARE_C) != 0;
  L.NB = lqr_shared_chunk(w, B, n, m, kMaxSmem);
  L.nchunk = L.NB ? (B + L.NB - 1) / L.NB : 0;
  auto take = [&](size_t bytes) { size_t at = o; o = al256(o + bytes); return at; };
  L.c0 = take(w * T * s); L.Ks = take(w * T * m * n); L.ks = take(w * T * m); L.fac = take(w * T * fac_elems_per_step(n, m));
  L.V = take(w * T * (size_t)(n * n + n)); L.part = take(w * (size_t)L.nchunk * T * shared_rec_elems(n, m, c_shared));
  L.park = c_shared ? take(w * (size_t)T * B * s) : 0;
  L.total = o + 256;
  return L;
}
inline char* ws_base(void* ws) { return (char*)al256((size_t)ws); }
}  // namespace

template <typename R>
static int lqr_solve_shared_impl(dmpc_handle h, int T, int B, int n, int m, const void* x0, const void* C, const void* c,
                                 const void* F, int F_T, const void* f, void* x, void* u, void* ws, int share,
                                 cudaStream_t st) {
  const SharedWs W = shared_ws(sizeof(R), T, B, n, m, share);
  const bool c_shared = (share & DMPC_SHARE_C) != 0, roll_only = c_shared && !f;
  char* w = ws_base(ws);
  // The sweep runs on a zero c unless c is shared and f is None: then its k_t is every element's k_t.
  if (!roll_only) CK(cudaMemsetAsync(w + W.c0, 0, sizeof(R) * (size_t)T * (n + m), st));
  LqrParams<R> p;                                    // the matrix sweep: the existing Riccati kernels at B = 1
  memset(&p, 0, sizeof(p));
  p.T = T; p.B = 1; p.n = n; p.m = m; p.flags = LQR_DO_FACTOR | LQR_SAVE_FAC;
  p.C = (const R*)C; p.c = roll_only ? (const R*)c : (const R*)(w + W.c0); p.F = (const R*)F; p.c_scale = R(1);
  p.Ks = (R*)(w + W.Ks); p.ks = (R*)(w + W.ks); p.fac = (R*)(w + W.fac); p.Vsave = (R*)(w + W.V);
  int rc = launch_lqr_solve<R>(p, st, &h->launches);
  if (rc) return fail(h, rc, rc == DMPC_ERR_UNSUPPORTED ? "lqr_solve_shared: no Riccati kernel for this shape" : "lqr_solve_shared: sweep launch failed");
  LqrSharedParams<R> q;
  memset(&q, 0, sizeof(q));
  q.T = T; q.B = B; q.n = n; q.m = m; q.F_T = F_T; q.NB = W.NB; q.c_shared = c_shared;
  q.x0 = (const R*)x0; q.C = (const R*)C; q.c = (const R*)c; q.F = (const R*)F; q.f = (const R*)f;
  q.Ks = p.Ks; q.ks = p.ks; q.fac = p.fac; q.Vsave = p.Vsave; q.x = (R*)x; q.u = (R*)u;
  rc = launch_lqr_shared_fwd<R>(q, st, &h->launches);
  if (rc) h->err = "lqr_solve_shared launch failed";
  return rc;
}

template <typename R>
static int lqr_adjoint_shared_impl(dmpc_handle h, int T, int B, int n, int m, const void* C, const void* c, const void* F,
                                   int F_T, const void* x, const void* u, const void* gx, const void* gu, void* ws,
                                   void* dx0, void* dC, void* dc, void* dF, void* df, int flags, int share,
                                   cudaStream_t st) {
  const SharedWs W = shared_ws(sizeof(R), T, B, n, m, share);
  const bool c_shared = (share & DMPC_SHARE_C) != 0;
  char* w = ws_base(ws);
  LqrSharedParams<R> q;
  memset(&q, 0, sizeof(q));
  q.T = T; q.B = B; q.n = n; q.m = m; q.F_T = F_T; q.NB = W.NB; q.c_shared = c_shared;
  q.flags = (flags & DMPC_ADJ_STRICT_REFERENCE) ? (ADJ_QUIRK_DC | ADJ_QUIRK_DF) : 0;
  q.C = (const R*)C; q.c = (const R*)c; q.F = (const R*)F;
  q.Ks = (const R*)(w + W.Ks); q.fac = (const R*)(w + W.fac); q.Vsave = (const R*)(w + W.V);
  q.x = (R*)x; q.u = (R*)u; q.gx = (const R*)gx; q.gu = (const R*)gu;
  q.dx0 = (R*)dx0; q.dc = (R*)dc; q.df = T > 1 ? (R*)df : nullptr; q.part = (R*)(w + W.part); q.dC = (R*)dC;
  q.park = c_shared ? (R*)(w + W.park) : (R*)dc;
  q.dF = F_T > 0 ? (R*)dF : nullptr;
  const int rc = launch_lqr_shared_adj<R>(q, st, &h->launches);
  if (rc) h->err = "lqr_adjoint_shared launch failed";
  return rc;
}

extern "C" {

int dmpc_version(void) { return 100; }

const char* dmpc_status_string(int s) {
  switch (s) {
    case DMPC_OK: return "ok";
    case DMPC_ERR_BAD_SHAPE: return "bad shape";
    case DMPC_ERR_BAD_BOUNDS: return "lower is larger than upper";
    case DMPC_ERR_NONFINITE: return "non-finite value";
    case DMPC_ERR_CUDA: return "CUDA error";
    case DMPC_ERR_UNSUPPORTED: return "unsupported configuration";
    case DMPC_ERR_NULL: return "null pointer";
    case DMPC_ERR_NO_DEVICE: return "no CUDA device (this library has no CPU fallback)";
    default: return "unknown status";
  }
}

int dmpc_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int dmpc_create(int device, dmpc_handle* out) {
  if (!out) return DMPC_ERR_NULL;
  *out = nullptr;
  int n = dmpc_device_count();
  if (n <= 0 || device < 0 || device >= n) return DMPC_ERR_NO_DEVICE;
  if (cudaSetDevice(device) != cudaSuccess) return DMPC_ERR_CUDA;
  dmpc_ctx* h = new dmpc_ctx();
  h->device = device;
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) { delete h; return DMPC_ERR_CUDA; }
  *out = h;
  return DMPC_OK;
}

int dmpc_destroy(dmpc_handle h) {
  if (!h) return DMPC_ERR_NULL;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamDestroy(h->stream);
  if (h->pinned) cudaFreeHost(h->pinned);
  for (int i = 0; i < 2; ++i) if (h->ev[i]) cudaEventDestroy(h->ev[i]);
  delete h;
  return DMPC_OK;
}

const char* dmpc_last_error(dmpc_handle h) { return h ? h->err.c_str() : "null handle"; }
long long dmpc_launch_count(dmpc_handle h) { return h ? h->launches : 0; }

int dmpc_malloc(dmpc_handle h, size_t bytes, void** d_ptr) {
  if (!h || !d_ptr) return DMPC_ERR_NULL;
  if (set_dev(h)) return DMPC_ERR_CUDA;
  CK(cudaMalloc(d_ptr, bytes ? bytes : 16));
  return DMPC_OK;
}
int dmpc_free(dmpc_handle h, void* d_ptr) {
  if (!h) return DMPC_ERR_NULL;
  if (set_dev(h)) return DMPC_ERR_CUDA;
  CK(cudaFree(d_ptr));
  return DMPC_OK;
}
int dmpc_host_alloc(dmpc_handle h, size_t bytes, void** h_ptr) {
  if (!h || !h_ptr) return DMPC_ERR_NULL;
  if (set_dev(h)) return DMPC_ERR_CUDA;
  CK(cudaHostAlloc(h_ptr, bytes ? bytes : 16, cudaHostAllocDefault));
  return DMPC_OK;
}
int dmpc_host_free(dmpc_handle h, void* h_ptr) {
  if (!h) return DMPC_ERR_NULL;
  CK(cudaFreeHost(h_ptr));
  return DMPC_OK;
}
int dmpc_memcpy_h2d(dmpc_handle h, void* d, const void* s, size_t bytes, void* stream) {
  if (!h) return DMPC_ERR_NULL;
  if (set_dev(h)) return DMPC_ERR_CUDA;
  if (bytes) CK(cudaMemcpyAsync(d, s, bytes, cudaMemcpyHostToDevice, pick(h, stream)));
  return DMPC_OK;
}
int dmpc_memcpy_d2h(dmpc_handle h, void* d, const void* s, size_t bytes, void* stream) {
  if (!h) return DMPC_ERR_NULL;
  if (set_dev(h)) return DMPC_ERR_CUDA;
  if (bytes) CK(cudaMemcpyAsync(d, s, bytes, cudaMemcpyDeviceToHost, pick(h, stream)));
  return DMPC_OK;
}
int dmpc_memset(dmpc_handle h, void* d, int value, size_t bytes, void* stream) {
  if (!h) return DMPC_ERR_NULL;
  if (set_dev(h)) return DMPC_ERR_CUDA;
  if (bytes) CK(cudaMemsetAsync(d, value, bytes, pick(h, stream)));
  return DMPC_OK;
}
int dmpc_sync(dmpc_handle h, void* stream) {
  if (!h) return DMPC_ERR_NULL;
  if (set_dev(h)) return DMPC_ERR_CUDA;
  CK(cudaStreamSynchronize(pick(h, stream)));
  return DMPC_OK;
}

// Quu^-1 | Qxu per (t,b), then V_t | v_t per (t,b) (the value function the two-sweep adjoint needs)
size_t dmpc_lqr_fac_elems(int T, int B, int n, int m) { return (size_t)T * B * (size_t)(m * m + n * m + n * n + n); }

int dmpc_lqr_solve(dmpc_handle h, int dtype, int T, int B, int n, int m, const void* d_x0, const void* d_C,
                   const void* d_c, const void* d_F, int F_T, const void* d_f, void* d_x, void* d_u, void* d_Ks,
                   void* d_ks, void* d_fac, int flags, void* stream) {
  if (!h) return DMPC_ERR_NULL;
  if (T < 1 || B < 1 || n < 1 || m < 1) return fail(h, DMPC_ERR_BAD_SHAPE, "T,B,n,m must be >= 1");
  if (T > 1 && F_T != T - 1 && F_T != T) return fail(h, DMPC_ERR_BAD_SHAPE, "F must have T-1 or T time rows");
  if (!d_Ks || !d_ks) return fail(h, DMPC_ERR_NULL, "Ks/ks buffers are required");
  if ((flags & DMPC_LQR_FACTOR) && (!d_C || !d_c || (T > 1 && !d_F))) return fail(h, DMPC_ERR_NULL, "C,c,F required");
  if ((flags & DMPC_LQR_ROLLOUT) && (!d_x0 || !d_x || !d_u || (T > 1 && !d_F))) return fail(h, DMPC_ERR_NULL, "x0,x,u,F required");
  if (!(flags & (DMPC_LQR_FACTOR | DMPC_LQR_ROLLOUT))) return fail(h, DMPC_ERR_UNSUPPORTED, "nothing to do");
  if (set_dev(h)) return DMPC_ERR_CUDA;
  cudaStream_t st = pick(h, stream);
  return by_dtype(h, dtype, [&](auto r) { return lqr_solve_impl<decltype(r)>(h, T, B, n, m, d_x0, d_C, d_c, d_F, d_f, d_x, d_u, d_Ks, d_ks, d_fac, flags, st); });
}

int dmpc_lqr_adjoint(dmpc_handle h, int dtype, int T, int B, int n, int m, const void* d_C, const void* d_c,
                     const void* d_F, const void* d_x, const void* d_u, const void* d_gx, const void* d_gu,
                     const void* d_Ks, const void* d_fac, void* d_dx0, void* d_dC, void* d_dc, void* d_dF,
                     void* d_df, int flags, void* stream) {
  if (!h) return DMPC_ERR_NULL;
  if (T < 1 || B < 1 || n < 1 || m < 1) return fail(h, DMPC_ERR_BAD_SHAPE, "T,B,n,m must be >= 1");
  if (!d_C || !d_c || !d_x || !d_u || !d_gx || !d_gu || !d_Ks || !d_fac || !d_dx0 || !d_dC || !d_dc || (T > 1 && (!d_F || !d_dF)))
    return fail(h, DMPC_ERR_NULL, "lqr_adjoint: required buffer is NULL");
  if (set_dev(h)) return DMPC_ERR_CUDA;
  cudaStream_t st = pick(h, stream);
  return by_dtype(h, dtype, [&](auto r) { return lqr_adjoint_impl<decltype(r)>(h, T, B, n, m, d_C, d_c, d_F, d_x, d_u, d_gx, d_gu, d_Ks, d_fac, d_dx0, d_dC, d_dc, d_dF, d_df, flags, st); });
}

int dmpc_pnqp(dmpc_handle h, int dtype, int B, int m, const void* d_H, const void* d_q, const void* d_lower,
              const void* d_upper, const void* d_x_init, int n_iter, int coupling, void* d_x, void* d_LU,
              void* d_piv, void* d_free, void* d_iters, void* d_flags, void* stream) {
  if (!h) return DMPC_ERR_NULL;
  if (B < 1 || m < 1) return fail(h, DMPC_ERR_BAD_SHAPE, "B,m must be >= 1");
  if (!d_H || !d_q || !d_lower || !d_upper || !d_x || !d_free || !d_iters) return fail(h, DMPC_ERR_NULL, "pnqp: required buffer is NULL");
  if (set_dev(h)) return DMPC_ERR_CUDA;
  cudaStream_t st = pick(h, stream);
  return by_dtype(h, dtype, [&](auto r) { return pnqp_impl<decltype(r)>(h, B, m, d_H, d_q, d_lower, d_upper, d_x_init, n_iter, coupling, d_x, d_LU, d_piv, d_free, d_iters, d_flags, st); });
}

int dmpc_mpc_step_forward(dmpc_handle h, int dtype, int T, int B, int n, int m, const void* d_C, const void* d_c,
                          const void* d_F, int F_T, const void* d_f, const void* d_x_nom, const void* d_u_nom,
                          const void* d_lower, const void* d_upper, const void* d_tC, const void* d_tc, int dynamics,
                          const void* d_tF, const void* d_tf, const double* h_dyn_params, double ls_decay,
                          int max_ls_trials, int need_expand, int coupling, void* d_x, void* d_u, void* d_Ks,
                          void* d_ks, void* d_u_first, void* d_objs, void* d_costs, void* d_old_costs, void* d_alphas,
                          void* d_n_qp, void* d_free, void* d_n_ls, void* d_flags, void* stream) {
  if (!h) return DMPC_ERR_NULL;
  if (T < 1 || B < 1 || n < 1 || m < 1) return fail(h, DMPC_ERR_BAD_SHAPE, "T,B,n,m must be >= 1");
  if (T > 1 && F_T != T - 1 && F_T != T) return fail(h, DMPC_ERR_BAD_SHAPE, "F_hat must have T-1 or T time rows");
  const bool sweep_only = max_ls_trials < 0;     // backward_rec only (Ks, ks, n_qp, free, flags): host-side line search
  if (!d_C || !d_c || (T > 1 && !d_F) || !d_x_nom || !d_u_nom || !d_lower || !d_upper || !d_Ks || !d_ks ||
      (!sweep_only && (!d_tC || !d_tc || !d_x || !d_u || !d_costs || !d_alphas)))
    return fail(h, DMPC_ERR_NULL, "mpc_step_forward: required buffer is NULL");
  if (!sweep_only && dynamics == DMPC_DYN_LINEAR && T > 1 && !d_tF) return fail(h, DMPC_ERR_NULL, "linear true dynamics need d_tF");
  if (dynamics == DMPC_DYN_PENDULUM && (n != 3 || m != 1 || !h_dyn_params)) return fail(h, DMPC_ERR_BAD_SHAPE, "pendulum dynamics: n=3, m=1, params required");
  if (dynamics != DMPC_DYN_LINEAR && dynamics != DMPC_DYN_PENDULUM) return fail(h, DMPC_ERR_UNSUPPORTED, "dynamics selector");
  if (set_dev(h)) return DMPC_ERR_CUDA;
  cudaStream_t st = pick(h, stream);
  return by_dtype(h, dtype, [&](auto r) { return mpc_forward_impl<decltype(r)>(h, T, B, n, m, d_C, d_c, d_F, F_T, d_f, d_x_nom, d_u_nom, d_lower, d_upper, d_tC, d_tc, dynamics, d_tF, d_tf, h_dyn_params, ls_decay, max_ls_trials, need_expand, coupling, d_x, d_u, d_Ks, d_ks, d_u_first, d_objs, d_costs, d_old_costs, d_alphas, d_n_qp, d_free, d_n_ls, d_flags, st); });
}

int dmpc_mpc_step_backward(dmpc_handle h, int dtype, int T, int B, int n, int m, const void* d_C, const void* d_c,
                           const void* d_F, int F_T, const void* d_x, const void* d_u, const void* d_lower,
                           const void* d_upper, const void* d_gx, const void* d_gu, void* d_ws_Ks, void* d_ws_ks,
                           void* d_ws_dtau, void* d_active, void* d_dx0, void* d_dC, void* d_dc, void* d_dF,
                           void* d_df, void* stream) {
  if (!h) return DMPC_ERR_NULL;
  if (T < 1 || B < 1 || n < 1 || m < 1) return fail(h, DMPC_ERR_BAD_SHAPE, "T,B,n,m must be >= 1");
  if (T > 1 && F_T != T - 1 && F_T != T) return fail(h, DMPC_ERR_BAD_SHAPE, "F_hat must have T-1 or T time rows");
  if (!d_C || !d_c || (T > 1 && (!d_F || !d_dF)) || !d_x || !d_u || !d_lower || !d_upper || !d_ws_Ks || !d_ws_ks || !d_ws_dtau ||
      !d_active || !d_dx0 || !d_dC || !d_dc)
    return fail(h, DMPC_ERR_NULL, "mpc_step_backward: required buffer is NULL");
  if (set_dev(h)) return DMPC_ERR_CUDA;
  cudaStream_t st = pick(h, stream);
  return by_dtype(h, dtype, [&](auto r) { return mpc_backward_impl<decltype(r)>(h, T, B, n, m, d_C, d_c, d_F, F_T, d_x, d_u, d_lower, d_upper, d_gx, d_gu, d_ws_Ks, d_ws_ks, d_ws_dtau, d_active, d_dx0, d_dC, d_dc, d_dF, d_df, st); });
}

int dmpc_lqr_active_solve(dmpc_handle h, int dtype, int T, int B, int n, int m, const void* d_x0, const void* d_C,
                          const void* d_c, const void* d_F, int F_T, const void* d_f, const void* d_active, void* d_x,
                          void* d_u, void* d_Ks, void* d_ks, void* stream) {
  if (!h) return DMPC_ERR_NULL;
  if (T < 1 || B < 1 || n < 1 || m < 1) return fail(h, DMPC_ERR_BAD_SHAPE, "T,B,n,m must be >= 1");
  if (T > 1 && F_T != T - 1 && F_T != T) return fail(h, DMPC_ERR_BAD_SHAPE, "F must have T-1 or T time rows");
  if (!d_x0 || !d_C || !d_c || (T > 1 && !d_F) || !d_active || !d_x || !d_u || !d_Ks || !d_ks) return fail(h, DMPC_ERR_NULL, "lqr_active: required buffer is NULL");
  if (set_dev(h)) return DMPC_ERR_CUDA;
  cudaStream_t st = pick(h, stream);
  return by_dtype(h, dtype, [&](auto r) { return lqr_active_impl<decltype(r)>(h, T, B, n, m, d_x0, d_C, d_c, d_F, d_f, d_active, d_x, d_u, d_Ks, d_ks, st); });
}

int dmpc_get_traj(dmpc_handle h, int dtype, int T, int B, int n, int m, int dynamics, const void* d_x0,
                  const void* d_u, const void* d_F, const void* d_f, const double* h_dyn_params, void* d_x,
                  void* d_Fout, void* d_fout, void* stream) {
  if (!h) return DMPC_ERR_NULL;
  if (T < 1 || B < 1 || n < 1 || m < 1) return fail(h, DMPC_ERR_BAD_SHAPE, "T,B,n,m must be >= 1");
  if (!d_x0 || !d_u || !d_x) return fail(h, DMPC_ERR_NULL, "get_traj: required buffer is NULL");
  if (dynamics == DMPC_DYN_LINEAR && T > 1 && !d_F) return fail(h, DMPC_ERR_NULL, "linear dynamics need d_F");
  if (dynamics == DMPC_DYN_PENDULUM && (n != 3 || m != 1 || !h_dyn_params)) return fail(h, DMPC_ERR_BAD_SHAPE, "pendulum dynamics: n=3, m=1, params required");
  if ((d_Fout == nullptr) != (d_fout == nullptr)) return fail(h, DMPC_ERR_NULL, "Fout and fout go together");
  if (set_dev(h)) return DMPC_ERR_CUDA;
  cudaStream_t st = pick(h, stream);
  return by_dtype(h, dtype, [&](auto r) { return traj_impl<decltype(r)>(h, T, B, n, m, dynamics, d_x0, d_u, d_F, d_f, h_dyn_params, d_x, d_Fout, d_fout, st); });
}

int dmpc_boxddp_workspace_bytes(int dtype, int T, int B, int n, int m, size_t* bytes) {
  if (!bytes || T < 1 || B < 1 || n < 1 || m < 1) return DMPC_ERR_BAD_SHAPE;
  if (dtype != DMPC_F64 && dtype != DMPC_F32) return DMPC_ERR_UNSUPPORTED;
  *bytes = box_ws(dtype == DMPC_F64 ? 8 : 4, T, B, n, m).total;
  return DMPC_OK;
}

int dmpc_boxddp_solve(dmpc_handle h, int dtype, int T, int B, int n, int m, const void* d_x_init, const void* d_C,
                      const void* d_c, const void* d_lower, const void* d_upper, int dynamics, const void* d_F, int F_T,
                      const void* d_f, const double* h_dyn_params, const void* d_u_init, const dmpc_boxddp_opts* opts,
                      void* d_ws, size_t ws_bytes, void* d_x_best, void* d_u_best, void* d_costs_best, void* d_du_best,
                      void* d_du_last, void* d_F_lin, void* d_f_lin, int* h_n_iter, int* h_status, int* h_flags,
                      void* stream) {
  if (!h) return DMPC_ERR_NULL;
  if (T < 1 || B < 1 || n < 1 || m < 1) return fail(h, DMPC_ERR_BAD_SHAPE, "T,B,n,m must be >= 1");
  if (!opts || opts->max_iter < 1) return fail(h, DMPC_ERR_BAD_SHAPE, "boxddp: opts with max_iter >= 1 required");
  if (!d_x_init || !d_C || !d_c || !d_lower || !d_upper || !d_u_init || !d_ws || !d_x_best || !d_u_best || !d_costs_best || !d_du_best)
    return fail(h, DMPC_ERR_NULL, "boxddp: required buffer is NULL");
  if (dynamics == DMPC_DYN_LINEAR && T > 1 && (!d_F || (F_T != T - 1 && F_T != T))) return fail(h, DMPC_ERR_BAD_SHAPE, "boxddp: linear dynamics need F with T-1 or T rows");
  if (dynamics == DMPC_DYN_PENDULUM && (n != 3 || m != 1 || !h_dyn_params || !d_F_lin || !d_f_lin))
    return fail(h, DMPC_ERR_BAD_SHAPE, "boxddp: pendulum needs n=3, m=1, params and F_lin/f_lin outputs");
  if (dynamics != DMPC_DYN_LINEAR && dynamics != DMPC_DYN_PENDULUM) return fail(h, DMPC_ERR_UNSUPPORTED, "dynamics selector");
  size_t need = 0;
  if (dmpc_boxddp_workspace_bytes(dtype, T, B, n, m, &need)) return fail(h, DMPC_ERR_UNSUPPORTED, "dtype");
  if (ws_bytes < need) return fail(h, DMPC_ERR_BAD_SHAPE, "boxddp: workspace too small (dmpc_boxddp_workspace_bytes)");
  if (set_dev(h)) return DMPC_ERR_CUDA;
  cudaStream_t st = pick(h, stream);
  return by_dtype(h, dtype, [&](auto r) { return boxddp_impl<decltype(r)>(h, dtype, T, B, n, m, d_x_init, d_C, d_c, d_lower, d_upper, dynamics, d_F, F_T, d_f, h_dyn_params, d_u_init, opts, d_ws, d_x_best, d_u_best, d_costs_best, d_du_best, d_du_last, d_F_lin, d_f_lin, h_n_iter, h_status, h_flags, st); });
}

int dmpc_expand_time_batch(dmpc_handle h, int dtype, int T, int B, int count, const void* d_src, void* d_dst, void* stream) {
  if (!h) return DMPC_ERR_NULL;
  if (T < 1 || B < 1 || count < 1) return fail(h, DMPC_ERR_BAD_SHAPE, "T,B,count must be >= 1");
  if (!d_src || !d_dst) return fail(h, DMPC_ERR_NULL, "expand_time_batch: src/dst required");
  if (set_dev(h)) return DMPC_ERR_CUDA;
  cudaStream_t st = pick(h, stream);
  const size_t total = (size_t)T * B * count;
  return by_dtype(h, dtype, [&](auto r) {
    using R = decltype(r);
    return launch_expand_time_batch<R>((const R*)d_src, (R*)d_dst, count, total, st, &h->launches);
  });
}

static int warmstart_impl(dmpc_handle h, int dtype, int T, int B, int m, int n_samples, void* d_cache, const int* d_idx,
                          void* d_u, bool put, void* stream) {
  if (!h) return DMPC_ERR_NULL;
  if (T < 1 || B < 1 || m < 1 || n_samples < 1) return fail(h, DMPC_ERR_BAD_SHAPE, "T,B,m,n_samples must be >= 1");
  if (!d_cache || !d_idx || !d_u) return fail(h, DMPC_ERR_NULL, "warmstart: cache, idx and u are required");
  if (set_dev(h)) return DMPC_ERR_CUDA;
  cudaStream_t st = pick(h, stream);
  const size_t total = (size_t)T * B * m;
  const int tpb = 256;
  const unsigned grid = (unsigned)((total + tpb - 1) / tpb);
  return by_dtype(h, dtype, [&](auto r) {
    using R = decltype(r);
    const int rc = launch(put ? warmstart_kernel<R, true> : warmstart_kernel<R, false>, grid, tpb, 0, st, &h->launches, T, B, m,
                          n_samples, (R*)d_cache, d_idx, (R*)d_u);
    return rc ? fail(h, rc, "warmstart launch failed") : DMPC_OK;
  });
}

int dmpc_warmstart_take(dmpc_handle h, int dtype, int T, int B, int m, int n_samples, const void* d_cache, const int32_t* d_idx,
                        void* d_u, void* stream) {
  return warmstart_impl(h, dtype, T, B, m, n_samples, const_cast<void*>(d_cache), (const int*)d_idx, d_u, false, stream);
}

int dmpc_warmstart_put(dmpc_handle h, int dtype, int T, int B, int m, int n_samples, void* d_cache, const int32_t* d_idx,
                       const void* d_u, void* stream) {
  return warmstart_impl(h, dtype, T, B, m, n_samples, d_cache, (const int*)d_idx, const_cast<void*>(d_u), true, stream);
}

size_t dmpc_reduced_grad_elems(int n, int m) { return (size_t)adj_red_elems(n, m); }

int dmpc_lqr_adjoint_reduced(dmpc_handle h, int dtype, int T, int B, int n, int m, const void* d_C, const void* d_c,
                             const void* d_F, const void* d_x, const void* d_u, const void* d_gx, const void* d_gu,
                             const void* d_Ks, const void* d_fac, void* d_ws_dtau, void* d_ws_partials, void* d_dx0,
                             void* d_sums, int flags, void* stream) {
  if (!h) return DMPC_ERR_NULL;
  if (T < 1 || B < 1 || n < 1 || m < 1) return fail(h, DMPC_ERR_BAD_SHAPE, "T,B,n,m must be >= 1");
  if (!d_C || !d_c || !d_x || !d_u || !d_gx || !d_gu || !d_Ks || !d_fac || !d_ws_dtau || !d_ws_partials || !d_dx0 || !d_sums || (T > 1 && !d_F))
    return fail(h, DMPC_ERR_NULL, "lqr_adjoint_reduced: required buffer is NULL");
  if (set_dev(h)) return DMPC_ERR_CUDA;
  cudaStream_t st = pick(h, stream);
  return by_dtype(h, dtype, [&](auto r) { return lqr_adjoint_impl<decltype(r)>(h, T, B, n, m, d_C, d_c, d_F, d_x, d_u, d_gx, d_gu, d_Ks, d_fac, d_dx0, nullptr, d_ws_dtau, nullptr, nullptr, flags, st, d_ws_partials, d_sums); });
}

int dmpc_mpc_step_backward_reduced(dmpc_handle h, int dtype, int T, int B, int n, int m, const void* d_C, const void* d_c,
                                   const void* d_F, int F_T, const void* d_x, const void* d_u, const void* d_lower,
                                   const void* d_upper, const void* d_gx, const void* d_gu, void* d_ws_Ks, void* d_ws_ks,
                                   void* d_ws_dtau, void* d_active, void* d_ws_partials, void* d_dx0, void* d_sums,
                                   void* stream) {
  if (!h) return DMPC_ERR_NULL;
  if (T < 1 || B < 1 || n < 1 || m < 1) return fail(h, DMPC_ERR_BAD_SHAPE, "T,B,n,m must be >= 1");
  if (T > 1 && F_T != T - 1 && F_T != T) return fail(h, DMPC_ERR_BAD_SHAPE, "F_hat must have T-1 or T time rows");
  if (!d_C || !d_c || (T > 1 && !d_F) || !d_x || !d_u || !d_lower || !d_upper || !d_ws_Ks || !d_ws_ks || !d_ws_dtau ||
      !d_active || !d_ws_partials || !d_dx0 || !d_sums)
    return fail(h, DMPC_ERR_NULL, "mpc_step_backward_reduced: required buffer is NULL");
  if (set_dev(h)) return DMPC_ERR_CUDA;
  cudaStream_t st = pick(h, stream);
  return by_dtype(h, dtype, [&](auto r) { return mpc_backward_impl<decltype(r)>(h, T, B, n, m, d_C, d_c, d_F, F_T, d_x, d_u, d_lower, d_upper, d_gx, d_gu, d_ws_Ks, d_ws_ks, d_ws_dtau, d_active, d_dx0, nullptr, nullptr, nullptr, nullptr, st, d_ws_partials, d_sums); });
}

int dmpc_lqr_shared_workspace_bytes_ex(int dtype, int T, int B, int n, int m, int share, size_t* bytes) {
  if (!bytes || T < 1 || B < 1 || n < 1 || m < 1) return DMPC_ERR_BAD_SHAPE;
  if (dtype != DMPC_F64 && dtype != DMPC_F32) return DMPC_ERR_UNSUPPORTED;
  if (m > 32 || (share & ~DMPC_SHARE_C)) return DMPC_ERR_UNSUPPORTED;
  const SharedWs W = shared_ws(dtype == DMPC_F64 ? 8 : 4, T, B, n, m, share);
  if (!W.NB) return DMPC_ERR_UNSUPPORTED;
  *bytes = W.total;
  return DMPC_OK;
}

int dmpc_lqr_shared_workspace_bytes(int dtype, int T, int B, int n, int m, size_t* bytes) {
  return dmpc_lqr_shared_workspace_bytes_ex(dtype, T, B, n, m, 0, bytes);
}

// common checks of the two shared-parameter calls; 0 or a status
static int shared_check(dmpc_handle h, int dtype, int T, int B, int n, int m, int F_T, const void* F, const void* ws,
                        size_t ws_bytes, int share) {
  if (T < 1 || B < 1 || n < 1 || m < 1) return fail(h, DMPC_ERR_BAD_SHAPE, "T,B,n,m must be >= 1");
  if (F_T != T - 1 && F_T != T) return fail(h, DMPC_ERR_BAD_SHAPE, "F must have T-1 or T time rows");
  if ((T > 1 && !F) || !ws) return fail(h, DMPC_ERR_NULL, "lqr shared: F (T > 1) and the workspace are required");
  if (dtype != DMPC_F64 && dtype != DMPC_F32) return fail(h, DMPC_ERR_UNSUPPORTED, "dtype");
  if (m > 32) return fail(h, DMPC_ERR_UNSUPPORTED, "lqr shared: m > 32");
  if (share & ~DMPC_SHARE_C) return fail(h, DMPC_ERR_UNSUPPORTED, "lqr shared: unknown bit in share");
  size_t need = 0;
  if (dmpc_lqr_shared_workspace_bytes_ex(dtype, T, B, n, m, share, &need)) return fail(h, DMPC_ERR_UNSUPPORTED, "lqr shared: shape too large for the chunk kernels");
  if (ws_bytes < need) return fail(h, DMPC_ERR_BAD_SHAPE, "lqr shared: workspace too small (dmpc_lqr_shared_workspace_bytes[_ex])");
  return DMPC_OK;
}

int dmpc_lqr_solve_shared_ex(dmpc_handle h, int dtype, int T, int B, int n, int m, const void* d_x0, const void* d_C,
                             const void* d_c, const void* d_F, int F_T, const void* d_f, void* d_x, void* d_u, void* d_ws,
                             size_t ws_bytes, int share, void* stream) {
  if (!h) return DMPC_ERR_NULL;
  if (!d_x0 || !d_C || !d_c || !d_x || !d_u) return fail(h, DMPC_ERR_NULL, "lqr_solve_shared: required buffer is NULL");
  if (int rc = shared_check(h, dtype, T, B, n, m, F_T, d_F, d_ws, ws_bytes, share)) return rc;
  if (set_dev(h)) return DMPC_ERR_CUDA;
  cudaStream_t st = pick(h, stream);
  return by_dtype(h, dtype, [&](auto r) { return lqr_solve_shared_impl<decltype(r)>(h, T, B, n, m, d_x0, d_C, d_c, d_F, F_T, d_f, d_x, d_u, d_ws, share, st); });
}

int dmpc_lqr_solve_shared(dmpc_handle h, int dtype, int T, int B, int n, int m, const void* d_x0, const void* d_C,
                          const void* d_c, const void* d_F, int F_T, const void* d_f, void* d_x, void* d_u, void* d_ws,
                          size_t ws_bytes, void* stream) {
  return dmpc_lqr_solve_shared_ex(h, dtype, T, B, n, m, d_x0, d_C, d_c, d_F, F_T, d_f, d_x, d_u, d_ws, ws_bytes, 0, stream);
}

int dmpc_lqr_adjoint_shared_ex(dmpc_handle h, int dtype, int T, int B, int n, int m, const void* d_C, const void* d_c,
                               const void* d_F, int F_T, const void* d_x, const void* d_u, const void* d_gx,
                               const void* d_gu, void* d_ws, size_t ws_bytes, void* d_dx0, void* d_dC, void* d_dc,
                               void* d_dF, void* d_df, int flags, int share, void* stream) {
  if (!h) return DMPC_ERR_NULL;
  const bool dc_nullable = (share & DMPC_SHARE_C) != 0;
  if (!d_C || !d_c || !d_x || !d_u || !d_dx0 || !d_dC || (!d_dc && !dc_nullable) || (F_T > 0 && !d_dF))
    return fail(h, DMPC_ERR_NULL, "lqr_adjoint_shared: required buffer is NULL");
  if (int rc = shared_check(h, dtype, T, B, n, m, F_T, d_F, d_ws, ws_bytes, share)) return rc;
  if (set_dev(h)) return DMPC_ERR_CUDA;
  cudaStream_t st = pick(h, stream);
  return by_dtype(h, dtype, [&](auto r) { return lqr_adjoint_shared_impl<decltype(r)>(h, T, B, n, m, d_C, d_c, d_F, F_T, d_x, d_u, d_gx, d_gu, d_ws, d_dx0, d_dC, d_dc, d_dF, d_df, flags, share, st); });
}

int dmpc_lqr_adjoint_shared(dmpc_handle h, int dtype, int T, int B, int n, int m, const void* d_C, const void* d_c,
                            const void* d_F, int F_T, const void* d_x, const void* d_u, const void* d_gx,
                            const void* d_gu, void* d_ws, size_t ws_bytes, void* d_dx0, void* d_dC, void* d_dc,
                            void* d_dF, void* d_df, int flags, void* stream) {
  return dmpc_lqr_adjoint_shared_ex(h, dtype, T, B, n, m, d_C, d_c, d_F, F_T, d_x, d_u, d_gx, d_gu, d_ws, ws_bytes, d_dx0,
                                    d_dC, d_dc, d_dF, d_df, flags, 0, stream);
}

}  // extern "C"
