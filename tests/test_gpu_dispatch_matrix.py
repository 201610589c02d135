"""GPU: every kernel the launchers (csrc/lqr_launch.cu, csrc/mpc_launch.cu) can select, against the fp64 oracle.

Each case names the kernel it is meant to reach and proves it: the call runs under torch.profiler (CUDA activity), which
records every kernel of the process, including the ones launched through the C ABI, and the case asserts a substring of
the expected kernel name (and, where a path is a fall-back, that the kernel it falls back from did not run).

Default-path cases run in the test process.  The A/B switches (DMPC_LQR_GROUP, DMPC_ADJ_GROUP, DMPC_LQR_TPE_EPW,
DMPC_DISABLE_DMMA, DMPC_ADJ_UNFUSED, DMPC_MPC_GROUP, DMPC_MPC_NO_SPEC, DMPC_MPC_NO_STASH) are read once per process, so
each setting runs its cases in a child process (`python test_gpu_dispatch_matrix.py --child SETTING OUT.npz`) and the
parent checks the outputs against the oracle.

Tolerances are the suite's: 1e-10 element-relative in fp64 (_helpers.rel_err), 1e-4 in fp32 (1e-3 for fp32 gradients),
PNQP active sets, iteration counts and line-search alphas bit-exact.  Large batches are checked on a slice at each end and
one in the middle (batch elements are independent, or - batch coupling - the oracle runs on the whole batch).

Launcher branch -> case that reaches it (kernel asserted from the profiler trace):
  launch_lqr_solve    DMMA (32,8, aligned)                  default  lqr-*-n32m8-*-pathdmma*
                      thread-per-element (2,1) (3,1) (4,2)  default  *-pathtpe*, epw8 / epw16 / epw_auto
                      specialised group <N,M,G>             lqr_group, active at (32,8), mpcb at (32,8), *-pathfused*
                      runtime group G = 8 / 16 / 32 / 256   default  lqr-*-pathgroup* (m > n included), active, mpcb
  launch_lqr_adjoint  lqr_dtau: tpe / specialised / runtime G   as above (adjoint of every lqr case)
                      adjoint_out: tpe (full) / specialised / runtime   as above; reduced: *-reduced*; adj_group
                      two sweeps where adjoint_fused_available  (32,8) full and reduced: *-pathdmma*, *-pathfused*; off: adj_unfused
  launch_mpc_forward  tpe (m = 1) / specialised / runtime   default mpcf cases, mpc_group (linear and pendulum <3,1,4>)
  launch_mpc_tpe      4 lanes with / without stash, 1 lane   default mpcf (stash threshold asserted), mpc_no_spec, mpc_no_stash
MPC step forward contract (mpcf keys, every kernel above in both couplings where the launcher has them):
  true_cost           separate tC, tc buffers (the oracle asserts they change the line search); elements e % 5 == 2 capped
  cap = 1 ... 6, 0    max_ls_trials (0 = 64): FLAG_LS_CAPPED exactly on the capped elements, n_ls = the cap, alpha of the
                      last pass; every cap mod 4 with and without the stash (test_mpcf_four_lane_coverage)
  decay = 0.7 / 0.9   true control gain 1 - 10 x the model's: winners on every lane and in later rounds of the 4-lane kernel
  expand / f / FT     need_expand = 0 with the model f (and without: f = False); F with T rows
  dyn = "pendulum"    g, m, l, dt = 0.03, max_torque = 1.5 off their defaults, bounds +-2 (the torque clip is active)
Every mpcf case checks n_qp, free, alphas, n_ls and the capped flag bit-exact, x, u, Ks, ks, objs, u_first, costs and
old costs against the oracle (1e-10; 1e-9 for element-coupled x, u), and that no decisive line-search comparison is within
1e3 ulp of the old cost.
  launch_pnqp         SG = 32 (17 <= m <= 32), both couplings  default pnqp cases (SG 4 / 8 / 16: tests/test_gpu_mpc.py)
Not reached here: batch-coupled launches spread over a thread-block cluster (tests/test_gpu_mpc.py covers them), the
one-lane element-coupled MPC kernel at T >= 454 (an oracle run that long is slow), the m > 32 errors.  The MPC step
backward (full and reduced, every kernel and A/B setting it can select, non-symmetric C, F with T rows, gx or gu NULL,
the active-set band) is in tests/test_gpu_mpc_backward_matrix.py; the mpcb cases here are its default-path subset.
"""
import os
import subprocess
import sys
import tempfile
import warnings

import numpy as np
import pytest

if __name__ == "__main__":                       # child process: the import paths tests/conftest.py sets up
    _root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    _pkg = os.path.join(_root, "chainer-differentiable-mpc_b200")
    for _p in (os.path.dirname(os.path.abspath(__file__)), _root, _pkg):
        if _p not in sys.path:
            sys.path.insert(0, _p)

import _native
from _helpers import rel_err, lqr_problem, psd_cost, stable_dynamics
from oracle import lqr as olqr, mpc as ompc, pendulum as opend, pnqp as opnqp

pytestmark = pytest.mark.gpu

F64, F32 = "f64", "f32"
NP = {F64: np.float64, F32: np.float32}
CNAME = {F64: "double", F32: "float"}


def tol(dt, grad=False):
    return 1e-10 if dt == F64 else (1e-3 if grad else 1e-4)


# ------------------------------------------------------------------------------------------------ device buffers
class _Buf:
    """A device tensor at `off` elements past the start of a torch allocation (the caching allocator's blocks are 512-byte
    aligned, so off = 1 gives a pointer that is aligned to its element type but not to 16 bytes)."""

    def __init__(self, t, off, shape):
        self.t, self.off, self.shape = t, off, tuple(shape)

    def __int__(self):
        return self.t.data_ptr() + self.off * self.t.element_size()

    def get(self):
        return self.t[self.off:].cpu().numpy().reshape(self.shape)


class Bufs:
    def __init__(self, off=0):
        import torch
        self.torch, self.off = torch, off

    def _tdt(self, dt):
        return {np.dtype(np.float64): self.torch.float64, np.dtype(np.float32): self.torch.float32,
                np.dtype(np.int32): self.torch.int32, np.dtype(np.uint8): self.torch.uint8}[np.dtype(dt)]

    def put(self, a, dt):
        a = np.ascontiguousarray(a, dtype=dt)
        t = self.torch.zeros(a.size + self.off, dtype=self._tdt(dt), device="cuda")
        t[self.off:].copy_(self.torch.from_numpy(a.reshape(-1)))
        return _Buf(t, self.off, a.shape)

    def empty(self, shape, dt):
        size = int(np.prod(shape))
        if np.dtype(dt).kind == "f":       # NaN: an output entry the kernel does not write fails the comparison
            t = self.torch.full((size + self.off,), float("nan"), dtype=self._tdt(dt), device="cuda")
        else:
            t = self.torch.zeros(size + self.off, dtype=self._tdt(dt), device="cuda")
        return _Buf(t, self.off, shape)

    def ready(self):
        self.torch.cuda.synchronize()     # the uploads ran on torch's stream, the library uses its own


def profiled(ctx, fn):
    """Runs fn() under the CUDA profiler; returns (fn's result, names of the dmpc:: kernels that ran)."""
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        ctx.sync()
    names = set()
    for e in prof.events():
        names.add(e.name)
    try:
        for e in prof.profiler.kineto_results.events():
            names.add(e.name())
    except AttributeError:
        pass
    return out, sorted(k for k in names if "dmpc::" in k)


def assert_kernels(names, expect, absent=()):
    for s in expect:
        assert any(s in k for k in names), ("kernel not launched", s, names)
    for s in absent:
        assert not any(s in k for k in names), ("kernel launched", s, names)


def slices(B):
    if B <= 64:
        return [slice(0, B)]
    return [slice(0, 16), slice(B // 2 - 8, B // 2 + 8), slice(B - 16, B)]


# ------------------------------------------------------------------------------------------------ problems
def pivot_problem(seed, T, B, n, m):
    """Non-symmetric C whose control block is made of 2 x 2 blocks [[0.2, 1], [1.5, 0.3]] (+ a small random part) and small
    F_u: Quu = C_uu + F_u^T V F_u stays close to C_uu, whose largest first-column entry lies below the diagonal, so the
    pivoted elimination swaps rows in every step (the reference factors Quu with pivoted LU and never symmetrises C)."""
    pr = lqr_problem(seed, T, B, n, m, with_f=True, sym=False)
    C = pr["C"]
    base = np.eye(m)
    for i in range(0, m - 1, 2):
        base[i:i + 2, i:i + 2] = [[0.2, 1.0], [1.5, 0.3]]
    C[..., n:, n:] = base + 0.1 * (C[..., n:, n:] - np.eye(m))
    pr["F"][..., n:] *= 0.01
    assert (np.abs(C[T - 1, :, n + 1, n]) > np.abs(C[T - 1, :, n, n])).all()
    return pr


def problem(sp):
    if sp.get("pivot"):
        return pivot_problem(sp["seed"], sp["T"], sp["B"], sp["n"], sp["m"])
    return lqr_problem(sp["seed"], sp["T"], sp["B"], sp["n"], sp["m"], with_f=sp.get("with_f", True),
                       sym=sp.get("sym", True))


def lqr_kernels(path, n, m, dt, G=None):
    """Expected kernel-name prefixes of forward, adjoint and reduced adjoint for one LQR dispatch path."""
    R = CNAME[dt]
    if path == "tpe":                 # s <= 6 thread-per-element kernels (lqr_tpe_kernel.cuh)
        return dict(fwd=["lqr_tpe_kernel<%s, %d, %d," % (R, n, m)],
                    adj=["lqr_dtau_tpe_kernel<%s, %d, %d," % (R, n, m), "adjoint_out_tpe_kernel<%s, %d, %d," % (R, n, m)],
                    red=["lqr_dtau_tpe_kernel<%s, %d, %d," % (R, n, m), "adjoint_out_kernel<%s, %d, %d, %d, true>" % (R, n, m, G)])
    if path == "tpe_adj_group":       # DMPC_ADJ_GROUP=1: adjoint_out_kernel next to the thread-per-element solves
        return dict(fwd=["lqr_tpe_kernel<%s, %d, %d," % (R, n, m)],
                    adj=["lqr_dtau_tpe_kernel<%s, %d, %d," % (R, n, m), "adjoint_out_kernel<%s, %d, %d, %d, false>" % (R, n, m, G)],
                    red=[])
    if path == "unfused":             # DMPC_ADJ_UNFUSED=1 at (32,8): DMMA forward, three-sweep adjoint
        return dict(fwd=["lqr_factor_dmma_warp_kernel"],
                    adj=["lqr_dtau_kernel<%s, 32, 8, 64, false>" % R, "adjoint_out_kernel<%s, 32, 8, 128, false>" % R],
                    red=["lqr_dtau_kernel<%s, 32, 8, 64, false>" % R, "adjoint_out_kernel<%s, 32, 8, 128, true>" % R])
    if path == "dmma":                # n = 32, m = 8, 16-byte aligned: DMMA warp kernel + two-sweep adjoint
        return dict(fwd=["lqr_factor_dmma_warp_kernel"],
                    adj=["lqr_dtau_kernel<%s, 32, 8, 64, true>" % R, "adjoint_fused_kernel<%s, 32, 8, 128, false>" % R],
                    red=["lqr_dtau_kernel<%s, 32, 8, 64, true>" % R, "adjoint_fused_kernel<%s, 32, 8, 128, true>" % R])
    if path == "fused":               # n = 32, m = 8 on the group kernel, V_t saved for the two-sweep adjoint
        return dict(fwd=["lqr_solve_kernel<%s, 32, 8, 256>" % R],
                    adj=["lqr_dtau_kernel<%s, 32, 8, 64, true>" % R, "adjoint_fused_kernel<%s, 32, 8, 128, false>" % R],
                    red=["lqr_dtau_kernel<%s, 32, 8, 64, true>" % R, "adjoint_fused_kernel<%s, 32, 8, 128, true>" % R])
    # group kernels: specialised (N, M) or runtime shape (0, 0), G lanes per element
    N, M = (n, m) if path == "spec" else (0, 0)
    Gd, Ga = (G if G <= 32 else 64), (G if G <= 32 else 128)
    return dict(fwd=["lqr_solve_kernel<%s, %d, %d, %d>" % (R, N, M, G)],
                adj=["lqr_dtau_kernel<%s, %d, %d, %d, false>" % (R, N, M, Gd), "adjoint_out_kernel<%s, %d, %d, %d, false>" % (R, N, M, Ga)],
                red=["lqr_dtau_kernel<%s, %d, %d, %d, false>" % (R, N, M, Gd), "adjoint_out_kernel<%s, %d, %d, %d, true>" % (R, N, M, Ga)])


# ------------------------------------------------------------------------------------------------ LQR: forward + adjoints
def _lqr_call(ctx, pr, dt, off, reduced, adjoint=True):
    T, B, n, m = pr["T"], pr["B"], pr["n"], pr["m"]
    s = n + m
    npd = NP[dt]
    b = Bufs(off)
    x0, C, c = b.put(pr["x0"], npd), b.put(pr["C"], npd), b.put(pr["c"], npd)
    F = b.put(pr["F"] if T > 1 else np.zeros((1, B, n, s)), npd)
    f = b.put(pr["f"] if T > 1 else np.zeros((1, B, n)), npd)
    x, u, Ks, ks = b.empty((T, B, n), npd), b.empty((T, B, m), npd), b.empty((T, B, m, n), npd), b.empty((T, B, m), npd)
    fac = b.empty((ctx.lqr_fac_elems(T, B, n, m),), npd)
    rs = np.random.RandomState(3)
    gx, gu = b.put(rs.randn(T, B, n), npd), b.put(rs.randn(T, B, m), npd)
    b.ready()
    out = {}

    def go():
        ctx.lqr_solve(npd, T, B, n, m, x0, C, c, F, T - 1, f, x, u, Ks, ks, fac,
                      _native.LQR_FACTOR | _native.LQR_ROLLOUT | _native.LQR_SAVE_FAC)
        if not adjoint:
            return
        for tag, flags in (("s", _native.ADJ_STRICT_REFERENCE), ("c", 0)):
            g = [b.empty((B, n), npd), b.empty((T, B, s, s), npd), b.empty((T, B, s), npd),
                 b.empty((max(T - 1, 1), B, n, s), npd), b.empty((max(T - 1, 1), B, n), npd)]
            ctx.lqr_adjoint(npd, T, B, n, m, C, c, F, x, u, gx, gu, Ks, fac, *g, flags)
            ctx.sync()
            for k, a in zip(("dx0", "dC", "dc", "dF", "df"), g):
                out[tag + "_" + k] = a.get()[:T - 1] if k in ("dF", "df") else a.get()
        if reduced:
            rsz = ctx.reduced_grad_elems(n, m)
            dtau, part, rdx0, sums = b.empty((T, B, s), npd), b.empty((B, rsz), npd), b.empty((B, n), npd), b.empty((rsz,), npd)
            ctx.lqr_adjoint_reduced(npd, T, B, n, m, C, c, F, x, u, gx, gu, Ks, fac, dtau, part, rdx0, sums,
                                    _native.ADJ_STRICT_REFERENCE)
            ctx.sync()
            out["r_dx0"], out["r_sums"] = rdx0.get(), sums.get()

    return out, go, dict(x=x, u=u, Ks=Ks, ks=ks)


def run_lqr(ctx, sp):
    """Forward, strict and corrected adjoints (and the reduced adjoint) under the profiler; with off=1 also the same call
    on aligned buffers (outside the profiler) for the aligned-vs-misaligned comparison."""
    pr = problem(sp)
    out, go, fw = _lqr_call(ctx, pr, sp["dt"], sp.get("off", 0), sp.get("reduced", False))
    _, names = profiled(ctx, go)
    for k, v in fw.items():
        out[k] = v.get()
    if sp.get("off", 0):
        ref, go2, fw2 = _lqr_call(ctx, pr, sp["dt"], 0, sp.get("reduced", False))
        go2()
        ctx.sync()
        for k, v in fw2.items():
            out["aligned_" + k] = v.get()
        for k, v in ref.items():
            out["aligned_" + k] = v
    return out, names


def check_lqr(sp, out, names):
    pr = problem(sp)
    T, B, n, m, dt = sp["T"], sp["B"], sp["n"], sp["m"], sp["dt"]
    ek = lqr_kernels(sp["path"], n, m, dt, sp.get("G"))
    assert_kernels(names, ek["fwd"] + ek["adj"] + (ek["red"] if sp.get("reduced") else []),
                   absent=() if sp["path"] in ("dmma", "unfused") else ("lqr_factor_dmma_warp_kernel",))
    tf, tg = tol(dt), tol(dt, grad=True)
    rs = np.random.RandomState(3)
    gx, gu = rs.randn(T, B, n), rs.randn(T, B, m)
    f = pr["f"] if T > 1 else None
    for sl in slices(B):
        F = pr["F"][:, sl]
        ox, ou, oK, ok = olqr.lqr_solve(pr["x0"][sl], pr["C"][:, sl], pr["c"][:, sl], F, None if f is None else f[:, sl], n, m)
        for k, w in (("x", ox), ("u", ou), ("Ks", oK), ("ks", ok)):
            assert rel_err(out[k][:, sl], w) < tf, (k, sl, rel_err(out[k][:, sl], w))
        for tag, strict in (("s", True), ("c", False)):
            want = olqr.difflqr_backward(pr["x0"][sl], pr["C"][:, sl], pr["c"][:, sl], F, ox, ou, gx[:, sl], gu[:, sl], n, m,
                                         quirk_dC=strict, quirk_df=strict)
            assert rel_err(out[tag + "_dx0"][sl], want[0]) < tg, (tag, "dx0")
            for k, w in zip(("dC", "dc", "dF", "df"), want[1:]):
                assert rel_err(out[tag + "_" + k][:, sl], w) < tg, (tag, k, sl, rel_err(out[tag + "_" + k][:, sl], w))
    if sp.get("reduced"):
        # the (T,B)-sums against the oracle's full gradients summed (a sum of T*B signed terms: tensor-wide scale), dx0 as is
        ox, ou, _, _ = olqr.lqr_solve(pr["x0"], pr["C"], pr["c"], pr["F"], f, n, m)
        want = olqr.difflqr_backward(pr["x0"], pr["C"], pr["c"], pr["F"], ox, ou, gx, gu, n, m)
        sums = _native.Context.split_reduced(out["r_sums"].astype(np.float64), n, m)
        assert rel_err(out["r_dx0"], want[0]) < tg
        for k, a, w in zip(("dC", "dc", "dF", "df"), sums, want[1:]):
            w = w.sum(axis=(0, 1))
            if T == 1 and k in ("dF", "df"):
                assert not a.any(), k
                continue
            assert np.max(np.abs(a - w)) / np.max(np.abs(w)) < tg, ("reduced", k)
    if sp.get("off"):
        # the misaligned call agrees with the aligned one (at n = 32, m = 8 the aligned fp64 call runs the DMMA kernel, a
        # different algorithm: agreement to the oracle tolerance, not bit for bit)
        for k in ("x", "u", "Ks", "ks", "s_dC", "s_dF", "c_dC", "c_df"):
            assert rel_err(out[k], out["aligned_" + k]) < (tg if "_" in k else tf), ("aligned vs misaligned", k)
        if sp.get("reduced"):
            a, w = out["r_sums"].astype(np.float64), out["aligned_r_sums"].astype(np.float64)
            assert np.max(np.abs(a - w)) / np.max(np.abs(w)) < tg, "aligned vs misaligned reduced sums"


# ------------------------------------------------------------------------------------------------ LQR_active / MPC backward
def active_problem(sp):
    T, B, n, m = sp["T"], sp["B"], sp["n"], sp["m"]
    pr = pivot_problem(sp["seed"], T, B, n, m) if sp.get("pivot") else lqr_problem(sp["seed"], T, B, n, m)
    rs = np.random.RandomState(sp["seed"] + 1)
    pr["active"] = rs.rand(T, B, m) < 0.4
    return pr


def run_active(ctx, sp):
    pr = active_problem(sp)
    T, B, n, m = sp["T"], sp["B"], sp["n"], sp["m"]
    npd = NP[sp["dt"]]
    b = Bufs(0)
    d = [b.put(pr[k], npd) for k in ("x0", "C", "c", "F", "f")]
    act = b.put(pr["active"].astype(np.uint8), np.uint8)
    o = [b.empty((T, B, n), npd), b.empty((T, B, m), npd), b.empty((T, B, m, n), npd), b.empty((T, B, m), npd)]
    b.ready()
    _, names = profiled(ctx, lambda: ctx.lqr_active_solve(npd, T, B, n, m, d[0], d[1], d[2], d[3], T - 1, d[4], act, *o))
    return dict(x=o[0].get(), u=o[1].get()), names


def check_active(sp, out, names):
    pr = active_problem(sp)
    assert_kernels(names, sp["expect"], absent=("lqr_factor_dmma_warp_kernel",))
    ox, ou = ompc.lqr_active(pr["x0"], pr["C"], pr["c"], pr["F"], pr["f"], pr["active"], sp["n"], sp["m"])
    assert rel_err(out["x"], ox) < tol(sp["dt"]) and rel_err(out["u"], ou) < tol(sp["dt"])
    assert (out["u"][pr["active"]] == 0).all()


def mpcb_problem(sp):
    T, B, n, m = sp["T"], sp["B"], sp["n"], sp["m"]
    rs = np.random.RandomState(sp["seed"])
    C, c = psd_cost(rs, T, B, n + m)
    F = stable_dynamics(rs, T, B, n, m)
    f = 0.1 * rs.randn(T - 1, B, n)
    x0 = rs.randn(B, n)
    u = np.clip(0.5 * rs.randn(T, B, m), -0.4, 0.4)            # about 40 % of the controls sit on a bound
    lo, hi = np.full((T, B, m), -0.4), np.full((T, B, m), 0.4)
    x = ompc.get_traj(x0, u, ("linear", F, f))
    gx, gu = rs.randn(T, B, n), rs.randn(T, B, m)
    return dict(C=C, c=c, F=F, f=f, x=x, u=u, lo=lo, hi=hi, gx=gx, gu=gu)


def run_mpcb(ctx, sp):
    pr = mpcb_problem(sp)
    T, B, n, m = sp["T"], sp["B"], sp["n"], sp["m"]
    s = n + m
    npd = np.float64
    b = Bufs(0)
    d = {k: b.put(v, npd) for k, v in pr.items()}
    ws = [b.empty((T, B, m, n), npd), b.empty((T, B, m), npd), b.empty((T, B, s), npd), b.empty((T, B, m), np.uint8)]
    g = [b.empty((B, n), npd), b.empty((T, B, s, s), npd), b.empty((T, B, s), npd), b.empty((T - 1, B, n, s), npd),
         b.empty((T - 1, B, n), npd)]
    b.ready()
    _, names = profiled(ctx, lambda: ctx.mpc_step_backward(npd, T, B, n, m, d["C"], d["c"], d["F"], T - 1, d["x"], d["u"],
                                                           d["lo"], d["hi"], d["gx"], d["gu"], *ws, *g))
    out = {k: a.get() for k, a in zip(("dx0", "dC", "dc", "dF", "df"), g)}
    out["active"] = ws[3].get()
    return out, names


def check_mpcb(sp, out, names):
    pr = mpcb_problem(sp)
    assert_kernels(names, sp["expect"], absent=("lqr_factor_dmma_warp_kernel",))
    want = ompc.step_backward(pr["C"], pr["c"], pr["F"], pr["f"], pr["x"], pr["u"], pr["lo"], pr["hi"], pr["gx"], pr["gu"],
                              sp["n"], sp["m"])
    for k, w in zip(("dx0", "dC", "dc", "dF", "df"), want):
        assert rel_err(out[k], w) < 1e-10, (k, rel_err(out[k], w))
    act = (np.abs(pr["u"] - pr["lo"]) <= 1e-8) | (np.abs(pr["u"] - pr["hi"]) <= 1e-8)
    assert act.any() and not act.all()
    assert np.array_equal(out["active"].astype(bool), act)


# ------------------------------------------------------------------------------------------------ MPC step forward
def tpe_stash(T, n, B, batch, itemsize=8):
    """Whether mpc_forward_tpe_kernel (four candidate lanes) stashes the candidate trajectories: the shared-memory
    arithmetic of launch_mpc_tpe in csrc/mpc_launch.cu (tpe_kk_stride / tpe_stash_stride of csrc/mpc_tpe_kernel.cuh,
    kMaxSmem = 227 KB; element coupling: 16 elements per CTA within a third of it; batch coupling: the whole batch in one
    CTA of at most 256 threads).  Returns None when the four-lane kernel is not used (one lane per element)."""
    kmax = 227 * 1024
    kk = ((T * (n + 1)) | 1) * itemsize
    ks = kk + 3 * ((T * (n + 2)) | 1) * itemsize
    if batch:
        t4 = (B * 4 + 31) // 32 * 32
        if not (t4 <= 256 and (t4 // 4) * kk <= kmax):
            return None
        return (t4 // 4) * ks <= kmax
    if not 16 * kk <= kmax:
        return None
    return 16 * ks <= kmax // 3


PEND = ((9.5, 1.3, 0.8), 0.03, 1.5)      # PendulumDx (g, m, l), dt, max_torque: none at its default (10, 1, 1), 0.05, 2.0
CAPPED = 5                               # true_cost: elements e % CAPPED == 2 are capped by construction


def mpcf_problem(sp):
    """Model (C, c, F, f) and true problem of one MPC step case.  Keys (all optional): gain = range of the true control
    gain over the model's (linear dynamics); dyn = "pendulum" (true dynamics PEND, model = its linearisation at the
    nominal point, bounds +-2 so that the torque clip at 1.5 is active); expand = False (need_expand = 0: the model c
    is the Taylor-shifted C tau_nom + c and the model f enters the sweep); f = False (no model f); FT = True (F with T
    rows, the last one junk); true_cost = True (a true cost that differs from the model's, and the elements
    e % CAPPED == 2 get 0.5 beta |tau - tau_nom|^2, which every alpha > 0 increases: capped by construction)."""
    T, B, n, m = sp["T"], sp["B"], sp["n"], sp["m"]
    rs = np.random.RandomState(sp["seed"])
    s = n + m
    C, c = psd_cost(rs, T, B, s)
    if sp.get("dyn") == "pendulum":
        assert (n, m) == (3, 1)
        bound = 2.0
        th = rs.uniform(-np.pi, np.pi, B)
        x0 = np.stack((np.cos(th), np.sin(th), 0.5 * rs.randn(B)), axis=1)
        u_nom = np.clip(1.2 * rs.randn(T, B, m), -bound, bound)
        dyn = ("pendulum",) + PEND
        x_nom = ompc.get_traj(x0, u_nom, dyn)
        F, f = opend.linearize(x0, u_nom, *PEND)
        tF = None
        assert ((np.abs(u_nom) > PEND[2]) & (np.abs(u_nom) < bound)).any()
    else:
        bound = 0.5
        F = stable_dynamics(rs, T, B, n, m, per_t=False)
        f = 0.1 * rs.randn(T - 1, B, n)
        tF = F.copy()
        # the true control gain is a multiple of the model's: the full step overshoots and the line search picks a
        # shorter one (the default 1.5 - 3.5 times; 1 - 10 times spreads the accepted trial over 1 ... 8 at decay 0.7)
        glo, ghi = sp.get("gain", (1.5, 3.5))
        tF[..., n:] *= glo + (ghi - glo) * rs.rand(1, B, 1, 1)
        x0 = rs.randn(B, n)
        u_nom = np.clip(0.2 * rs.randn(T, B, m), -bound, bound)
        dyn = ("linear", tF, f)
        x_nom = ompc.get_traj(x0, u_nom, dyn)
    tC, tc = C, c
    capped = np.zeros(B, dtype=bool)
    if sp.get("true_cost"):
        tC, tc = psd_cost(rs, T, B, s)
        tC, tc = 0.5 * (tC + C), 0.5 * (tc + c)
        capped = np.arange(B) % CAPPED == 2
        beta = 2.0
        tau = np.concatenate((x_nom, u_nom), axis=2)
        tC[:, capped] = beta * np.eye(s)
        tc[:, capped] = -beta * tau[:, capped]
    cm, fm = c, f
    if not sp.get("expand", True):
        cm = np.einsum("tbij,tbj->tbi", C, np.concatenate((x_nom, u_nom), axis=2)) + c
        fm = 0.3 * f
    if not sp.get("f", True):
        fm = None
    Fm = np.concatenate((F, 1e3 * rs.randn(1, B, n, s))) if sp.get("FT") else F
    return dict(C=C, c=cm, F=Fm, f=fm, tC=tC, tc=tc, tF=tF, tf=None if tF is None else f, dyn=dyn, x_nom=x_nom,
                u_nom=u_nom, lo=np.full((T, B, m), -bound), hi=np.full((T, B, m), bound), capped=capped)


def mpcf_cap(sp):
    return sp.get("cap", 64) or 64          # max_ls_trials = 0 means 64


def run_mpcf(ctx, sp):
    pr = mpcf_problem(sp)
    T, B, n, m = sp["T"], sp["B"], sp["n"], sp["m"]
    npd = np.float64
    b = Bufs(sp.get("off", 0))
    d = {k: b.put(pr[k], npd) for k in ("C", "c", "F", "f", "tF", "tf", "x_nom", "u_nom", "lo", "hi") if pr[k] is not None}
    for k, km in (("tC", "C"), ("tc", "c")):             # the true cost aliases the model's where it is the same array
        d[k] = d[km] if pr[k] is pr[km] else b.put(pr[k], npd)
    o = dict(x=b.empty((T, B, n), npd), u=b.empty((T, B, m), npd), Ks=b.empty((T, B, m, n), npd), ks=b.empty((T, B, m), npd),
             u_first=b.empty((T, B, m), npd), objs=b.empty((T, B), npd), costs=b.empty((B,), npd), old=b.empty((B,), npd),
             alphas=b.empty((B,), npd), n_qp=b.empty((T, B), np.int32), free=b.empty((T, B, m), np.uint8),
             n_ls=b.empty((B,), np.int32), flags=b.empty((B,), np.int32))
    b.ready()
    coupling = _native.COUPLING_BATCH if sp["batch"] else _native.COUPLING_ELEMENT
    if sp.get("dyn") == "pendulum":
        dyn, dynp = _native.DYN_PENDULUM, PEND[0] + PEND[1:]
    else:
        dyn, dynp = _native.DYN_LINEAR, None

    def go():
        ctx.mpc_step_forward(npd, T, B, n, m, d["C"], d["c"], d["F"], pr["F"].shape[0], d.get("f"), d["x_nom"], d["u_nom"],
                             d["lo"], d["hi"], d["tC"], d["tc"], dyn, d.get("tF"), d.get("tf"), dynp,
                             sp.get("decay", 0.2), sp.get("cap", 64), sp.get("expand", True), coupling, o["x"], o["u"],
                             o["Ks"], o["ks"], o["u_first"], o["objs"], o["costs"], o["old"], o["alphas"], o["n_qp"],
                             o["free"], o["n_ls"], o["flags"])
    _, names = profiled(ctx, go)
    return {k: v.get() for k, v in o.items()}, names


def _pow(decay, k):
    a = 1.0
    for _ in range(k):                       # the line search's repeated multiplication, bit for bit
        a *= decay
    return a


_MPCF_EXPECT = {}


def mpcf_expect(sp):
    """The oracle's step (line search capped at the case's max_ls_trials) and what each output must be, with the checks
    that make the case discriminating: every decisive line-search comparison clears ~1e3 ulp of the old cost, and a
    separate true cost changes the oracle's alphas."""
    key = (case_id(sp), sp["seed"], sp.get("gain"))
    if key in _MPCF_EXPECT:
        return _MPCF_EXPECT[key]
    pr = mpcf_problem(sp)
    T, B, n, m = sp["T"], sp["B"], sp["n"], sp["m"]
    decay, cap = sp.get("decay", 0.2), mpcf_cap(sp)
    coupling = "batch" if sp["batch"] else "element"

    def oracle(cost):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            return ompc.step_forward(pr["C"], pr["c"], pr["F"], pr["f"], pr["x_nom"], pr["u_nom"], pr["lo"], pr["hi"],
                                     cost, pr["dyn"], decay, 10, n, m, need_expand=sp.get("expand", True),
                                     coupling=coupling, max_trials=cap)
    cost = (pr["tC"], pr["tc"])
    ox, ou, fo, aux = oracle(cost)
    old = ompc.traj_cost(pr["x_nom"], pr["u_nom"], cost)
    capped = fo.costs > old
    assert np.array_equal(capped[pr["capped"]], np.ones(pr["capped"].sum(), bool)), "a capped-by-construction element accepted"
    # passes per element: decays of the oracle's alpha + 1 (a capped element's alpha has one decay more than its last pass)
    n_ls = np.zeros(B, dtype=np.int64)
    for e in range(B):
        k = 0
        while _pow(decay, k) != fo.alphas[e]:
            k += 1
            assert k <= cap, (e, fo.alphas[e])
        n_ls[e] = cap if capped[e] else k + 1
    assert (n_ls[capped] == cap).all() and (n_ls <= cap).all()
    if not sp["batch"]:
        assert np.array_equal(n_ls, fo.n_ls), (n_ls, fo.n_ls)           # the per-element recursion counts the same
    alphas = fo.alphas.copy()
    alphas[capped] = _pow(decay, cap - 1)                              # the alpha of the trajectory the last pass wrote
    assert (alphas[capped] * decay == fo.alphas[capped]).all()
    # margins: pass k of element e compares the cost at decay^k with the old cost
    for k in range(int(n_ls.max())):
        al = np.full(B, _pow(decay, k))
        *_, cur = ompc.ls_pass(aux["Ks"], aux["ks"], pr["x_nom"], pr["u_nom"], pr["lo"], pr["hi"], cost, pr["dyn"], al)
        live = k < n_ls
        margin = np.abs(cur - old) / np.spacing(np.abs(old))
        assert (margin[live] > 1e3).all(), ("line-search comparison near a tie", k, margin[live].min())
        assert ((cur > old) == ((k < n_ls - 1) | capped))[live].all(), k
    if sp.get("true_cost"):
        assert (oracle((pr["C"], pr["c"]))[2].alphas != fo.alphas).any(), "the true cost does not change the line search"
    want = dict(x=ox, u=ou, Ks=aux["Ks"], ks=aux["ks"], objs=fo.objs, u_first=fo.u_first, costs=fo.costs, old=old,
                alphas=alphas, n_qp=aux["n_qp"], free=aux["free"], n_ls=n_ls, capped=capped)
    _MPCF_EXPECT[key] = want
    return want


def check_mpcf(sp, out, names):
    T, B, n, m = sp["T"], sp["B"], sp["n"], sp["m"]
    assert_kernels(names, sp["expect"], absent=sp.get("absent", ()))
    if "stash" in sp:
        assert tpe_stash(T, n, B, sp["batch"]) == sp["stash"], (T, n, B, tpe_stash(T, n, B, sp["batch"]))
    w = mpcf_expect(sp)
    assert np.array_equal(out["n_qp"], w["n_qp"])
    assert np.array_equal(out["free"].astype(float), w["free"])
    assert np.array_equal(out["alphas"], w["alphas"]), (out["alphas"], w["alphas"])
    assert np.array_equal(out["n_ls"], w["n_ls"]), ("n_ls", out["n_ls"], w["n_ls"])
    assert np.array_equal((out["flags"] & _native.FLAG_LS_CAPPED) != 0, w["capped"]), (out["flags"], w["capped"])
    assert not (out["flags"] & ~_native.FLAG_LS_CAPPED).any(), out["flags"]
    if sp.get("line_search"):
        assert (w["alphas"] < 1).any(), "no element took a shortened step: the candidate selection is not exercised"
        assert w["alphas"].min() > 1e-6, "an element found no descent: its line search ends on a rounding-level tie"
    tx = 1e-10 if sp["batch"] else 1e-9
    for k in ("Ks", "ks", "objs", "u_first", "costs", "old"):
        assert rel_err(out[k], w[k]) < 1e-10, (k, rel_err(out[k], w[k]))
    assert rel_err(out["x"], w["x"]) < tx and rel_err(out["u"], w["u"]) < tx, (rel_err(out["x"], w["x"]), rel_err(out["u"], w["u"]))


# ------------------------------------------------------------------------------------------------ PNQP
def pnqp_problem(sp):
    B, m = sp["B"], sp["m"]
    rs = np.random.RandomState(sp["seed"])
    Lm = rs.randn(B, m, m)
    H = Lm @ Lm.transpose(0, 2, 1) + 0.5 * np.eye(m)
    return H, 3 * rs.randn(B, m), -rs.rand(B, m), rs.rand(B, m)


def run_pnqp(ctx, sp):
    H, q, lo, hi = pnqp_problem(sp)
    B, m = sp["B"], sp["m"]
    b = Bufs(0)
    d = [b.put(a, np.float64) for a in (H, q, lo, hi)]
    o = [b.empty((B, m), np.float64), b.empty((B, m, m), np.float64), b.empty((B, m), np.int32), b.empty((B, m), np.float64),
         b.empty((B,), np.int32), b.empty((B,), np.int32)]
    b.ready()
    coupling = _native.COUPLING_BATCH if sp["batch"] else _native.COUPLING_ELEMENT
    _, names = profiled(ctx, lambda: ctx.pnqp(np.float64, B, m, *d, None, *o, n_iter=20, coupling=coupling))
    return dict(zip(("x", "LU", "piv", "free", "it", "flags"), (a.get() for a in o))), names


def check_pnqp(sp, out, names):
    H, q, lo, hi = pnqp_problem(sp)
    assert_kernels(names, sp["expect"])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ox, _, ofree, oit = opnqp.pnqp(H, q, lo, hi, coupling="batch" if sp["batch"] else "element")
    assert np.array_equal(out["free"], ofree)
    assert (out["it"] == oit).all()
    assert rel_err(out["x"], ox) < 1e-10
    assert not out["flags"].any()


# ------------------------------------------------------------------------------------------------ case tables
RUN = {"lqr": run_lqr, "active": run_active, "mpcb": run_mpcb, "mpcf": run_mpcf, "pnqp": run_pnqp}
CHECK = {"lqr": check_lqr, "active": check_active, "mpcb": check_mpcb, "mpcf": check_mpcf, "pnqp": check_pnqp}


def L(T, B, n, m, dt, path, G=None, **kw):
    return dict(op="lqr", T=T, B=B, n=n, m=m, dt=dt, path=path, G=G, seed=kw.pop("seed", T * 1009 + B * 7 + n * 3 + m), **kw)


def MF(T, B, n, m, batch, seed, expect, **kw):
    """An MPC step forward case; the cases with a line-search decay of their own spread the true control gain over 1 - 10
    times the model's."""
    if "decay" in kw and kw.get("dyn") != "pendulum":
        kw.setdefault("gain", (1.0, 10.0))
    return dict(op="mpcf", T=T, B=B, n=n, m=m, batch=batch, seed=seed, expect=[expect], **kw)


def TPE(n, batch, NA):
    return "mpc_forward_tpe_kernel<double, %d, %s, 256, %d>" % (n, "true" if batch else "false", NA)


def GRP(N, M, G, batch):
    return "mpc_forward_kernel<double, %d, %d, %d, %s>" % (N, M, G, "true" if batch else "false")


def case_id(sp):
    bits = [sp["op"], "T%d" % sp.get("T", 1), "B%d" % sp["B"], "n%dm%d" % (sp["n"], sp["m"]), sp.get("dt", F64)]
    for k in ("path", "pivot", "off", "reduced", "batch", "dyn", "true_cost", "decay"):
        if sp.get(k) not in (None, False, 0):
            bits.append(k if sp[k] is True else "%s%s" % (k, sp[k]))
    for k, v in (("expand", False), ("f", False)):
        if sp.get(k, True) is v:
            bits.append("no" + k)
    if sp.get("FT"):
        bits.append("FT")
    if "cap" in sp:
        bits.append("cap%d" % sp["cap"])
    return "-".join(str(b) for b in bits)


DEFAULT = [
    # runtime-shape group kernels, s <= 6 outside the three thread-per-element shapes (G = 8), m > n included
    L(1, 5, 1, 1, F64, "group", 8), L(2, 37, 2, 2, F64, "group", 8), L(2, 37, 2, 2, F32, "group", 8),
    L(9, 300, 3, 2, F64, "group", 8), L(7, 33, 5, 1, F64, "group", 8), L(6, 17, 1, 5, F64, "group", 8),
    L(5, 130, 3, 3, F64, "group", 8),
    # G = 16, 32, 256, m > n
    L(8, 21, 2, 6, F64, "group", 16, reduced=True), L(8, 21, 2, 6, F32, "group", 16),
    L(6, 9, 4, 12, F64, "group", 32), L(6, 9, 4, 12, F32, "group", 32), L(2, 5, 2, 22, F64, "group", 32),
    L(5, 3, 8, 24, F64, "group", 256), L(5, 3, 8, 24, F32, "group", 256), L(4, 3, 1, 32, F64, "group", 256),
    # row swaps in every m = 2 step: thread-per-element (4,2), a runtime group shape, the DMMA kernel at (32,8)
    L(12, 40, 4, 2, F64, "tpe", 8, pivot=True), L(12, 40, 3, 2, F64, "group", 8, pivot=True),
    L(10, 6, 32, 8, F64, "dmma", pivot=True),
    # config 5 at T = 100 on the DMMA kernel (setting no_dmma runs the same inputs on the group kernel)
    L(100, 33, 32, 8, F64, "dmma", seed=77, reduced=True),
    # pointers one element past a 16-byte boundary: (32,8) leaves the DMMA kernel for the group kernel + fused adjoint
    L(6, 7, 32, 8, F64, "fused", off=1, reduced=True), L(6, 7, 32, 8, F32, "fused", off=1, reduced=True),
    L(7, 45, 4, 2, F64, "tpe", G=8, off=1, reduced=True),
    # LQR_active (masked group kernel) and the MPC backward (masked solve with the split cx/cu right-hand side, c_scale -1)
    dict(op="active", T=6, B=5, n=32, m=8, dt=F64, seed=41, expect=["lqr_solve_kernel<double, 32, 8, 256>"]),
    dict(op="active", T=9, B=23, n=3, m=2, dt=F64, seed=42, expect=["lqr_solve_kernel<double, 0, 0, 8>"]),
    dict(op="active", T=9, B=23, n=3, m=2, dt=F64, seed=43, pivot=True, expect=["lqr_solve_kernel<double, 0, 0, 8>"]),
    dict(op="mpcb", T=6, B=5, n=32, m=8, seed=51,
         expect=["lqr_solve_kernel<double, 32, 8, 256>", "adjoint_out_kernel<double, 32, 8, 128, false>"]),
    dict(op="mpcb", T=8, B=21, n=3, m=2, seed=52,
         expect=["lqr_solve_kernel<double, 0, 0, 8>", "adjoint_out_kernel<double, 0, 0, 8, false>"]),
    dict(op="mpcb", T=7, B=9, n=2, m=4, seed=53,
         expect=["lqr_solve_kernel<double, 0, 0, 8>", "adjoint_out_kernel<double, 0, 0, 8, false>"]),
    # MPC step forward, m = 1: thread-per-element kernel past the candidate stash, and with one lane per element
    dict(op="mpcf", T=40, B=20, n=3, m=1, batch=False, seed=61, stash=False, line_search=True,
         expect=["mpc_forward_tpe_kernel<double, 3, false, 256, 4>"]),
    dict(op="mpcf", T=45, B=20, n=2, m=1, batch=False, seed=62, stash=False, line_search=True,
         expect=["mpc_forward_tpe_kernel<double, 2, false, 256, 4>"]),
    dict(op="mpcf", T=30, B=64, n=3, m=1, batch=True, seed=63, stash=False, line_search=True,
         expect=["mpc_forward_tpe_kernel<double, 3, true, 256, 4>"]),
    dict(op="mpcf", T=20, B=150, n=3, m=1, batch=True, seed=64, stash=None, line_search=True,
         expect=["mpc_forward_tpe_kernel<double, 3, true, 256, 1>"]),
    # runtime-shape group MPC kernel with m > n, and the MPC step on misaligned buffers
    dict(op="mpcf", T=8, B=9, n=2, m=3, batch=False, seed=65, expect=["mpc_forward_kernel<double, 0, 0, 8, false>"]),
    dict(op="mpcf", T=8, B=21, n=4, m=2, batch=False, seed=66, off=1, expect=["mpc_forward_kernel<double, 4, 2, 8, false>"]),
    # MPC step forward, the whole contract: a separate true cost (with elements capped by construction), the line-search
    # cap (max_ls_trials 1 ... 6 and 0 = 64, every residue mod 4 with and without the stash), decays 0.7 / 0.9 (the
    # accepted trial spreads over the four candidate lanes and later rounds), need_expand = 0 with / without the model f,
    # F with T rows, and the pendulum at non-default g, m, l, dt, max_torque.  Four lanes, stash:
    MF(20, 16, 3, 1, False, 143, TPE(3, False, 4), stash=True, true_cost=True, decay=0.7, cap=1),
    MF(20, 24, 3, 1, True, 102, TPE(3, True, 4), stash=True, true_cost=True, decay=0.7, cap=2, expand=False),
    MF(20, 16, 2, 1, False, 103, TPE(2, False, 4), stash=True, true_cost=True, decay=0.7, cap=3),
    MF(20, 16, 2, 1, True, 104, TPE(2, True, 4), stash=True, true_cost=True, decay=0.9, cap=0),
    MF(20, 16, 3, 1, False, 105, TPE(3, False, 4), stash=True, true_cost=True, decay=0.9, cap=0, dyn="pendulum"),
    MF(20, 20, 3, 1, True, 106, TPE(3, True, 4), stash=True, true_cost=True, decay=0.7, cap=6, dyn="pendulum"),
    # four lanes, no stash
    MF(40, 16, 3, 1, False, 107, TPE(3, False, 4), stash=False, true_cost=True, decay=0.7, cap=5),
    MF(30, 64, 3, 1, True, 108, TPE(3, True, 4), stash=False, true_cost=True, decay=0.7, cap=6),
    MF(45, 16, 2, 1, False, 109, TPE(2, False, 4), stash=False, true_cost=True, decay=0.9, cap=0, expand=False),
    MF(32, 64, 2, 1, True, 110, TPE(2, True, 4), stash=False, true_cost=True, decay=0.7, cap=3, FT=True),
    MF(40, 16, 3, 1, False, 111, TPE(3, False, 4), stash=False, true_cost=True, decay=0.7, cap=4, expand=False, f=False),
    # one lane per element (batch coupling past 64 elements)
    MF(20, 100, 3, 1, True, 112, TPE(3, True, 1), stash=None, true_cost=True, decay=0.7, cap=5),
    # group kernels: specialised <4,2,8> <8,4,16>, runtime shape G = 8 / 16 / 32 / 256, both couplings
    MF(8, 21, 4, 2, True, 113, GRP(4, 2, 8, True), true_cost=True, decay=0.7, cap=3),
    MF(8, 21, 4, 2, False, 114, GRP(4, 2, 8, False), true_cost=True, decay=0.9, cap=0, expand=False, f=False, FT=True),
    MF(6, 10, 8, 4, False, 115, GRP(8, 4, 16, False), true_cost=True, decay=0.9, cap=0),
    MF(6, 10, 8, 4, True, 116, GRP(8, 4, 16, True), true_cost=True, decay=0.7, cap=5, expand=False),
    MF(8, 9, 2, 3, False, 117, GRP(0, 0, 8, False), true_cost=True, decay=0.7, cap=2, expand=False, FT=True),
    MF(8, 9, 2, 3, True, 118, GRP(0, 0, 8, True), true_cost=True, decay=0.9, cap=0),
    MF(6, 9, 6, 5, False, 119, GRP(0, 0, 16, False), true_cost=True, decay=0.7, cap=4),
    MF(6, 9, 6, 5, True, 120, GRP(0, 0, 16, True), true_cost=True, decay=0.7, cap=6, expand=False),
    MF(5, 7, 12, 6, False, 121, GRP(0, 0, 32, False), true_cost=True, decay=0.9, cap=0, expand=False, f=False),
    MF(5, 7, 12, 6, True, 122, GRP(0, 0, 32, True), true_cost=True, decay=0.7, cap=3),
    MF(6, 3, 32, 8, False, 123, GRP(0, 0, 256, False), true_cost=True, decay=0.7, cap=4, expand=False),
    # PNQP with 17 <= m <= 32: 32 lanes per element
    dict(op="pnqp", B=40, n=0, m=20, batch=False, seed=91, expect=["pnqp_kernel<double, 0, 32, false>"]),
    dict(op="pnqp", B=17, n=0, m=32, batch=False, seed=92, expect=["pnqp_kernel<double, 0, 32, false>"]),
    dict(op="pnqp", B=9, n=0, m=24, batch=True, seed=93, expect=["pnqp_kernel<double, 0, 32, true>"]),
]


def _grp(n, m, dt, path, G, masked=False):
    R = CNAME[dt]
    if masked:
        return dict(op="active", T=9, B=37, n=n, m=m, dt=dt, seed=70 + n, expect=["lqr_solve_kernel<%s, %d, %d, %d>" % (R, n, m, G)])
    return L(9, 37, n, m, dt, path, G)


def _tpe_adj_group(n, m, dt, G):
    sp = L(9, 37, n, m, dt, "tpe", G)
    sp["path"] = "tpe_adj_group"
    return sp


_M1_BATCH = dict(T=20, B=64, n=3, m=1, batch=True, seed=81, line_search=True)
_M1_ELEM = dict(T=20, B=40, n=3, m=1, batch=False, seed=82, line_search=True)

CHILD = {
    "lqr_group": (dict(DMPC_LQR_GROUP="1"),
                  [_grp(n, m, dt, "spec", G, masked) for (n, m, G) in ((2, 1, 4), (3, 1, 4), (4, 2, 8))
                   for dt in (F64, F32) for masked in (False, True)]),
    "adj_group": (dict(DMPC_ADJ_GROUP="1"),
                  [_tpe_adj_group(n, m, dt, G) for (n, m, G) in ((2, 1, 4), (3, 1, 4), (4, 2, 8)) for dt in (F64, F32)]),
    "epw8": (dict(DMPC_LQR_TPE_EPW="8"), [L(5, B, 4, 2, F64, "tpe", G=8) for B in (37, 9601, 19003)]),
    "epw16": (dict(DMPC_LQR_TPE_EPW="16"), [L(5, B, 4, 2, F64, "tpe", G=8) for B in (37, 9601, 19003)]),
    "epw_auto": (dict(DMPC_LQR_TPE_EPW="auto"),
                 [L(5, B, 4, 2, F64, "tpe", G=8) for B in (37, 9601, 19003)] +
                 [L(T, B, n, m, F64, "tpe", G=G) for (T, B, n, m, G) in ((50, 4096, 4, 2, 8), (20, 8192, 3, 1, 4),
                                                                         (7, 4737, 4, 2, 8), (6, 130, 2, 1, 4))]),
    "no_dmma": (dict(DMPC_DISABLE_DMMA="1"), [L(100, 33, 32, 8, F64, "fused", seed=77, reduced=True),
                                             L(10, 6, 32, 8, F64, "fused", pivot=True)]),
    "adj_unfused": (dict(DMPC_ADJ_UNFUSED="1"), [L(8, 21, 32, 8, F64, "unfused", 256, reduced=True)]),
    "mpc_group": (dict(DMPC_MPC_GROUP="1"),
                  [dict(_M1_BATCH, op="mpcf", expect=["mpc_forward_kernel<double, 3, 1, 4, true>"]),
                   dict(_M1_ELEM, op="mpcf", expect=["mpc_forward_kernel<double, 3, 1, 4, false>"]),
                   MF(20, 16, 3, 1, False, 131, GRP(3, 1, 4, False), true_cost=True, decay=0.7, cap=5, dyn="pendulum"),
                   MF(20, 20, 3, 1, True, 132, GRP(3, 1, 4, True), true_cost=True, decay=0.9, cap=0, dyn="pendulum"),
                   MF(20, 24, 3, 1, True, 133, GRP(3, 1, 4, True), true_cost=True, decay=0.7, cap=2, expand=False)]),
    "mpc_no_spec": (dict(DMPC_MPC_NO_SPEC="1"),
                    [dict(_M1_BATCH, op="mpcf", expect=["mpc_forward_tpe_kernel<double, 3, true, 256, 1>"]),
                     dict(_M1_ELEM, op="mpcf", expect=["mpc_forward_tpe_kernel<double, 3, false, 256, 1>"]),
                     MF(20, 16, 3, 1, False, 134, TPE(3, False, 1), true_cost=True, decay=0.7, cap=3, dyn="pendulum"),
                     MF(20, 24, 2, 1, True, 135, TPE(2, True, 1), true_cost=True, decay=0.9, cap=0, expand=False)]),
    # the default launch would stash at these horizons (stash=True); the switch turns the stash off, same kernel
    "mpc_no_stash": (dict(DMPC_MPC_NO_STASH="1"),
                     [dict(_M1_BATCH, op="mpcf", stash=True, expect=["mpc_forward_tpe_kernel<double, 3, true, 256, 4>"]),
                      dict(_M1_ELEM, op="mpcf", stash=True, expect=["mpc_forward_tpe_kernel<double, 3, false, 256, 4>"]),
                      MF(20, 16, 3, 1, False, 136, TPE(3, False, 4), stash=True, true_cost=True, decay=0.7, cap=3),
                      MF(20, 24, 3, 1, True, 137, TPE(3, True, 4), stash=True, true_cost=True, decay=0.9, cap=0,
                         dyn="pendulum")]),
}


# ------------------------------------------------------------------------------------------------ tests
@pytest.fixture(scope="module")
def ctx():
    return _native.default_context(0)


@pytest.mark.parametrize("sp", DEFAULT, ids=case_id)
def test_default_dispatch(ctx, sp):
    out, names = RUN[sp["op"]](ctx, sp)
    CHECK[sp["op"]](sp, out, names)


_CHILD_RESULTS = {}


def _child_results(setting):
    """Runs the cases of one A/B setting in a child process (once per test session) and loads its outputs."""
    if setting not in _CHILD_RESULTS:
        env = {k: v for k, v in os.environ.items() if not k.startswith("DMPC_")}
        env.update(CHILD[setting][0])
        with tempfile.TemporaryDirectory() as td:
            path = os.path.join(td, "out.npz")
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", setting, path], env=env,
                               capture_output=True, text=True, timeout=600)
            assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-4000:])
            with np.load(path, allow_pickle=False) as z:
                _CHILD_RESULTS[setting] = {k: z[k] for k in z.files}
    return _CHILD_RESULTS[setting]


@pytest.mark.parametrize("setting,sp", [(s, sp) for s, (_, cases) in CHILD.items() for sp in cases],
                         ids=[s + ":" + case_id(sp) for s, (_, cases) in CHILD.items() for sp in cases])
def test_ab_switch(setting, sp):
    res = _child_results(setting)
    cid = case_id(sp) + "/"
    out = {k[len(cid):]: v for k, v in res.items() if k.startswith(cid)}
    names = list(out.pop("__kernels__"))
    CHECK[sp["op"]](sp, out, names)


def test_mpcf_four_lane_coverage():
    """Together, the cases of the four-lane MPC kernel (mpc_forward_tpe_kernel<..., 4>) have winners on every candidate
    lane (n_ls mod 4) and in a later round, and line-search caps at every residue mod 4 (the capped winner's lane is
    (cap - 1) mod 4), both with the candidate stash and without it.  From the oracle."""
    lanes, late, caps = set(), False, {True: set(), False: set()}
    for setting, sp in [(None, sp) for sp in DEFAULT] + [(s, sp) for s, (_, cs) in CHILD.items() for sp in cs]:
        if sp["op"] != "mpcf" or not any(k.startswith("mpc_forward_tpe_kernel") and k.endswith(", 4>") for k in sp["expect"]):
            continue
        w = mpcf_expect(sp)
        won = w["n_ls"][~w["capped"]]
        lanes |= set((won - 1) % 4)
        late |= bool((won > 4).any())
        if w["capped"].any():
            caps[bool(sp["stash"]) and setting != "mpc_no_stash"].add(mpcf_cap(sp) % 4)
    assert lanes == {0, 1, 2, 3} and late, (lanes, late)
    assert caps[True] == {0, 1, 2, 3} and caps[False] == {0, 1, 2, 3}, caps


def _child_main(setting, path):
    ctx = _native.default_context(0)
    save = {}
    for sp in CHILD[setting][1]:
        out, names = RUN[sp["op"]](ctx, sp)
        cid = case_id(sp) + "/"
        for k, v in out.items():
            save[cid + k] = v
        save[cid + "__kernels__"] = np.array(names if names else [""], dtype=str)
    np.savez(path, **save)
    ctx.close()


if __name__ == "__main__":
    assert sys.argv[1] == "--child", sys.argv
    _child_main(sys.argv[2], sys.argv[3])
