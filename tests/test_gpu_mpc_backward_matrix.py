"""GPU: the MPC step backward (dmpc_mpc_step_backward / dmpc_mpc_step_backward_reduced) and dmpc_lqr_active_solve on every
kernel they can select, against the fp64 oracle (oracle.mpc.step_backward / lqr_active).

The backward is active_mask_kernel, then the masked LQR solve with c := -d_taus (split cx | cu right-hand side, c_scale -1,
output into tau_out), then adjoint_out_tpe_kernel / adjoint_out_kernel with ADJ_NEGATE | ADJ_NEG_RHS, and for the reduced
call reduce_partials_kernel (csrc/capi.cu mpc_backward_impl).  Every case runs both calls, each under torch.profiler, and
asserts the kernels that ran, as tests/test_gpu_dispatch_matrix.py does (whose device buffers and profiler helpers this
file uses).  The A/B switches DMPC_LQR_GROUP, DMPC_ADJ_GROUP and DMPC_LQR_TPE_EPW are read once per process, so each
setting runs its cases in a child process (`python test_gpu_mpc_backward_matrix.py --child SETTING OUT.npz`); the
default-path cases run in a child of their own (setting "default"), and the parent checks every output.

Problem keys (mpcb_problem; mpc_step.py:330-460 is the contract):
  sym = False   C plus a non-symmetric part (the lambda recursion reads the top n rows of C_t, the masked solve Qux and
                Qxu separately: a transposed index passes with symmetric C)
  FT            F with T rows, the last one junk: the last row of dF must come back zero (the buffers start as NaN)
  f = False     no f: df = NULL
  grads         "both", "u_only" (gx = NULL: the imitation-learning call) or "x_only" (gu = NULL)
  band          controls at lo + delta, delta in {0, 0.5e-8, 1e-8, 1e-8 (1 + 2^-40), 2e-8} with lo = 0 (exact
                subtraction), outside the box by 1e-9 and 1e-6, and lo == hi: the mask |u - lo| <= 1e-8 or |u - hi| <= 1e-8
                is checked bit for bit, so < for <= or a float threshold in the double kernel fails
  off = 1       every tensor one element past a 16-byte boundary
Bounds vary per (t, b); in every case the elements b % 4 == 0 have every control active at t = T // 2 and the elements
b % 4 == 1 none.  x is get_traj of u through F, f.

Checks: the active mask bit-exact; the full call's dx0, dC, dc, dF (all F_T rows) and df at 1e-10 element-relative in fp64,
1e-3 in fp32 (the oracle runs on the fp32-rounded inputs), on dm.slices(B) for large batches; the reduced call's dx0 at the
same tolerance and each entry of the four (T,B)-sums within tol x sum_{t,b} |term| of the oracle's full gradients summed
(tol = 1e-10 fp64, 2e-5 fp32: the right scale for a sum that cancels).  Each case asserts from the oracle that the sums
without element B - 1, and without the last step, violate that bound, so a reduction that drops the partial last CTA or
the last step fails.  A second reduced call returns bit-identical sums.
"""
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

if __name__ == "__main__":                       # child process: the import paths tests/conftest.py sets up
    _root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    _pkg = os.path.join(_root, "chainer-differentiable-mpc_b200")
    for _p in (os.path.dirname(os.path.abspath(__file__)), _root, _pkg):
        if _p not in sys.path:
            sys.path.insert(0, _p)

import _native
import test_gpu_dispatch_matrix as dm
from _helpers import rel_err, psd_cost, stable_dynamics, lqr_problem
from oracle import mpc as ompc

F64, F32 = dm.F64, dm.F32
NP, CNAME = dm.NP, dm.CNAME
SPEC = {(2, 1): 4, (3, 1): 4, (4, 2): 8, (8, 4): 16, (32, 8): 256}     # DMPC_SHAPES of csrc/lqr_launch.cu
TPE = ((2, 1), (3, 1), (4, 2))
ACT_TOL = 1e-8                                                        # mpc_step.py:363-364

# band entries (u, lo, hi) and whether the control is active
BAND = [(0.0, 0.0, 0.5, True), (0.5e-8, 0.0, 0.5, True), (1e-8, 0.0, 0.5, True), (1e-8 * (1 + 2.0 ** -40), 0.0, 0.5, False),
        (2e-8, 0.0, 0.5, False), (-1e-9, 0.0, 0.5, True), (-1e-6, 0.0, 0.5, False), (0.5 + 1e-9, 0.0, 0.5, True),
        (0.5 + 1e-6, 0.0, 0.5, False), (0.3, 0.3, 0.3, True), (-0.2, -0.2, -0.2, True)]


def gtol(dt):
    return 1e-10 if dt == F64 else 1e-3


def stol(dt):
    return 1e-10 if dt == F64 else 2e-5


def r32(a):
    return None if a is None else a.astype(np.float32).astype(np.float64)


# ------------------------------------------------------------------------------------------------ problems
def extreme_rows(T, B, m):
    """[T,B] masks of the rows forced all-active (b % 4 == 0) and none-active (b % 4 == 1) at t = T // 2.  Element B - 1
    has no active control at T - 1 (at T = 1 an all-active last element would add nothing to the sums, and the
    dropped-element check could not tell it missing)."""
    allr, noner = np.zeros((T, B), bool), np.zeros((T, B), bool)
    allr[T // 2, 0:B - 1:4] = True
    noner[T // 2, 1::4] = True
    noner[T - 1, B - 1] = True
    return allr, noner


def mpcb_problem(sp):
    T, B, n, m = sp["T"], sp["B"], sp["n"], sp["m"]
    s = n + m
    rs = np.random.RandomState(sp["seed"])
    C, c = psd_cost(rs, T, B, s, sym=sp.get("sym", True))
    F = stable_dynamics(rs, T, B, n, m)
    if T == 1:
        F = np.zeros((0, B, n, s))
    f = 0.1 * rs.randn(T - 1, B, n) if sp.get("f", True) else None
    x0 = rs.randn(B, n)
    lo = -(0.2 + 0.4 * rs.rand(T, B, m))
    hi = 0.2 + 0.4 * rs.rand(T, B, m)
    u = np.clip(0.5 * rs.randn(T, B, m), lo, hi)
    allr, noner = extreme_rows(T, B, m)
    ext = np.repeat((allr | noner)[:, :, None], m, axis=2)
    sgn = np.where(np.arange(m) % 2 == 0, 0, 1)[None, :]
    u[allr] = np.where(sgn == 0, lo[allr], hi[allr])
    u[noner] = 0.5 * (lo[noner] + hi[noner])
    band = np.zeros((T, B, m), bool)
    if sp.get("band"):
        k = 0
        for t in range(T):
            for b in range(B):
                if (t * B + b) % 2 or ext[t, b, 0]:
                    continue
                u[t, b, 0], lo[t, b, 0], hi[t, b, 0], _ = BAND[k % len(BAND)]
                band[t, b, 0] = True
                k += 1
    x = ompc.get_traj(x0, u, ("linear", F, f))
    if sp.get("FT") or T == 1:
        F = np.concatenate((F, 1e3 * rs.randn(1, B, n, s)))           # the junk last row (F with T rows)
    grads = sp.get("grads", "both")
    gx = rs.randn(T, B, n) if grads != "u_only" else None
    gu = rs.randn(T, B, m) if grads != "x_only" else None
    pr = dict(C=C, c=c, F=F, f=f, x=x, u=u, lo=lo, hi=hi, gx=gx, gu=gu)
    if sp["dt"] == F32:
        pr = {k: r32(v) for k, v in pr.items()}
    pr.update(band=band, ext=ext, allr=allr, noner=noner)
    return pr


def mask_of(pr):
    return (np.abs(pr["u"] - pr["lo"]) <= ACT_TOL) | (np.abs(pr["u"] - pr["hi"]) <= ACT_TOL)


def idx_of(B):
    return np.concatenate([np.arange(B)[sl] for sl in dm.slices(B)])


_EXPECT = {}


def mpcb_expect(sp):
    """The oracle's full gradients (on the elements of dm.slices(B)), dx0, the active mask, and the (T,B)-sums with their
    scales sum |term|; asserts that dropping element B - 1 or the last step of each sum violates the sum bound."""
    key = (case_id(sp), sp["seed"])
    if key in _EXPECT:
        return _EXPECT[key]
    pr = mpcb_problem(sp)
    T, B, n, m, dt = sp["T"], sp["B"], sp["n"], sp["m"], sp["dt"]
    f = pr["f"] if pr["f"] is not None else np.zeros((T - 1, B, n))   # step_backward reads f only for df's presence
    dx0, dC, dc, dF, df = ompc.step_backward(pr["C"], pr["c"], pr["F"], f, pr["x"], pr["u"], pr["lo"], pr["hi"], pr["gx"],
                                             pr["gu"], n, m)
    idx = idx_of(B)
    want = dict(active=mask_of(pr), dx0=dx0, idx=idx, dC=dC[:, idx], dc=dc[:, idx], dF=dF[:, idx], df=df[:, idx])
    tol = stol(dt)
    terms = dict(dC=dC, dc=dc, dF=dF[:T - 1], df=df)
    for k, a in terms.items():
        w, S = a.sum(axis=(0, 1)), np.abs(a).sum(axis=(0, 1))
        want["sum_" + k], want["abs_" + k] = w, S
        if a.shape[0] == 0:
            continue
        # the bound catches a reduction that loses element B - 1, or the last step of the sum
        last = a.shape[0] - 1
        for drop in (a[:, :B - 1].sum(axis=(0, 1)), a[:last].sum(axis=(0, 1))):
            assert (np.abs(drop - w) > tol * S).any(), ("sum bound does not catch a dropped term", k)
    _EXPECT[key] = want
    return want


def mpcb_kernels(sp, setting=None):
    """(expected substrings of the full call, of the reduced call, absent substrings of both)."""
    n, m, R = sp["n"], sp["m"], CNAME[sp["dt"]]
    s = n + m
    G = SPEC.get((n, m)) or (8 if s <= 6 else (16 if s <= 14 else (32 if s <= 24 else 256)))
    N, M = (n, m) if (n, m) in SPEC else (0, 0)
    Ga = G if G <= 32 else 128
    tpe = (n, m) in TPE
    solve = ("lqr_tpe_kernel<%s, %d, %d," % (R, n, m)) if tpe and setting != "lqr_group" else \
        "lqr_solve_kernel<%s, %d, %d, %d>" % (R, N, M, G)
    full_adj = ("adjoint_out_tpe_kernel<%s, %d, %d," % (R, n, m)) if tpe and setting not in ("lqr_group", "adj_group") else \
        "adjoint_out_kernel<%s, %d, %d, %d, false>" % (R, N, M, Ga)
    mask = "active_mask_kernel<%s>" % R
    absent = ["lqr_factor_dmma_warp_kernel"]
    if setting == "lqr_group":
        absent += ["lqr_tpe_kernel", "adjoint_out_tpe_kernel"]
    if setting == "adj_group":
        absent += ["adjoint_out_tpe_kernel"]
    return ([mask, solve, full_adj], [mask, solve, "adjoint_out_kernel<%s, %d, %d, %d, true>" % (R, N, M, Ga),
                                      "reduce_partials_kernel<%s>" % R], absent)


# ------------------------------------------------------------------------------------------------ run / check
def run_mpcb(ctx, sp):
    pr = mpcb_problem(sp)
    T, B, n, m, npd = sp["T"], sp["B"], sp["n"], sp["m"], NP[sp["dt"]]
    s, FT = n + m, pr["F"].shape[0]
    b = dm.Bufs(sp.get("off", 0))
    d = {k: (None if pr[k] is None else b.put(pr[k], npd)) for k in ("C", "c", "F", "x", "u", "lo", "hi", "gx", "gu")}
    args = (npd, T, B, n, m, d["C"], d["c"], d["F"], FT, d["x"], d["u"], d["lo"], d["hi"], d["gx"], d["gu"])

    def ws():      # the active buffer starts as 7: an entry the mask kernel does not write fails the comparison
        return [b.empty((T, B, m, n), npd), b.empty((T, B, m), npd), b.empty((T, B, s), npd),
                b.put(np.full((T, B, m), 7, np.uint8), np.uint8)]
    wf = ws()
    g = [b.empty((B, n), npd), b.empty((T, B, s, s), npd), b.empty((T, B, s), npd), b.empty((FT, B, n, s), npd),
         b.empty((T - 1, B, n), npd) if (pr["f"] is not None and T > 1) else None]
    rsz = ctx.reduced_grad_elems(n, m)
    red = [ws() for _ in range(2)]
    ro = [[b.empty((B, rsz), npd), b.empty((B, n), npd), b.empty((rsz,), npd)] for _ in range(2)]
    b.ready()
    _, names_full = dm.profiled(ctx, lambda: ctx.mpc_step_backward(*args, *wf, *g))
    _, names_red = dm.profiled(ctx, lambda: ctx.mpc_step_backward_reduced(*args, *red[0], *ro[0]))
    ctx.mpc_step_backward_reduced(*args, *red[1], *ro[1])
    ctx.sync()
    out = {"full_" + k: a.get() for k, a in zip(("dx0", "dC", "dc", "dF", "df"), g) if a is not None}
    out["full_active"] = wf[3].get()
    for i in range(2):
        out["red%d_active" % i], out["red%d_dx0" % i], out["red%d_sums" % i] = red[i][3].get(), ro[i][1].get(), ro[i][2].get()
    return out, names_full, names_red


def check_mpcb(sp, out, names_full, names_red, setting=None):
    T, B, n, m, dt = sp["T"], sp["B"], sp["n"], sp["m"], sp["dt"]
    ek_full, ek_red, absent = mpcb_kernels(sp, setting)
    dm.assert_kernels(names_full, ek_full, absent=absent + ["reduce_partials_kernel"])
    dm.assert_kernels(names_red, ek_red, absent=absent + ["adjoint_out_tpe_kernel"])
    w = mpcb_expect(sp)
    for k in ("full_active", "red0_active"):
        assert np.array_equal(out[k], w["active"].astype(np.uint8)), (k, np.argwhere(out[k] != w["active"])[:8])
    tg = gtol(dt)
    # full call: every output on the slices, the last row of dF (F with T rows) exactly zero
    assert rel_err(out["full_dx0"], w["dx0"]) < tg, ("dx0", rel_err(out["full_dx0"], w["dx0"]))
    idx = w["idx"]
    for k in ("dC", "dc", "dF", "df"):
        if k == "df" and (sp.get("f", True) is False or T == 1):
            assert "full_df" not in out
            continue
        e = rel_err(out["full_" + k][:, idx], w[k])
        assert e < tg, (k, e)
    if out["full_dF"].shape[0] == T:
        assert (out["full_dF"][T - 1] == 0).all(), "dF row T-1 is not zero"
    # reduced call: dx0, the sums against the oracle within tol x sum |term|, bit-identical on a second call
    assert rel_err(out["red0_dx0"], w["dx0"]) < tg, ("reduced dx0", rel_err(out["red0_dx0"], w["dx0"]))
    tol = stol(dt)
    sums = _native.Context.split_reduced(out["red0_sums"].astype(np.float64), n, m)
    for k, a in zip(("dC", "dc", "dF", "df"), sums):
        err = np.abs(a - w["sum_" + k])
        bound = tol * w["abs_" + k]
        assert (err <= bound).all(), ("reduced", k, float(np.max(err - bound)), float(np.max(err / np.maximum(w["abs_" + k], 1e-300))))
    assert np.array_equal(out["red0_sums"], out["red1_sums"]) and np.array_equal(out["red0_dx0"], out["red1_dx0"]), \
        "reduced call not deterministic"
    assert np.array_equal(out["red1_active"], out["red0_active"])


# ------------------------------------------------------------------------------------------------ dmpc_lqr_active_solve
def la_problem(sp):
    T, B, n, m = sp["T"], sp["B"], sp["n"], sp["m"]
    pr = lqr_problem(sp["seed"], T, B, n, m, with_f=sp.get("f", True), sym=sp.get("sym", True))
    rs = np.random.RandomState(sp["seed"] + 1)
    act = rs.rand(T, B, m) < 0.4
    allr, noner = extreme_rows(T, B, m)
    act[allr], act[noner] = True, False
    out = dict(x0=pr["x0"], C=pr["C"], c=pr["c"], F=pr["F"], f=pr["f"])
    if sp["dt"] == F32:
        out = {k: r32(v) for k, v in out.items()}
    out.update(active=act, allr=allr, noner=noner)
    return out


def run_la(ctx, sp):
    pr = la_problem(sp)
    T, B, n, m, npd = sp["T"], sp["B"], sp["n"], sp["m"], NP[sp["dt"]]
    b = dm.Bufs(sp.get("off", 0))
    d = {k: (None if pr[k] is None else b.put(pr[k], npd)) for k in ("x0", "C", "c", "F", "f")}
    act = b.put(pr["active"].astype(np.uint8), np.uint8)
    o = [b.empty((T, B, n), npd), b.empty((T, B, m), npd), b.empty((T, B, m, n), npd), b.empty((T, B, m), npd)]
    b.ready()
    _, names = dm.profiled(ctx, lambda: ctx.lqr_active_solve(npd, T, B, n, m, d["x0"], d["C"], d["c"], d["F"], T - 1,
                                                             d["f"], act, *o))
    return dict(x=o[0].get(), u=o[1].get()), names


def la_expect(sp):
    pr = la_problem(sp)
    return ompc.lqr_active(pr["x0"], pr["C"], pr["c"], pr["F"], pr["f"], pr["active"], sp["n"], sp["m"])


def check_la(sp, out, names):
    solve = mpcb_kernels(sp)[0][1]
    dm.assert_kernels(names, [solve], absent=("lqr_factor_dmma_warp_kernel",))
    pr = la_problem(sp)
    ox, ou = la_expect(sp)
    t = dm.tol(sp["dt"])
    assert rel_err(out["x"], ox) < t and rel_err(out["u"], ou) < t, (rel_err(out["x"], ox), rel_err(out["u"], ou))
    assert (out["u"][pr["active"]] == 0).all()


# ------------------------------------------------------------------------------------------------ case tables
def case_id(sp):
    bits = [sp["op"], "T%d" % sp["T"], "B%d" % sp["B"], "n%dm%d" % (sp["n"], sp["m"]), sp["dt"]]
    if sp.get("sym", True) is False:
        bits.append("nonsym")
    for k in ("FT", "band"):
        if sp.get(k):
            bits.append(k)
    if sp.get("f", True) is False:
        bits.append("nof")
    if sp.get("grads", "both") != "both":
        bits.append(sp["grads"])
    if sp.get("off"):
        bits.append("off%d" % sp["off"])
    return "-".join(bits)


def K(T, B, n, m, dt, **kw):
    return dict(op="mpcb", T=T, B=B, n=n, m=m, dt=dt, seed=kw.pop("seed", T * 1013 + B * 11 + n * 5 + m * 3 + (dt == F32)), **kw)


def LA(T, B, n, m, dt, **kw):
    return dict(op="la", T=T, B=B, n=n, m=m, dt=dt, seed=kw.pop("seed", T * 917 + B * 13 + n * 7 + m), **kw)


NS = dict(sym=False)
DEFAULT = [
    # thread-per-element shapes (masked lqr_tpe_kernel, adjoint_out_tpe_kernel; reduced: adjoint_out_kernel<R, n, m, G, true>)
    K(9, 45, 2, 1, F64, FT=True, **NS), K(9, 45, 2, 1, F32, grads="x_only", **NS), K(1, 33, 2, 1, F64, **NS),
    K(2, 70, 2, 1, F32, f=False),
    K(20, 8229, 3, 1, F64, grads="u_only"),                      # BASELINE config 4: the imitation-learning gradient
    K(8, 67, 3, 1, F64, band=True, FT=True, **NS), K(20, 200, 3, 1, F32, grads="u_only", **NS),
    K(6, 33, 3, 1, F64, f=False, grads="x_only", off=1, **NS), K(1, 48, 3, 1, F32, **NS),
    K(5, 4101, 4, 2, F64, off=1, FT=True, **NS), K(2, 40, 4, 2, F32, grads="u_only", **NS),
    K(12, 100, 4, 2, F32, FT=True, f=False, **NS), K(7, 37, 4, 2, F64, f=False),
    # specialised group shapes; (32,8) reduced is adjoint_out_kernel<R, 32, 8, 128, true> with ADJ_NEGATE
    K(6, 21, 8, 4, F64, FT=True, **NS), K(6, 21, 8, 4, F32, grads="u_only", **NS), K(2, 9, 8, 4, F64, f=False, grads="x_only", off=1),
    K(6, 5, 32, 8, F64, **NS), K(4, 30, 32, 8, F32, FT=True, grads="u_only", **NS), K(1, 7, 32, 8, F64, off=1),
    K(3, 30, 32, 8, F64, f=False, grads="u_only", off=1, **NS),
    # runtime shapes: G = 8 (3,2) (2,4); 16 (6,5); 32 (12,6) (2,22, m > n); 256 / 128 (8,24)
    K(8, 50, 3, 2, F64, band=True, **NS), K(9, 37, 3, 2, F32, FT=True, grads="u_only", **NS), K(1, 20, 3, 2, F64, f=False),
    K(7, 29, 2, 4, F64, f=False, **NS), K(7, 29, 2, 4, F32, grads="x_only"), K(2, 29, 2, 4, F64, grads="u_only", FT=True, **NS),
    K(6, 17, 6, 5, F64, FT=True, grads="u_only", **NS), K(6, 17, 6, 5, F32, **NS), K(3, 17, 6, 5, F64, f=False, off=1),
    K(5, 9, 12, 6, F64, f=False, **NS), K(5, 30, 12, 6, F32, FT=True, off=1), K(2, 9, 12, 6, F64, grads="u_only", **NS),
    K(3, 5, 2, 22, F64, grads="u_only", FT=True, **NS), K(3, 30, 2, 22, F32, **NS), K(2, 5, 2, 22, F64, f=False, off=1),
    K(4, 3, 8, 24, F64, grads="x_only", **NS), K(4, 30, 8, 24, F32, f=False, off=1, **NS), K(2, 3, 8, 24, F64, grads="u_only", FT=True),
]

LA_CASES = [
    LA(9, 45, 2, 1, F32), LA(12, 70, 3, 1, F32, f=False, sym=False), LA(7, 37, 4, 2, F32, sym=False),
    LA(7, 37, 4, 2, F64, f=False, sym=False, off=1), LA(6, 21, 8, 4, F32, f=False), LA(4, 5, 32, 8, F32, sym=False),
    LA(9, 23, 3, 2, F32, sym=False), LA(6, 17, 6, 5, F32, f=False), LA(5, 9, 12, 6, F32, sym=False),
    LA(4, 3, 8, 24, F32, f=False, sym=False),
]

# the settings' cases (their tpe switches are read once per process)
CHILD = {
    "lqr_group": (dict(DMPC_LQR_GROUP="1"),
                  [K(9, 45, 2, 1, F64, FT=True, **NS), K(9, 45, 2, 1, F32, grads="u_only", **NS),
                   K(8, 37, 3, 1, F64, grads="u_only", **NS), K(8, 37, 3, 1, F32, f=False, **NS),
                   K(7, 37, 4, 2, F64, f=False, off=1, **NS), K(7, 37, 4, 2, F32, FT=True, grads="x_only", **NS)]),
    "adj_group": (dict(DMPC_ADJ_GROUP="1"),
                  [K(9, 45, 2, 1, F64, grads="u_only", **NS), K(9, 45, 2, 1, F32, FT=True, **NS),
                   K(8, 37, 3, 1, F64, FT=True, f=False, **NS), K(8, 37, 3, 1, F32, grads="u_only", **NS),
                   K(7, 37, 4, 2, F64, off=1, **NS), K(7, 37, 4, 2, F32, f=False, grads="u_only", **NS)]),
}
# elements per warp of the tpe kernels: 8 up to B = 4736, 16 up to 9472; 64-thread CTAs from B = 18944
for _s, _v in (("epw8", "8"), ("epw16", "16"), ("epw_auto", "auto")):
    CHILD[_s] = (dict(DMPC_LQR_TPE_EPW=_v),
                 [K(3, 4736, 4, 2, F64, **NS), K(3, 4737, 3, 1, F64, grads="u_only", **NS),
                  K(2, 9473, 4, 2, F64, FT=True), K(2, 19000, 3, 1, F64, grads="u_only", **NS),
                  K(2, 18944, 2, 1, F64, f=False, **NS), K(20, 150, 2, 1, F32, **NS)])


# ------------------------------------------------------------------------------------------------ tests
# The default-path cases run in a child process of their own as well: in a process that has already run the rest of the
# GPU suite, torch.profiler was seen to return traces with some or all of the library's kernels missing.
SETTINGS = dict(CHILD, default=({}, DEFAULT + LA_CASES))
_CHILD_RESULTS = {}


def _child_results(setting):
    """Runs the cases of one setting in a child process (once per test session) and loads its outputs."""
    if setting not in _CHILD_RESULTS:
        env = {k: v for k, v in os.environ.items() if not k.startswith("DMPC_")}
        env.update(SETTINGS[setting][0])
        with tempfile.TemporaryDirectory() as td:
            path = os.path.join(td, "out.npz")
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", setting, path], env=env,
                               capture_output=True, text=True, timeout=600)
            assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-4000:])
            with np.load(path, allow_pickle=False) as z:
                _CHILD_RESULTS[setting] = {k: z[k] for k in z.files}
    return _CHILD_RESULTS[setting]


def _outputs(setting, sp):
    res = _child_results(setting)
    cid = case_id(sp) + "/"
    out = {k[len(cid):]: v for k, v in res.items() if k.startswith(cid)}
    return out, list(out.pop("__kernels_full__")), list(out.pop("__kernels_red__"))


@pytest.mark.gpu
@pytest.mark.parametrize("sp", DEFAULT, ids=case_id)
def test_mpc_backward(sp):
    check_mpcb(sp, *_outputs("default", sp))


@pytest.mark.gpu
@pytest.mark.parametrize("sp", LA_CASES, ids=case_id)
def test_lqr_active_solve(sp):
    out, names, _ = _outputs("default", sp)
    check_la(sp, out, names)


@pytest.mark.gpu
@pytest.mark.parametrize("setting,sp", [(s, sp) for s, (_, cases) in CHILD.items() for sp in cases],
                         ids=[s + ":" + case_id(sp) for s, (_, cases) in CHILD.items() for sp in cases])
def test_ab_switch(setting, sp):
    check_mpcb(sp, *_outputs(setting, sp), setting)


def test_case_table():
    """Without a device: every case is what it claims to be, and every oracle expectation (with its sum-bound self-checks)
    is computed and memoised for the GPU tests."""
    seen = set()
    for setting, sp in [(None, sp) for sp in DEFAULT] + [(s, sp) for s, (_, cs) in CHILD.items() for sp in cs]:
        cid = case_id(sp)
        assert (setting, cid) not in seen, cid
        seen.add((setting, cid))
        T, B, n, m = sp["T"], sp["B"], sp["n"], sp["m"]
        pr = mpcb_problem(sp)
        w = mpcb_expect(sp)
        act = w["active"]
        assert np.array_equal(act, mask_of(pr))
        if sp.get("sym", True) is False:
            asym = np.abs(pr["C"] - np.swapaxes(pr["C"], 2, 3)).max(axis=(2, 3))
            assert (asym > 1e-4).all() and np.median(asym) > 1e-2, cid
        else:
            assert np.array_equal(pr["C"], np.swapaxes(pr["C"], 2, 3)), cid
        assert pr["F"].shape[0] == (T if (sp.get("FT") or T == 1) else T - 1)
        # every control of an element active at one step, none at another
        assert act[pr["allr"]].all() and pr["allr"].any(), cid
        assert not act[pr["noner"]].any() and pr["noner"].any(), cid
        rest = ~(pr["band"] | pr["ext"])
        frac = act[rest].mean()
        assert 0.1 < frac < 0.9, (cid, frac)
        if sp.get("band"):
            assert sp["dt"] == F64
            d = np.abs(pr["u"] - pr["lo"])[pr["band"]]
            assert (d == 1e-8).any() and (d == 1e-8 * (1 + 2.0 ** -40)).any() and (d == 2e-8).any(), cid
            assert (pr["lo"] == pr["hi"])[pr["band"]].any(), cid
            bu, blo, bhi = (pr[k][pr["band"]] for k in ("u", "lo", "hi"))
            for u_, lo_, hi_, a_ in BAND:
                hit = (bu == u_) & (blo == lo_) & (bhi == hi_)
                assert hit.any() and (act[pr["band"]][hit] == a_).all(), (cid, u_, lo_, hi_)
        if sp["dt"] == F32:
            assert T * B <= 4000, cid
    for sp in LA_CASES:
        pr = la_problem(sp)
        assert pr["active"][pr["allr"]].all() and not pr["active"][pr["noner"]].any()
        ox, ou = la_expect(sp)
        assert (ou[pr["active"]] == 0).all()
        if sp.get("sym", True) is False:
            assert (np.abs(pr["C"] - np.swapaxes(pr["C"], 2, 3)).max(axis=(2, 3)) > 1e-2).all()


def test_kernel_coverage():
    """Without a device: the cases, together, expect every kernel of the backward, in fp64 and fp32 - the runtime-shape
    reductions (G = 32, 128), the (32,8) reduction, the masked thread-per-element solve - and every key on every shape."""
    expect = set()
    by_shape = {}
    for setting, sp in [(None, sp) for sp in DEFAULT] + [(s, sp) for s, (_, cs) in CHILD.items() for sp in cs]:
        full, red, _ = mpcb_kernels(sp, setting)
        expect |= set(full) | set(red)
        keys = by_shape.setdefault((sp["n"], sp["m"]), set())
        keys |= {sp["dt"]} | {k for k in ("FT", "band", "off") if sp.get(k)}
        keys |= {"nonsym"} if sp.get("sym", True) is False else set()
        keys |= {"nof"} if sp.get("f", True) is False else set()
        keys |= {sp.get("grads", "both"), "T%d" % min(sp["T"], 3)}
    for sp in LA_CASES:
        expect.add("la:" + mpcb_kernels(sp)[0][1])
    for R in ("double", "float"):
        need = ["active_mask_kernel<%s>" % R, "reduce_partials_kernel<%s>" % R,
                "adjoint_out_kernel<%s, 0, 0, 8, true>" % R, "adjoint_out_kernel<%s, 0, 0, 16, true>" % R,
                "adjoint_out_kernel<%s, 0, 0, 32, true>" % R, "adjoint_out_kernel<%s, 0, 0, 128, true>" % R,
                "adjoint_out_kernel<%s, 8, 4, 16, true>" % R, "adjoint_out_kernel<%s, 32, 8, 128, true>" % R,
                "adjoint_out_kernel<%s, 32, 8, 128, false>" % R, "adjoint_out_kernel<%s, 0, 0, 128, false>" % R,
                "lqr_solve_kernel<%s, 8, 4, 16>" % R, "lqr_solve_kernel<%s, 32, 8, 256>" % R]
        need += ["lqr_solve_kernel<%s, 0, 0, %d>" % (R, G) for G in (8, 16, 32, 256)]
        for (n, m), G in ((2, 1), 4), ((3, 1), 4), ((4, 2), 8):
            need += ["lqr_tpe_kernel<%s, %d, %d," % (R, n, m), "adjoint_out_tpe_kernel<%s, %d, %d," % (R, n, m),
                     "adjoint_out_kernel<%s, %d, %d, %d, true>" % (R, n, m, G),
                     "adjoint_out_kernel<%s, %d, %d, %d, false>" % (R, n, m, G), "lqr_solve_kernel<%s, %d, %d, %d>" % (R, n, m, G)]
        missing = [k for k in need if k not in expect]
        assert not missing, missing
    # dmpc_lqr_active_solve in fp32 on the thread-per-element, specialised group and runtime-shape kernels
    for k in ("lqr_tpe_kernel<float, 2, 1,", "lqr_tpe_kernel<float, 3, 1,", "lqr_tpe_kernel<float, 4, 2,",
              "lqr_solve_kernel<float, 8, 4, 16>", "lqr_solve_kernel<float, 32, 8, 256>", "lqr_solve_kernel<float, 0, 0, 8>",
              "lqr_solve_kernel<float, 0, 0, 16>", "lqr_solve_kernel<float, 0, 0, 32>", "lqr_solve_kernel<float, 0, 0, 256>"):
        assert "la:" + k in expect, k
    for shape, keys in by_shape.items():
        for k in ("f64", "f32", "nonsym", "FT", "nof", "u_only"):
            assert k in keys, (shape, k)
    assert {"T1", "T2"} <= set().union(*by_shape.values())
    assert {"band"} <= by_shape[(3, 1)] and {"band"} <= by_shape[(3, 2)]


def _child_main(setting, path):
    ctx = _native.default_context(0)
    save = {}
    for sp in SETTINGS[setting][1]:
        if sp["op"] == "la":
            (out, nf), nr = run_la(ctx, sp), []
        else:
            out, nf, nr = run_mpcb(ctx, sp)
        cid = case_id(sp) + "/"
        for k, v in out.items():
            save[cid + k] = v
        save[cid + "__kernels_full__"] = np.array(nf if nf else [""], dtype=str)
        save[cid + "__kernels_red__"] = np.array(nr if nr else [""], dtype=str)
    np.savez(path, **save)
    ctx.close()


if __name__ == "__main__":
    assert sys.argv[1] == "--child", sys.argv
    _child_main(sys.argv[2], sys.argv[3])
