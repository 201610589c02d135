"""GPU: the box-constrained MPC step, its backward, LQR_active, get_traj and BoxDDP at shapes too large for one CTA's
shared memory (mpc_large_kernels.cuh, lqr_large_kernels.cuh, DESIGN.md §4.9).

Every case runs through the C ABI (or the facades) and compares with the reference recursions (oracle/mpc.py,
oracle/boxddp.py): rel_err 1e-10 in fp64, the suite's 1e-4 (trajectories, gains) / 1e-3 (gradients) in fp32 on
fp32-rounded inputs.  Outputs start as NaN, so an entry the kernels skip fails.  The bounds clamp a share of the controls
that the oracle asserts (at least 20 %), and every line-search decision clears a margin of 1e3 ulp of the old cost in
fp64 (the oracle asserts it).  fp32 integer decisions (n_ls, alpha, flags) are asserted only where the oracle's margin
is above 1e-3 of the old cost, well past fp32 rounding.  Which kernels ran is read from a torch.profiler trace taken in a
child process; the boundaries of the selection come from the layout functions' sizes, computed here.
"""
import os
import subprocess
import sys
import tempfile
import zlib

import numpy as np
import pytest

if __name__ == "__main__":                   # the child process of test_kernels_reached: the paths conftest.py would set
    _root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    _pkg = os.path.join(_root, "chainer-differentiable-mpc_b200")
    sys.path[:0] = [os.path.dirname(os.path.abspath(__file__)), _root, _pkg, os.path.join(_pkg, "lqr"),
                    os.path.join(_pkg, "mpc")]

from _helpers import rel_err  # noqa: E402
from oracle import mpc as ompc  # noqa: E402
from oracle import boxddp as obox  # noqa: E402
from test_gpu_lqr_large import Bufs, assert_sum  # noqa: E402

pytestmark = pytest.mark.gpu

F64, F32 = "f64", "f32"
NP = {F64: np.float64, F32: np.float32}
FLAG_QP, FLAG_LS_CAPPED = 1, 4
K_MAX_SMEM = 227 * 1024


def tol(dt, grad=False):
    return 1e-10 if dt == F64 else (1e-3 if grad else 1e-4)


def sum_tol(dt):
    return 1e-10 if dt == F64 else 2e-5


# ------------------------------------------------------------------------------------------------ layout sizes
# host restatements of mpc_layout, lqr_layout (no SAVE_FAC) and adj_layout (csrc/mpc_kernels.cuh, lqr_kernels.cuh):
# the per-element kernels run a shape exactly when these fit (kMpcMaxSmem = kMaxSmem - 256 for the MPC forward)
def _rup(a, w):
    return (a + w - 1) // w * w


def mpc_bytes(n, m, w):
    W, s = 16 // w, n + m
    st = sum(_rup(a, W) for a in (s * s, s, n * s, n, n, m, m, m, m * n, m))
    o = 2 * st + sum(_rup(a, W) for a in (s * s, s, n * n, n, n * s, n, m * m, m * (n + 1), m * (n + 1), s, m, m, m, m,
                                           m, m, s, n, n, (m * 4 + w - 1) // w))
    return (_rup(o, 128 // w) + W) * w


def lqr_bytes(n, m, w):
    W, s = 16 // w, n + m
    st = sum(_rup(a, W) for a in (s * s, s, n * s, n))
    o = 2 * st + sum(_rup(a, W) for a in (s * s, s, n * n, n, n * s, m * m, m * (n + 1), m * (n + 1), n, s,
                                           (m * 4 + w - 1) // w))
    return (_rup(o, 128 // w) + W) * w


def adj_bytes(n, m, w, red):
    W, s = 16 // w, n + m
    st = _rup(n * s, W) + _rup(s, W) + _rup(n * s, W) + _rup(n, W) + _rup(m, W) + _rup(s, W) + _rup(n, W)
    o = 2 * st + 4 * _rup(n, W) + (_rup(s * s + s + n * s + n, W) if red else 0)
    return (_rup(o, 128 // w) + W) * w


def fwd_large(n, m, w=8):
    return n + m > 24 and mpc_bytes(n, m, w) > K_MAX_SMEM - 256


def solve_large(n, m, w=8):
    return lqr_bytes(n, m, w) > K_MAX_SMEM


def adj_large(n, m, red, w=8):
    return adj_bytes(n, m, w, red) > K_MAX_SMEM


def test_layout_restatement_matches_the_issue_table():
    """The host restatement reproduces the largest per-element shapes (fp64 forward: (56, 8); masked solve: (57, 8))."""
    assert not fwd_large(56, 8) and fwd_large(57, 8)
    assert not solve_large(57, 8) and solve_large(58, 8)
    assert not adj_large(63, 8, True) and adj_large(64, 8, True) and not adj_large(64, 8, False)


# ------------------------------------------------------------------------------------------------ problems
def problem(seed, T, B, n, m, F_T=None, pivot=False, with_f=True, dt=F64, clamp=0.25):
    """Non-symmetric C_t, F_t varying with t and b; nominal trajectory = rollout of u_nom; symmetric bounds at the
    (1 - clamp) quantile of |u| of an unconstrained step, so that about `clamp` of the controls end on a bound.  pivot: the
    control block of C is made of 2 x 2 blocks [[0.2, 0.6], [-0.5, 0.3]] (positive definite symmetric part, so PNQP stays
    well posed) and F_u is small, so Quu stays close to C_uu and the pivoted elimination swaps rows."""
    rs = np.random.RandomState(seed)
    s = n + m
    F_T = T - 1 if F_T is None else F_T
    L = 0.85 / np.sqrt(s) * rs.randn(T, B, s, s)
    C = L @ np.swapaxes(L, 2, 3) + np.eye(s) + 0.002 * rs.randn(T, B, s, s)
    F = np.concatenate((0.9 * np.eye(n) + 0.1 / np.sqrt(n) * rs.randn(F_T, B, n, n), 0.3 * rs.randn(F_T, B, n, m)), axis=3)
    if pivot:
        base = np.eye(m)
        for i in range(0, m - 1, 2):
            base[i:i + 2, i:i + 2] = [[0.2, 0.6], [-0.5, 0.3]]
        C[:, :, n:, n:] = base + 0.1 * (C[:, :, n:, n:] - np.eye(m))
        F[:, :, :, n:] *= 0.01
    c = rs.randn(T, B, s)
    f = 0.1 * rs.randn(T - 1, B, n) if with_f else None
    x0 = rs.randn(B, n)
    u_nom = 0.1 * rs.randn(T, B, m)
    pr = dict(T=T, B=B, n=n, m=m, F_T=F_T, C=C, c=c, F=F, f=f, x0=x0, u_nom=u_nom)
    if dt == F32:
        pr = {k: (v.astype(np.float32).astype(np.float64) if isinstance(v, np.ndarray) else v) for k, v in pr.items()}
    pr["x_nom"] = ompc.get_traj(pr["x0"], pr["u_nom"], ("linear", pr["F"], pr["f"]))
    if dt == F32:
        pr["x_nom"] = pr["x_nom"].astype(np.float32).astype(np.float64)
    big = np.full((T, B, m), 1e6)
    _, u, _, _ = ompc.step_forward(pr["C"], pr["c"], pr["F"], None, pr["x_nom"], pr["u_nom"], -big, big,
                                   (pr["C"], pr["c"]), ("linear", pr["F"], pr["f"]), 0.2, 64, n, m, True,
                                   coupling="element")
    b = float(np.quantile(np.abs(u), 1.0 - clamp))
    lo, hi = np.full((T, B, m), -b), np.full((T, B, m), b)
    if dt == F32:
        lo, hi = lo.astype(np.float32).astype(np.float64), hi.astype(np.float32).astype(np.float64)
    pr.update(lo=lo, hi=hi, tC=pr["C"], tc=pr["c"], tF=pr["F"], tf=pr["f"])
    return pr


def fwd_oracle(pr, need_expand=True, decay=0.2, max_ls=64):
    T, B, n, m = pr["T"], pr["B"], pr["n"], pr["m"]
    f = None if need_expand else pr["f"]
    x, u, fo, aux = ompc.step_forward(pr["C"], pr["c"], pr["F"], f, pr["x_nom"], pr["u_nom"], pr["lo"], pr["hi"],
                                      (pr["tC"], pr["tc"]), ("linear", pr["tF"], pr["tf"]), decay, max_ls, n, m,
                                      need_expand, coupling="element", max_trials=max_ls)
    old = ompc.traj_cost(pr["x_nom"], pr["u_nom"], (pr["tC"], pr["tc"]))
    # the cost of every pass each element ran, against the old cost: the decisions' margins
    margins = np.full(B, np.inf)
    for b in range(B):
        sl = slice(b, b + 1)
        for k in range(int(fo.n_ls[b])):
            al = np.array([decay ** k])
            _, _, _, cst = ompc.ls_pass(aux["Ks"][:, sl], aux["ks"][:, sl], pr["x_nom"][:, sl], pr["u_nom"][:, sl],
                                        pr["lo"][:, sl], pr["hi"][:, sl], (pr["tC"][:, sl], pr["tc"][:, sl]),
                                        ("linear", pr["tF"][:, sl], None if pr["tf"] is None else pr["tf"][:, sl]), al)
            margins[b] = min(margins[b], abs(cst[0] - old[b]) / abs(old[b]))
    capped = (fo.n_ls >= max_ls) & (fo.costs > old)
    at_bound = np.mean((np.abs(u - pr["lo"]) < 1e-12) | (np.abs(u - pr["hi"]) < 1e-12))
    return dict(x=x, u=u, Ks=aux["Ks"], ks=aux["ks"], n_qp=aux["n_qp"], free=aux["free"], objs=fo.objs,
                u_first=fo.u_first, costs=fo.costs, old=old, alphas=fo.alphas, n_ls=fo.n_ls, capped=capped,
                margins=margins, at_bound=at_bound)


def run_forward(ctx, pr, dt, need_expand=True, decay=0.2, max_ls=64, off=0, coupling=0, sweep_only=False):
    import _native
    T, B, n, m = pr["T"], pr["B"], pr["n"], pr["m"]
    R = NP[dt]
    bf = Bufs(off)
    put = lambda k: None if pr[k] is None else bf.put(pr[k], R)
    C, c, F, xn, un, lo, hi = (put(k) for k in ("C", "c", "F", "x_nom", "u_nom", "lo", "hi"))
    f = None if need_expand else put("f")
    tC = C if pr["tC"] is pr["C"] else put("tC")
    tc = c if pr["tc"] is pr["c"] else put("tc")
    tF = F if pr["tF"] is pr["F"] else put("tF")
    tf = put("tf")
    o = {k: bf.empty(v, d) for k, (v, d) in dict(
        x=((T, B, n), R), u=((T, B, m), R), Ks=((T, B, m, n), R), ks=((T, B, m), R), u_first=((T, B, m), R),
        objs=((T, B), R), costs=((B,), R), old=((B,), R), alphas=((B,), R)).items()}
    import torch
    ints = {}
    for k, v, d in (("n_qp", (T, B), torch.int32), ("n_ls", (B,), torch.int32), ("flags", (B,), torch.int32),
                    ("free", (T, B, m), torch.uint8)):
        t = torch.full((int(np.prod(v)) + off,), -1 if d == torch.int32 else 255, dtype=d, device="cuda")
        bf.keep.append(t)
        ints[k] = (t, v)
    P = {k: bf.ptr(v) for k, v in list(o.items()) + list(ints.items())}
    ctx.mpc_step_forward(R, T, B, n, m, C, c, F, pr["F_T"], f, xn, un, lo, hi, tC, tc, _native.DYN_LINEAR, tF, tf,
                         None, decay, -1 if sweep_only else max_ls, need_expand, coupling, P["x"], P["u"], P["Ks"],
                         P["ks"], P["u_first"], P["objs"], P["costs"], P["old"], P["alphas"], P["n_qp"], P["free"],
                         P["n_ls"], P["flags"])
    ctx.sync()
    out = {k: bf.get(v) for k, v in o.items()}
    out.update({k: v[0][off:].cpu().numpy().reshape(v[1]) for k, v in ints.items()})
    return out


def check_forward(pr, dt, out, o, decay=0.2):
    assert o["at_bound"] >= 0.2, o["at_bound"]                         # the bounds do clamp
    exact = dt == F64 or np.all(o["margins"] > 1e-3)
    if dt == F64:
        old = np.abs(o["old"])
        assert np.all(o["margins"] * old > 1e3 * np.spacing(old)), o["margins"]
    assert np.array_equal(out["n_qp"], o["n_qp"])
    assert np.array_equal(out["free"].astype(float), o["free"])
    if exact:
        assert np.array_equal(out["n_ls"], o["n_ls"]), (out["n_ls"], o["n_ls"])
        # alpha of the pass written: decay^(n_ls - 1), by repeated products as the kernel forms it (the oracle multiplies
        # once more after a capped element's last pass)
        alpha = np.ones(pr["B"])
        for b in range(pr["B"]):
            for _ in range(int(o["n_ls"][b]) - 1):
                alpha[b] *= decay
        assert np.array_equal(out["alphas"], alpha.astype(NP[dt]))
        assert np.array_equal((out["flags"] & FLAG_LS_CAPPED) != 0, o["capped"])
    # PNQP hit its iteration cap at some step (n_qp = 20 is 1 + the last iteration index)
    assert np.array_equal((out["flags"] & FLAG_QP) != 0, np.any(o["n_qp"] == 20, axis=0))
    assert np.all((out["flags"] & ~(FLAG_LS_CAPPED | FLAG_QP)) == 0), out["flags"]
    for k in ("x", "u", "Ks", "ks", "u_first", "objs"):
        assert rel_err(out[k], o[k]) < tol(dt), k
    for k, ok in (("costs", "costs"), ("old", "old")):
        assert rel_err(out[k], o[ok]) < tol(dt), k


@pytest.fixture(scope="module")
def ctx():
    import _native
    return _native.default_context(0)


FWD = [
    dict(dt=F64, n=64, m=16, T=5, B=4, expand=True, extra=0, pivot=False, off=0),
    dict(dt=F64, n=80, m=8, T=2, B=4, expand=False, extra=1, pivot=True, off=1),
    dict(dt=F64, n=128, m=32, T=2, B=3, expand=True, extra=1, pivot=False, off=0),
    dict(dt=F64, n=60, m=32, T=5, B=3, expand=True, extra=0, pivot=False, off=1),
    dict(dt=F64, n=57, m=8, T=1, B=3, expand=True, extra=0, pivot=False, off=0),
    dict(dt=F32, n=80, m=16, T=5, B=4, expand=True, extra=0, pivot=False, off=0),
    dict(dt=F32, n=128, m=32, T=2, B=3, expand=False, extra=0, pivot=False, off=1),
]


def fid(c):
    return "%s-n%d-m%d-T%d-B%d-e%d-x%d-p%d-o%d" % (c["dt"], c["n"], c["m"], c["T"], c["B"], c["expand"], c["extra"],
                                                  c["pivot"], c["off"])


def fwd_problem(c):
    return problem(zlib.crc32(fid(c).encode()) % 1000, c["T"], c["B"], c["n"], c["m"], c["T"] - 1 + c["extra"] if c["T"] > 1 else 0,
                   c["pivot"], True, c["dt"], clamp=0.45 if c["pivot"] else 0.25)


@pytest.mark.parametrize("c", FWD, ids=fid)
def test_forward_against_oracle(ctx, c):
    assert fwd_large(c["n"], c["m"], 8 if c["dt"] == F64 else 4)
    pr = fwd_problem(c)
    o = fwd_oracle(pr, c["expand"])
    out = run_forward(ctx, pr, c["dt"], c["expand"], off=c["off"])
    check_forward(pr, c["dt"], out, o)
    if c["dt"] == F64 and c["off"] == 0:                 # a repeated call returns the same bits
        again = run_forward(ctx, pr, c["dt"], c["expand"], off=c["off"])
        for k, v in again.items():
            assert np.array_equal(v, out[k], equal_nan=True), k


def true_model_problem(seed, dt=F64):
    """A true cost and true dynamics in their own buffers that make the line search backtrack."""
    T, B, n, m = 5, 6, 64, 16
    pr = problem(seed, T, B, n, m, dt=dt)
    rs = np.random.RandomState(seed + 1)
    s = n + m
    scale = np.linspace(0.0, 1.5, B)[None, :, None, None]
    Lt = rs.randn(T, B, s, s) / np.sqrt(s)
    tC = pr["C"] + scale * (Lt @ np.swapaxes(Lt, 2, 3))
    tF = pr["F"] + 0.3 * scale[:, :, :, :1] * rs.randn(*pr["F"].shape) / np.sqrt(s)
    tc = pr["c"] + 0.5 * rs.randn(T, B, s)
    if dt == F32:
        tC, tF, tc = (a.astype(np.float32).astype(np.float64) for a in (tC, tF, tc))
    pr.update(tC=tC, tc=tc, tF=tF, tf=pr["f"])
    return pr


def test_true_model_line_search_and_cap(ctx):
    """True cost / dynamics that differ from the model: the line search backtracks (n_ls > 1 somewhere, the oracle shows
    it); with max_ls_trials = 2, FLAG_LS_CAPPED is set on exactly the elements whose second pass is still worse."""
    pr = true_model_problem(21)
    o = fwd_oracle(pr)
    assert np.any(o["n_ls"] > 1) and np.any(o["n_ls"] == 1)
    check_forward(pr, F64, run_forward(ctx, pr, F64), o)
    o2 = fwd_oracle(pr, max_ls=2)
    assert 1 <= int(np.sum(o2["capped"])) < pr["B"], o2["capped"]
    check_forward(pr, F64, run_forward(ctx, pr, F64, max_ls=2), o2)
    o3 = fwd_oracle(pr, decay=0.7)
    check_forward(pr, F64, run_forward(ctx, pr, F64, decay=0.7), o3, decay=0.7)


def test_sweep_only_gains_equal_full_call(ctx):
    """max_ls_trials < 0: the gains, n_qp, free and flags of the full call, bit for bit; nothing else is written."""
    pr = fwd_problem(FWD[0])
    full = run_forward(ctx, pr, F64)
    sw = run_forward(ctx, pr, F64, sweep_only=True)
    for k in ("Ks", "ks", "n_qp", "free", "flags"):
        assert np.array_equal(sw[k], full[k]), k
    assert np.all(np.isnan(sw["x"])) and np.all(np.isnan(sw["costs"]))


def test_batch_coupling_unsupported(ctx):
    import _native
    pr = fwd_problem(FWD[0])
    before = ctx.launches
    with pytest.raises(_native.DiffMpcError, match="batch coupling"):
        run_forward(ctx, pr, F64, coupling=_native.COUPLING_BATCH)
    assert ctx.launches == before


# ------------------------------------------------------------------------------------------------ backward
def bwd_problem(seed, T, B, n, m, dt, F_T=None, with_f=True, pinned=True):
    """x, u, bounds, upstream gradients.  pinned: controls at exactly 0, 1e-8 and 2e-8 from a bound (fp64 only: the active
    test |u - bound| <= 1e-8 runs in the tensor's dtype)."""
    rs = np.random.RandomState(seed)
    s = n + m
    F_T = T - 1 if F_T is None else F_T
    base = problem(seed, T, B, n, m, F_T=F_T, with_f=with_f, dt=dt)
    x = rs.randn(T, B, n)
    u = rs.uniform(-1, 1, (T, B, m))
    lo, hi = np.full((T, B, m), -1.0), np.full((T, B, m), 1.0)
    band = rs.rand(T, B, m)
    if pinned and dt == F64:
        d = np.choose((band * 6).astype(int), [0.0, 1e-8, 2e-8, 0.0, 0.3, 0.6])
    else:
        d = np.choose((band * 4).astype(int), [0.0, 2e-3, 0.3, 0.6])
    side = rs.rand(T, B, m) < 0.5
    u = np.where(side, lo + d, hi - d)
    gx, gu = rs.randn(T, B, n), rs.randn(T, B, m)
    pr = dict(T=T, B=B, n=n, m=m, F_T=F_T, C=base["C"], c=base["c"], F=base["F"], f=base["f"], x=x, u=u, lo=lo, hi=hi,
              gx=gx, gu=gu)
    if dt == F32:
        pr = {k: (v.astype(np.float32).astype(np.float64) if isinstance(v, np.ndarray) else v) for k, v in pr.items()}
    return pr


def bwd_oracle(pr, gx_null=False, gu_null=False):
    T, B, n, m = pr["T"], pr["B"], pr["n"], pr["m"]
    gx = None if gx_null else pr["gx"]
    gu = None if gu_null else pr["gu"]
    dx0, dC, dc, dF, df = ompc.step_backward(pr["C"], pr["c"], pr["F"], pr["f"], pr["x"], pr["u"], pr["lo"], pr["hi"],
                                             gx, gu, n, m)
    # sum |term| bounds of the reduced sums
    xu = np.concatenate((pr["x"], pr["u"]), 2)
    dxu = -dc
    gxa = np.zeros((T, B, n)) if gx is None else gx
    lam, dlam = np.zeros((T, B, n)), np.zeros((T, B, n))
    for t in range(T - 1, -1, -1):
        lam[t] = np.einsum("bij,bj->bi", pr["C"][t][:, :n], xu[t]) + pr["c"][t][:, :n]
        dlam[t] = np.einsum("bij,bj->bi", pr["C"][t][:, :n], dxu[t]) - gxa[t]
        if t < T - 1:
            lam[t] += np.einsum("bji,bj->bi", pr["F"][t][:, :, :n], lam[t + 1])
            dlam[t] += np.einsum("bji,bj->bi", pr["F"][t][:, :, :n], dlam[t + 1])
    a = np.einsum("tbi,tbj->tbij", np.abs(dxu), np.abs(xu))
    bC = 0.5 * (a + np.swapaxes(a, 2, 3))
    bF = (np.einsum("tbi,tbj->tbij", np.abs(dlam[1:]), np.abs(xu[:-1])) +
          np.einsum("tbi,tbj->tbij", np.abs(lam[1:]), np.abs(dxu[:-1])))
    active = (np.abs(pr["u"] - pr["lo"]) <= 1e-8) | (np.abs(pr["u"] - pr["hi"]) <= 1e-8)
    # the reduced df is sum_t -d-lambda_{t+1} whether or not f is given
    return dict(dx0=dx0, dC=dC, dc=dc, dF=dF, df=df, bC=bC, bF=bF, bf=np.abs(dlam[1:]), df_sum=-dlam[1:].sum((0, 1)),
                active=active)


def run_backward(ctx, pr, dt, gx_null=False, gu_null=False, df_null=False, off=0):
    T, B, n, m, F_T = pr["T"], pr["B"], pr["n"], pr["m"], pr["F_T"]
    s, R = n + m, NP[dt]
    bf = Bufs(off)
    C, c, F, x, u, lo, hi = (bf.put(pr[k], R) for k in ("C", "c", "F", "x", "u", "lo", "hi"))
    gx = None if gx_null else bf.put(pr["gx"], R)
    gu = None if gu_null else bf.put(pr["gu"], R)
    rsz = ctx.reduced_grad_elems(n, m)
    o = {k: bf.empty(v, R) for k, v in dict(wK=(T, B, m, n), wk=(T, B, m), wd=(T, B, s), dx0=(B, n), dC=(T, B, s, s),
                                             dc=(T, B, s), dF=(F_T, B, n, s), df=(T - 1, B, n), rdx0=(B, n),
                                             part=(B, rsz), sums=(rsz,)).items()}
    import torch
    act = torch.full((T * B * m + off,), 7, dtype=torch.uint8, device="cuda")
    bf.keep.append(act)
    pa = act.data_ptr() + off
    P = {k: bf.ptr(v) for k, v in o.items()}
    ctx.mpc_step_backward(R, T, B, n, m, C, c, F, F_T, x, u, lo, hi, gx, gu, P["wK"], P["wk"], P["wd"], pa, P["dx0"],
                          P["dC"], P["dc"], P["dF"], None if df_null else P["df"])
    ctx.sync()
    out = {k: bf.get(o[k]) for k in ("dx0", "dC", "dc", "dF", "df")}
    out["active"] = act[off:].cpu().numpy().reshape(T, B, m)
    ctx.mpc_step_backward_reduced(R, T, B, n, m, C, c, F, F_T, x, u, lo, hi, gx, gu, P["wK"], P["wk"], P["wd"], pa,
                                  P["part"], P["rdx0"], P["sums"])
    ctx.sync()
    out["rdx0"], out["sums"] = bf.get(o["rdx0"]), bf.get(o["sums"])
    return out


def check_backward(pr, dt, out, o, df_null=False):
    T, n, m = pr["T"], pr["n"], pr["m"]
    s = n + m
    assert np.array_equal(out["active"].astype(bool), o["active"])
    for k in ("dx0", "dC", "dc"):
        assert rel_err(out[k], o[k]) < tol(dt, True), k
    assert rel_err(out["dF"][:T - 1], o["dF"][:T - 1]) < tol(dt, True)
    if pr["F_T"] == T:
        assert np.all(out["dF"][T - 1] == 0)
    if not df_null and pr["f"] is not None:
        assert rel_err(out["df"], o["df"]) < tol(dt, True)
    assert rel_err(out["rdx0"], o["dx0"]) < tol(dt, True)
    sm = out["sums"]
    sC, sc = sm[:s * s].reshape(s, s), sm[s * s:s * s + s]
    sF, sf = sm[s * s + s:s * s + s + n * s].reshape(n, s), sm[s * s + s + n * s:]
    eps = sum_tol(dt)
    assert_sum(sC, o["dC"].sum((0, 1)), o["bC"].sum((0, 1)), eps, "sum dC")
    assert_sum(sc, o["dc"].sum((0, 1)), np.abs(o["dc"]).sum((0, 1)), eps, "sum dc")
    if T > 1:
        assert_sum(sF, o["dF"][:T - 1].sum((0, 1)), o["bF"].sum((0, 1)), eps, "sum dF")
        assert_sum(sf, o["df_sum"], o["bf"].sum((0, 1)), eps, "sum df")
    # leaving out element B-1 or the last step moves a sum by more than its bound somewhere
    lim = lambda b: eps * b + 1e-300
    B = pr["B"]
    bC = o["bC"].sum((0, 1))
    assert np.max(np.abs(o["dC"][:, B - 1].sum(0)) / lim(bC)) > 1.0
    assert np.max(np.abs(o["dC"][T - 1].sum(0)) / lim(bC)) > 1.0


BWD = [
    dict(dt=F64, n=64, m=16, T=5, B=4, extra=0, f=True, gx=False, gu=False, off=0),
    dict(dt=F64, n=58, m=8, T=5, B=3, extra=1, f=True, gx=True, gu=False, off=1),
    dict(dt=F64, n=64, m=8, T=2, B=5, extra=0, f=False, gx=False, gu=True, off=0),
    dict(dt=F64, n=60, m=32, T=5, B=3, extra=1, f=True, gx=False, gu=False, off=0),
    dict(dt=F64, n=128, m=32, T=2, B=3, extra=0, f=True, gx=False, gu=False, off=1),
    dict(dt=F64, n=80, m=8, T=1, B=4, extra=0, f=False, gx=False, gu=False, off=0),
    dict(dt=F32, n=96, m=16, T=5, B=4, extra=1, f=True, gx=False, gu=False, off=0),
    dict(dt=F32, n=128, m=32, T=2, B=3, extra=0, f=False, gx=True, gu=False, off=0),
]


def bid(c):
    return "%s-n%d-m%d-T%d-B%d-x%d-f%d-gx%d-gu%d-o%d" % (c["dt"], c["n"], c["m"], c["T"], c["B"], c["extra"], c["f"],
                                                        c["gx"], c["gu"], c["off"])


def bwd_problem_of(c):
    return bwd_problem(zlib.crc32(bid(c).encode()) % 1000, c["T"], c["B"], c["n"], c["m"], c["dt"],
                       F_T=(c["T"] - 1 + c["extra"]) if c["T"] > 1 else 0, with_f=c["f"])


@pytest.mark.parametrize("c", BWD, ids=bid)
def test_backward_against_oracle(ctx, c):
    pr = bwd_problem_of(c)
    w = 8 if c["dt"] == F64 else 4
    assert solve_large(c["n"], c["m"], w) or adj_large(c["n"], c["m"], True, w)
    o = bwd_oracle(pr, c["gx"], c["gu"])
    out = run_backward(ctx, pr, c["dt"], c["gx"], c["gu"], off=c["off"])
    check_backward(pr, c["dt"], out, o)
    if c["dt"] == F64 and c["off"] == 0:
        again = run_backward(ctx, pr, c["dt"], c["gx"], c["gu"], off=c["off"])
        assert np.array_equal(again["sums"], out["sums"]) and np.array_equal(again["rdx0"], out["rdx0"])


@pytest.mark.parametrize("dt", [F64, F32])
def test_lqr_active_against_oracle(ctx, dt):
    T, B, n, m = 5, 4, 64, 16
    pr = problem(31, T, B, n, m, dt=dt)
    rs = np.random.RandomState(5)
    active = rs.rand(T, B, m) < 0.3
    x, u = ompc.lqr_active(pr["x0"], pr["C"], pr["c"], pr["F"], pr["f"], active, n, m)
    R = NP[dt]
    bf = Bufs(1)
    x0, C, c, F, f = (bf.put(pr[k], R) for k in ("x0", "C", "c", "F", "f"))
    import torch
    a = torch.zeros(T * B * m + 1, dtype=torch.uint8, device="cuda")
    a[1:].copy_(torch.from_numpy(active.astype(np.uint8).reshape(-1)))
    bf.keep.append(a)
    o = {k: bf.empty(v, R) for k, v in dict(x=(T, B, n), u=(T, B, m), Ks=(T, B, m, n), ks=(T, B, m)).items()}
    ctx.lqr_active_solve(R, T, B, n, m, x0, C, c, F, T - 1, f, a.data_ptr() + 1, *(bf.ptr(o[k]) for k in ("x", "u", "Ks", "ks")))
    ctx.sync()
    assert rel_err(bf.get(o["x"]), x) < tol(dt) and rel_err(bf.get(o["u"]), u) < tol(dt)
    assert np.all(bf.get(o["u"])[active] == 0)


# ------------------------------------------------------------------------------------------------ get_traj, BoxDDP
@pytest.mark.parametrize("dt", [F64, F32])
@pytest.mark.parametrize("nm", [(80, 16), (128, 32)])
def test_get_traj_and_line_search_agree(ctx, dt, nm):
    """dmpc_get_traj (LinDx) against the oracle, and get_traj of the accepted controls reproduces the line search's x bit
    for bit."""
    import _native
    n, m = nm
    assert fwd_large(n, m, 8 if dt == F64 else 4) and n + m > 64
    T, B = 5, 3
    pr = problem(41, T, B, n, m, dt=dt)
    R = NP[dt]
    out = run_forward(ctx, pr, dt)
    bf = Bufs()
    x0, F, f = bf.put(pr["x_nom"][0], R), bf.put(pr["F"], R), bf.put(pr["f"], R)
    u = bf.put(out["u"], R)
    x = bf.empty((T, B, n), R)
    ctx.get_traj(R, T, B, n, m, _native.DYN_LINEAR, x0, u, F, f, None, bf.ptr(x))
    ctx.sync()
    xg = bf.get(x)
    assert np.array_equal(xg, out["x"])
    xo = ompc.get_traj(pr["x_nom"][0], out["u"].astype(np.float64), ("linear", pr["F"], pr["f"]))
    assert rel_err(xg, xo) < tol(dt)


def test_boxddp_facade_device_and_host_loop(ctx):
    from box_ddp import BoxDDP
    from util import QuadCost, LinDx
    T, B, n, m = 5, 4, 64, 16
    pr = problem(51, T, B, n, m)
    b = float(pr["hi"][0, 0, 0])
    kw = dict(T=T, u_lower=-b, u_upper=b, n_batch=B, n_state=n, n_ctrl=m, u_init=None, eps=1e-4, max_iter=20,
              line_search_decay=0.2, max_line_search_iter=10)
    o = obox.box_ddp(pr["x0"], (pr["C"], pr["c"]), ("linear", pr["F"], pr["f"]), T, -b, b, n, m, eps=1e-4,
                     ls_decay=0.2, max_ls_iter=10, max_iter=20, coupling="element")
    assert np.mean(np.abs(np.abs(o["u"]) - b) < 1e-12) >= 0.2 and o["status"] == "converged"
    res = {}
    for mode in (True, False):
        solver = BoxDDP(device_loop=mode, coupling="element", **kw)
        x, u, costs = solver((pr["x0"], QuadCost(pr["C"], pr["c"]), LinDx(pr["F"], pr["f"])))
        res[mode] = (np.asarray(getattr(x, "array", x)), np.asarray(getattr(u, "array", u)), np.asarray(costs), solver.info)
    for mode in (True, False):
        x, u, costs, info = res[mode]
        assert info["n_iter"] == o["n_iter"] and info["status"] == o["status"], (mode, info["n_iter"], o["n_iter"])
        assert rel_err(x, o["x"]) < 1e-9 and rel_err(u, o["u"]) < 1e-9 and rel_err(costs, o["costs"]) < 1e-9
    for i in range(3):
        assert np.array_equal(res[True][i], res[False][i])


def test_facades_mpcstep_and_lqr_active(ctx):
    """MPCstep.apply + backward_numpy / backward_reduced_numpy and LQR_active.solve_recursion at (64, 16), numpy arrays."""
    from mpc_step import MPCstep
    from active_constrained_lqr import LQR_active
    from util import QuadCost, LinDx
    T, B, n, m = 5, 4, 64, 16
    pr = problem(61, T, B, n, m)
    step = MPCstep(pr["u_nom"], T, pr["hi"], pr["lo"], B, n, m, pr["x_nom"], QuadCost(pr["C"], pr["c"]),
                   LinDx(pr["F"], pr["f"]), 0.2, 64, need_expand=True, coupling="element")
    x, u = step.apply((pr["x0"], pr["C"], pr["c"], pr["F"], None))
    x, u = np.asarray(getattr(x, "array", x)), np.asarray(getattr(u, "array", u))
    o = fwd_oracle(pr)
    assert rel_err(x, o["x"]) < 1e-10 and rel_err(u, o["u"]) < 1e-10
    rs = np.random.RandomState(7)
    gx, gu = rs.randn(T, B, n), rs.randn(T, B, m)
    g = step.backward_numpy(gx, gu)
    ob = ompc.step_backward(pr["C"], pr["c"], pr["F"], None, x, u, pr["lo"], pr["hi"], gx, gu, n, m)
    for a, b in zip(g[:4], ob[:4]):
        assert rel_err(a, b) < 1e-10
    r = step.backward_reduced_numpy(gx, gu)
    assert rel_err(r[0], ob[0]) < 1e-10
    assert rel_err(r[1], ob[1].sum((0, 1))) < 1e-9 and rel_err(r[3], ob[3].sum((0, 1))) < 1e-9
    active = rs.rand(T, B, m) < 0.3
    la = LQR_active(pr["x0"], pr["C"], pr["c"], pr["F"], pr["f"], T, n, m, u_zero_Index=active)
    xa, ua = la.solve_recursion()
    xo, uo = ompc.lqr_active(pr["x0"], pr["C"], pr["c"], pr["F"], pr["f"], active, n, m)
    assert rel_err(xa, xo) < 1e-10 and rel_err(ua, uo) < 1e-10


def test_unsupported_shapes(ctx):
    """m = 33 and n = 129 return DMPC_ERR_UNSUPPORTED with a message and launch nothing."""
    import _native
    for n, m in ((8, 33), (129, 8)):
        T, B = 2, 2
        pr = bwd_problem(3, T, B, n, m, F64, pinned=False)
        pr.update(x_nom=pr["x"], u_nom=pr["u"], tC=pr["C"], tc=pr["c"], tF=pr["F"], tf=pr["f"])
        before = ctx.launches
        with pytest.raises(_native.DiffMpcError, match="unsupported|128"):
            run_forward(ctx, pr, F64)
        with pytest.raises(_native.DiffMpcError, match="128"):
            run_backward(ctx, pr, F64)
        assert ctx.launches == before
        bf = Bufs()
        x = bf.empty((T, B, n), np.float64)
        if n + m <= 64:                                 # traj_kernel runs any m at n + m <= 64
            continue
        with pytest.raises(_native.DiffMpcError, match="128"):
            ctx.get_traj(np.float64, T, B, n, m, _native.DYN_LINEAR, bf.put(pr["x"][0], np.float64),
                         bf.put(pr["u"], np.float64), bf.put(pr["F"], np.float64), None, None, bf.ptr(x))
        assert ctx.launches == before


# ------------------------------------------------------------------------------------------------ dispatch
def _first(pred, rng):
    return next(v for v in rng if pred(v))


def selection_shapes():
    """(key, n, m, dt): the boundaries of each selection, derived from the layout sizes."""
    n_fwd = _first(lambda n: fwd_large(n, 8), range(20, 129))            # first n at m = 8 with the large forward
    n_sol = _first(lambda n: solve_large(n, 8), range(20, 129))          # masked solve large
    n_red = _first(lambda n: adj_large(n, 8, True), range(20, 129))      # reduced adjoint large
    n_full = _first(lambda n: adj_large(n, 8, False), range(20, 129))    # full adjoint large
    assert n_sol < n_red < n_full
    return dict(fwd_keep=(n_fwd - 1, 8), fwd_large=(n_fwd, 8), solve_only=(n_sol, 8), red_only=(n_red, 8),
                both=(n_full, 8), traj_keep=(48, 16), traj_large=(49, 16))


def test_kernels_reached():
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "names.npz")
        env = {k: v for k, v in os.environ.items() if not k.startswith("DMPC_")}
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", path], env=env, capture_output=True,
                           text=True, timeout=1200)
        assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-4000:])
        with np.load(path, allow_pickle=False) as z:
            names = {k: list(z[k]) for k in z.files}
    has = lambda key, k: any(k in g for g in names[key])
    assert has("fwd_keep", "mpc_forward_kernel<double, 0, 0, 256") and not has("fwd_keep", "mpc_large")
    for k in ("mpc_large_chat_kernel<double>", "mpc_large_pnqp_kernel<double>", "mpc_large_ls_kernel<double>",
              "lqr_large_q_kernel<double>", "lqr_large_v_kernel<double>"):
        assert has("fwd_large", k), (k, names["fwd_large"])
    assert not has("fwd_large", "mpc_forward_kernel")
    # backward, full and reduced call each: (masked solve, full adjoint, reduced adjoint)
    assert has("solve_only-full", "lqr_large_rollout_kernel<double>") and has("solve_only-full", "adjoint_out_kernel<double")
    assert not has("solve_only-full", "lqr_large_adj_kernel")
    assert has("solve_only-red", "lqr_large_factor_kernel<double>") and has("solve_only-red", "adjoint_out_kernel<double")
    assert has("red_only-red", "lqr_large_adj_kernel<double>") and has("red_only-red", "lqr_large_red_kernel<double>")
    assert has("red_only-full", "adjoint_out_kernel<double") and not has("red_only-full", "lqr_large_adj_kernel")
    assert has("both-full", "lqr_large_adj_kernel<double>") and has("both-full", "lqr_large_outer_kernel<double>")
    assert not has("both-full", "adjoint_out_kernel")
    assert has("traj_keep", "traj_kernel<double, 64>") and not has("traj_keep", "traj_large")
    assert has("traj_large", "traj_large_kernel<double>") and not has("traj_large", "traj_kernel<")


def _child_main(path):
    import torch  # noqa: F401
    from torch.profiler import profile, ProfilerActivity
    import _native
    ctx = _native.default_context(0)
    sh = selection_shapes()
    res = {}

    def trace(key, fn):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            ctx.sync()
        names = set(e.name for e in prof.events())
        try:
            for e in prof.profiler.kineto_results.events():
                names.add(e.name())
        except AttributeError:
            pass
        res[key] = np.array(sorted(k for k in names if "dmpc::" in k))

    for key in ("fwd_keep", "fwd_large"):
        n, m = sh[key]
        pr = problem(1, 3, 2, n, m)
        trace(key, lambda: run_forward(ctx, pr, F64))
    for key in ("solve_only", "red_only", "both"):
        n, m = sh[key]
        pr = bwd_problem(2, 3, 2, n, m, F64)
        T, B, s = 3, 2, n + m
        bf = Bufs()
        C, c, F, x, u, lo, hi, gx, gu = (bf.put(pr[k], np.float64) for k in ("C", "c", "F", "x", "u", "lo", "hi", "gx", "gu"))
        rsz = ctx.reduced_grad_elems(n, m)
        o = {k: bf.ptr(bf.empty(v, np.float64)) for k, v in dict(wK=(T, B, m, n), wk=(T, B, m), wd=(T, B, s), dx0=(B, n),
                                                                   dC=(T, B, s, s), dc=(T, B, s), dF=(T - 1, B, n, s),
                                                                   part=(B, rsz), sums=(rsz,), act=(T * B * m,)).items()}
        trace(key + "-full", lambda: ctx.mpc_step_backward(np.float64, T, B, n, m, C, c, F, T - 1, x, u, lo, hi, gx, gu,
                                                           o["wK"], o["wk"], o["wd"], o["act"], o["dx0"], o["dC"],
                                                           o["dc"], o["dF"], None))
        trace(key + "-red", lambda: ctx.mpc_step_backward_reduced(np.float64, T, B, n, m, C, c, F, T - 1, x, u, lo, hi, gx,
                                                                  gu, o["wK"], o["wk"], o["wd"], o["act"], o["part"],
                                                                  o["dx0"], o["sums"]))
    for key in ("traj_keep", "traj_large"):
        n, m = sh[key]
        T, B = 3, 2
        rs = np.random.RandomState(0)
        bf = Bufs()
        x0, u, F = bf.put(rs.randn(B, n), np.float64), bf.put(rs.randn(T, B, m), np.float64), bf.put(rs.randn(T - 1, B, n, n + m), np.float64)
        x = bf.empty((T, B, n), np.float64)
        trace(key, lambda: ctx.get_traj(np.float64, T, B, n, m, _native.DYN_LINEAR, x0, u, F, None, None, bf.ptr(x)))
    np.savez(path, **res)


if __name__ == "__main__" and len(sys.argv) == 3 and sys.argv[1] == "--child":
    _child_main(sys.argv[2])
