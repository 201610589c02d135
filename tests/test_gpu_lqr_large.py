"""GPU: LQR solve and adjoint at shapes too large for one CTA's shared memory (lqr_large_kernels.cuh, DESIGN.md §4.8).

Every case runs dmpc_lqr_solve (FACTOR | ROLLOUT | SAVE_FAC), dmpc_lqr_adjoint and dmpc_lqr_adjoint_reduced through the
C ABI and compares with the reference recursions (oracle/lqr.py): rel_err 1e-10 in fp64, the suite's 1e-4 / 1e-3 in fp32
on fp32-rounded inputs.  Each entry of a reduced sum must lie within 1e-10 (fp32: 2e-5) times sum |term| of the oracle's
sum, and every case shows from the oracle that this bound fails when element B-1 or the last step is left out.
Outputs start as NaN, so an entry the kernels skip fails.  Which kernels ran is read from a torch.profiler trace taken
in a child process; the largest shapes that fit the per-element kernels are shown to keep them.
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
    sys.path[:0] = [os.path.dirname(os.path.abspath(__file__)), _root, _pkg, os.path.join(_pkg, "lqr")]

from _helpers import rel_err  # noqa: E402
from oracle import lqr as olqr  # noqa: E402

pytestmark = pytest.mark.gpu

F64, F32 = "f64", "f32"
NP = {F64: np.float64, F32: np.float32}
CNAME = {F64: "double", F32: "float"}


def tol(dt, grad=False):
    return 1e-10 if dt == F64 else (1e-3 if grad else 1e-4)


def sum_tol(dt):
    return 1e-10 if dt == F64 else 2e-5


def problem(seed, T, B, n, m, with_f=True, pivot=False, F_T=None, dt=F64):
    """Per-element non-symmetric C_t and F_t that vary with t.  pivot: the control block of C is made of 2 x 2 blocks
    [[0.2, 1], [1.5, 0.3]] and F_u is small, so Quu stays close to C_uu and the pivoted elimination swaps rows."""
    rs = np.random.RandomState(seed)
    s = n + m
    F_T = T - 1 if F_T is None else F_T
    L = 0.85 / np.sqrt(s) * rs.randn(T, B, s, s)
    C = L @ np.swapaxes(L, 2, 3) + np.eye(s) + 0.05 * rs.randn(T, B, s, s)
    F = np.concatenate((0.9 * np.eye(n) + 0.1 / np.sqrt(n) * rs.randn(F_T, B, n, n), 0.3 * rs.randn(F_T, B, n, m)), axis=3)
    if pivot:
        base = np.eye(m)
        for i in range(0, m - 1, 2):
            base[i:i + 2, i:i + 2] = [[0.2, 1.0], [1.5, 0.3]]
        C[:, :, n:, n:] = base + 0.1 * (C[:, :, n:, n:] - np.eye(m))
        F[:, :, :, n:] *= 0.01
    pr = dict(T=T, B=B, n=n, m=m, F_T=F_T, C=C, F=F, c=rs.randn(T, B, s), x0=rs.randn(B, n),
              f=0.1 * rs.randn(T - 1, B, n) if with_f else None, gx=rs.randn(T, B, n), gu=rs.randn(T, B, m))
    if dt == F32:
        pr = {k: (v.astype(np.float32).astype(np.float64) if isinstance(v, np.ndarray) else v) for k, v in pr.items()}
    return pr


def oracle(pr, strict):
    T, B, n, m = pr["T"], pr["B"], pr["n"], pr["m"]
    F = pr["F"][:T - 1]
    x, u, Ks, ks = olqr.lqr_solve(pr["x0"], pr["C"], pr["c"], F, pr["f"], n, m)
    dx0, dC, dc, dF, df = olqr.difflqr_backward(pr["x0"], pr["C"], pr["c"], F, x, u, pr["gx"], pr["gu"], n, m, strict, strict)
    # sum |term| bounds of the reduced sums, from lambda / d-lambda of the reference recursions
    tau, dtau = np.concatenate((x, u), 2), dc
    lam, dlam = np.zeros((T, B, n)), np.zeros((T, B, n))
    for t in range(T - 1, -1, -1):
        lam[t] = np.einsum("bij,bj->bi", pr["C"][t][:, :n], tau[t]) + pr["c"][t][:, :n]
        dlam[t] = np.einsum("bij,bj->bi", pr["C"][t][:, :n], dtau[t]) + pr["gx"][t]
        if t < T - 1:
            lam[t] += np.einsum("bji,bj->bi", F[t][:, :, :n], lam[t + 1])
            dlam[t] += np.einsum("bji,bj->bi", F[t][:, :, :n], dlam[t + 1])
    a = np.einsum("tbi,tbj->tbij", np.abs(dtau), np.abs(tau))
    bC = 0.5 * a + np.swapaxes(a, 2, 3) if strict else 0.5 * (a + np.swapaxes(a, 2, 3))
    bF = (np.einsum("tbi,tbj->tbij", np.abs(dlam[1:]), np.abs(tau[:-1])) +
          np.einsum("tbi,tbj->tbij", np.abs(lam[1:]), np.abs(dtau[:-1])))
    bf = np.abs(dlam[:T - 1]) if strict else np.abs(dlam[1:])
    return dict(x=x, u=u, Ks=Ks, ks=ks, dx0=dx0, dC=dC, dc=dc, dF=dF, df=df, bC=bC, bF=bF, bf=bf)


def assert_sum(got, want, bound, eps, what):
    err = np.abs(np.asarray(got, np.float64) - want)
    worst = float(np.max(err / (eps * bound + 1e-300))) if err.size else 0.0
    assert worst <= 1.0, (what, worst)


def assert_bounds_are_sharp(o, eps):
    """Leaving out element B-1, or the last step, moves a sum by more than its bound somewhere."""
    T, B = o["dC"].shape[:2]
    lim = lambda b: eps * b + 1e-300
    bC = o["bC"].sum((0, 1))
    assert np.max(np.abs(o["dC"][:, B - 1].sum(0)) / lim(bC)) > 1.0
    assert np.max(np.abs(o["dC"][T - 1].sum(0)) / lim(bC)) > 1.0
    if T > 1:
        bF = o["bF"].sum((0, 1))
        assert np.max(np.abs(o["dF"][:, B - 1].sum(0)) / lim(bF)) > 1.0
        assert np.max(np.abs(o["dF"][T - 2].sum(0)) / lim(bF)) > 1.0


class Bufs:
    """Device tensors `off` elements past the start of a torch allocation (off = 1: aligned to the element type, not to
    16 bytes).  Outputs start as NaN."""

    def __init__(self, off=0):
        import torch
        self.torch, self.off, self.keep = torch, off, []

    def _t(self, dt):
        return {np.dtype(np.float64): self.torch.float64, np.dtype(np.float32): self.torch.float32}[np.dtype(dt)]

    def put(self, a, dt):
        a = np.ascontiguousarray(a, dtype=dt)
        t = self.torch.zeros(a.size + self.off, dtype=self._t(dt), device="cuda")
        t[self.off:].copy_(self.torch.from_numpy(a.reshape(-1)))
        self.keep.append(t)
        return t.data_ptr() + self.off * t.element_size()

    def empty(self, shape, dt):
        t = self.torch.full((int(np.prod(shape)) + self.off,), float("nan"), dtype=self._t(dt), device="cuda")
        self.keep.append(t)
        return (t, shape)

    def ptr(self, b):
        return b[0].data_ptr() + self.off * b[0].element_size()

    def get(self, b):
        return b[0][self.off:].cpu().numpy().reshape(b[1])


def run(ctx, pr, dt, strict, off=0, df_null=False, repeat=False):
    """Forward (FACTOR | ROLLOUT | SAVE_FAC), full and reduced adjoint through the C ABI; a dict of host arrays."""
    import _native
    T, B, n, m, F_T = pr["T"], pr["B"], pr["n"], pr["m"], pr["F_T"]
    s, R = n + m, NP[dt]
    bf = Bufs(off)
    x0, C, c = bf.put(pr["x0"], R), bf.put(pr["C"], R), bf.put(pr["c"], R)
    F = bf.put(pr["F"], R) if F_T else None
    f = bf.put(pr["f"], R) if pr["f"] is not None else None
    gx, gu = bf.put(pr["gx"], R), bf.put(pr["gu"], R)
    Tm = max(T - 1, 1)
    rsz = ctx.reduced_grad_elems(n, m)
    o = {k: bf.empty(v, R) for k, v in dict(x=(T, B, n), u=(T, B, m), Ks=(T, B, m, n), ks=(T, B, m),
                                             fac=(ctx.lqr_fac_elems(T, B, n, m),), dx0=(B, n), dC=(T, B, s, s),
                                             dc=(T, B, s), dF=(Tm, B, n, s), df=(Tm, B, n), rdx0=(B, n),
                                             wdt=(T, B, s), part=(B, rsz), sums=(rsz,)).items()}
    P = {k: bf.ptr(v) for k, v in o.items()}
    flags = _native.ADJ_STRICT_REFERENCE if strict else 0

    def call():
        ctx.lqr_solve(R, T, B, n, m, x0, C, c, F, F_T, f, P["x"], P["u"], P["Ks"], P["ks"], P["fac"],
                      _native.LQR_FACTOR | _native.LQR_ROLLOUT | _native.LQR_SAVE_FAC)
        ctx.lqr_adjoint(R, T, B, n, m, C, c, F, P["x"], P["u"], gx, gu, P["Ks"], P["fac"], P["dx0"], P["dC"], P["dc"],
                        P["dF"], None if df_null else P["df"], flags)
        ctx.lqr_adjoint_reduced(R, T, B, n, m, C, c, F, P["x"], P["u"], gx, gu, P["Ks"], P["fac"], P["wdt"],
                                P["part"], P["rdx0"], P["sums"], flags)
        ctx.sync()
        out = {k: bf.get(v) for k, v in o.items() if k not in ("fac", "wdt", "part")}
        out["dF"], out["df"] = out["dF"][:T - 1], out["df"][:T - 1]
        return out

    out = call()
    if repeat:
        out["again"] = call()
    return out


def check(pr, dt, strict, out, df_null=False):
    o = oracle(pr, strict)
    T, n, m = pr["T"], pr["n"], pr["m"]
    for k in ("x", "u", "Ks", "ks"):
        assert rel_err(out[k], o[k]) < tol(dt), k
    for k in ("dx0", "dC", "dc", "dF") + (() if df_null else ("df",)):
        assert rel_err(out[k], o[k]) < tol(dt, True), k
    assert rel_err(out["rdx0"], o["dx0"]) < tol(dt, True)
    sC, sc, sF, sf = (out["sums"][:(n + m) ** 2].reshape(n + m, n + m), out["sums"][(n + m) ** 2:(n + m) * (n + m + 1)],
                      out["sums"][(n + m) * (n + m + 1):(n + m) * (n + m + 1) + n * (n + m)].reshape(n, n + m),
                      out["sums"][(n + m) * (n + m + 1) + n * (n + m):])
    eps = sum_tol(dt)
    assert_sum(sC, o["dC"].sum((0, 1)), o["bC"].sum((0, 1)), eps, "sum dC")
    assert_sum(sc, o["dc"].sum((0, 1)), np.abs(o["dc"]).sum((0, 1)), eps, "sum dc")
    if T > 1:
        assert_sum(sF, o["dF"].sum((0, 1)), o["bF"].sum((0, 1)), eps, "sum dF")
        assert_sum(sf, o["df"].sum((0, 1)), o["bf"].sum((0, 1)), eps, "sum df")
    else:
        assert not np.any(sF) and not np.any(sf)
    assert_bounds_are_sharp(o, eps)


# (dt, n, m, T, B, f given, strict, pointer offset, F_T - (T - 1), pivoting Quu, df NULL)
CASES = [
    dict(dt=F64, n=58, m=8, T=17, B=3, with_f=True, strict=True, off=0, extra=0, pivot=False, df_null=False),
    dict(dt=F64, n=64, m=1, T=2, B=3, with_f=True, strict=False, off=1, extra=1, pivot=False, df_null=False),
    dict(dt=F64, n=64, m=8, T=50, B=3, with_f=False, strict=True, off=0, extra=0, pivot=True, df_null=False),
    dict(dt=F64, n=64, m=16, T=17, B=1, with_f=True, strict=False, off=0, extra=1, pivot=False, df_null=True),
    dict(dt=F64, n=61, m=7, T=17, B=37, with_f=True, strict=True, off=1, extra=0, pivot=True, df_null=False),
    dict(dt=F64, n=100, m=1, T=1, B=3, with_f=False, strict=True, off=0, extra=0, pivot=False, df_null=False),
    dict(dt=F64, n=96, m=32, T=17, B=3, with_f=True, strict=False, off=0, extra=0, pivot=True, df_null=False),
    dict(dt=F64, n=128, m=32, T=2, B=3, with_f=True, strict=True, off=1, extra=0, pivot=False, df_null=False),
    dict(dt=F32, n=85, m=8, T=17, B=3, with_f=True, strict=True, off=1, extra=0, pivot=False, df_null=False),
    dict(dt=F32, n=128, m=32, T=17, B=3, with_f=False, strict=False, off=0, extra=1, pivot=True, df_null=False),
]
# the largest shapes the per-element kernels hold: they keep those kernels
KEEP = [dict(dt=F64, n=57, m=8), dict(dt=F64, n=63, m=1), dict(dt=F32, n=84, m=8)]


def case_id(c):
    return "%s-n%d-m%d-T%d-B%d-f%d-s%d-o%d-x%d-p%d-d%d" % (c["dt"], c["n"], c["m"], c["T"], c["B"], c["with_f"], c["strict"],
                                                         c["off"], c["extra"], c["pivot"], c["df_null"])


def problem_of(c):
    return problem(zlib.crc32(case_id(c).encode()) % 1000, c["T"], c["B"], c["n"], c["m"], c["with_f"], c["pivot"],
                   c["T"] - 1 + c["extra"], c["dt"])


@pytest.fixture(scope="module")
def ctx():
    import _native
    return _native.default_context(0)


@pytest.mark.parametrize("c", CASES, ids=case_id)
def test_large_against_oracle(ctx, c):
    pr = problem_of(c)
    out = run(ctx, pr, c["dt"], c["strict"], c["off"], c["df_null"], repeat=True)
    check(pr, c["dt"], c["strict"], out, c["df_null"])
    for k, v in out["again"].items():                                 # a repeated call returns the same bits
        assert np.array_equal(v, out[k], equal_nan=True), k


@pytest.mark.parametrize("dt", [F64, F32])
def test_factor_only_and_rollout_only(ctx, dt):
    """FACTOR alone (no SAVE_FAC) gives the oracle's gains; ROLLOUT alone on the oracle's gains gives its trajectory."""
    import _native
    T, B, n, m = 17, 3, 96, 16
    pr = problem(5, T, B, n, m, dt=dt)
    o = oracle(pr, True)
    R = NP[dt]
    bf = Bufs(1)
    x0, C, c, F, f = (bf.put(pr[k], R) for k in ("x0", "C", "c", "F", "f"))
    Ks, ks, x, u = (bf.empty(v, R) for v in ((T, B, m, n), (T, B, m), (T, B, n), (T, B, m)))
    ctx.lqr_solve(R, T, B, n, m, x0, C, c, F, T - 1, f, None, None, bf.ptr(Ks), bf.ptr(ks), None, _native.LQR_FACTOR)
    ctx.sync()
    assert rel_err(bf.get(Ks), o["Ks"]) < tol(dt) and rel_err(bf.get(ks), o["ks"]) < tol(dt)
    oK, ok_ = bf.put(o["Ks"], R), bf.put(o["ks"], R)
    ctx.lqr_solve(R, T, B, n, m, x0, None, None, F, T - 1, f, bf.ptr(x), bf.ptr(u), oK, ok_, None, _native.LQR_ROLLOUT)
    ctx.sync()
    assert rel_err(bf.get(x), o["x"]) < tol(dt) and rel_err(bf.get(u), o["u"]) < tol(dt)


def test_unsupported_shapes(ctx):
    """m = 33 and n = 129 return DMPC_ERR_UNSUPPORTED with a message and launch nothing."""
    import _native
    bf = Bufs()
    for n, m in ((8, 33), (129, 8)):
        T, B, s = 2, 2, n + m
        pr = problem(1, T, B, n, m)
        C, c, F, x0 = (bf.put(pr[k], np.float64) for k in ("C", "c", "F", "x0"))
        o = {k: bf.ptr(bf.empty(v, np.float64)) for k, v in dict(x=(T, B, n), u=(T, B, m), Ks=(T, B, m, n), ks=(T, B, m),
                                                                   fac=(ctx.lqr_fac_elems(T, B, n, m),), dx0=(B, n),
                                                                   dC=(T, B, s, s), dc=(T, B, s), dF=(1, B, n, s),
                                                                   part=(B, ctx.reduced_grad_elems(n, m)),
                                                                   sums=(ctx.reduced_grad_elems(n, m),)).items()}
        before = ctx.launches
        with pytest.raises(_native.DiffMpcError, match="unsupported"):
            ctx.lqr_solve(np.float64, T, B, n, m, x0, C, c, F, T - 1, None, o["x"], o["u"], o["Ks"], o["ks"], o["fac"],
                          _native.LQR_FACTOR | _native.LQR_ROLLOUT | _native.LQR_SAVE_FAC)
        if n > 128:
            with pytest.raises(_native.DiffMpcError, match="n <= 128"):
                ctx.lqr_adjoint(np.float64, T, B, n, m, C, c, F, o["x"], o["u"], x0, o["ks"], o["Ks"], o["fac"],
                                o["dx0"], o["dC"], o["dc"], o["dF"], None)
            with pytest.raises(_native.DiffMpcError, match="n <= 128"):
                ctx.lqr_adjoint_reduced(np.float64, T, B, n, m, C, c, F, o["x"], o["u"], x0, o["ks"], o["Ks"], o["fac"],
                                        o["dc"], o["part"], o["dx0"], o["sums"])
        assert ctx.launches == before
        assert "128" in ctx.lib.dmpc_last_error(ctx.h).decode()


# ------------------------------------------------------------------------------------------------ facades
def test_difflqr_and_recursion(ctx):
    """DiffLqr forward + backward + backward_reduced_numpy and LqrRecursion at fp64 (64, 8): the large forward feeds
    the per-element full adjoint (it still fits at this shape) and the large reduced adjoint."""
    from differentiable_lqr import DiffLqr
    from lqr_recursion import LqrRecursion
    T, B, n, m = 17, 5, 64, 8
    pr = problem(11, T, B, n, m, pivot=True)
    o = oracle(pr, True)
    node = DiffLqr(T, B, n, m)
    x, u = node.apply_numpy(pr["x0"], pr["C"], pr["c"], pr["F"], pr["f"])
    assert rel_err(x, o["x"]) < 1e-10 and rel_err(u, o["u"]) < 1e-10
    g = node.backward_numpy(pr["gx"], pr["gu"])
    for k, v in zip(("dx0", "dC", "dc", "dF", "df"), g):
        assert rel_err(v, o[k]) < 1e-10, k
    r = node.backward_reduced_numpy(pr["gx"], pr["gu"])
    assert rel_err(r[0], o["dx0"]) < 1e-10
    assert_sum(r[1], o["dC"].sum((0, 1)), o["bC"].sum((0, 1)), 1e-10, "sum dC")
    assert_sum(r[3], o["dF"].sum((0, 1)), o["bF"].sum((0, 1)), 1e-10, "sum dF")
    rec = LqrRecursion(pr["x0"], pr["C"], pr["c"], pr["F"], pr["f"], T, n, m)
    res = rec.solve_recursion()
    assert rel_err(np.asarray(res[0]), o["x"]) < 1e-10 and rel_err(np.asarray(res[1]), o["u"]) < 1e-10


def test_difflqr_shared_past_old_sweep_limit(ctx):
    """DiffLqrShared at fp64 (64, 8): its B = 1 sweep needs the large kernels; the chunk kernels still hold the shape."""
    from differentiable_lqr import DiffLqrShared
    T, B, n, m = 17, 6, 64, 8
    pr = problem(13, T, 1, n, m)
    C, F = pr["C"][:, 0], pr["F"][:, 0]
    rs = np.random.RandomState(3)
    x0, c, f = rs.randn(B, n), rs.randn(T, B, n + m), 0.1 * rs.randn(T - 1, B, n)
    gx, gu = rs.randn(T, B, n), rs.randn(T, B, m)
    Cb = np.ascontiguousarray(np.broadcast_to(C[:, None], (T, B, n + m, n + m)))
    Fb = np.ascontiguousarray(np.broadcast_to(F[:, None], (T - 1, B, n, n + m)))
    x_o, u_o, _, _ = olqr.lqr_solve(x0, Cb, c, Fb, f, n, m)
    dx0_o, dC_o, dc_o, dF_o, df_o = olqr.difflqr_backward(x0, Cb, c, Fb, x_o, u_o, gx, gu, n, m)
    node = DiffLqrShared(T, B, n, m)
    x, u = node.apply_numpy(x0, C, c, F, f)
    assert rel_err(x, x_o) < 1e-10 and rel_err(u, u_o) < 1e-10
    dx0, dC, dc, dF, df = node.backward_numpy(gx, gu)
    assert rel_err(dx0, dx0_o) < 1e-10 and rel_err(dc, dc_o) < 1e-10 and rel_err(df, df_o) < 1e-10
    assert np.max(np.abs(dC - dC_o.sum(1))) <= 1e-10 * np.max(np.abs(dC_o).sum(1))
    assert np.max(np.abs(dF - dF_o.sum(1))) <= 1e-10 * np.max(np.abs(dF_o).sum(1))


def test_lqrnet_links_beyond_chunk_layout(ctx):
    """LqrNet and LqrNet_cost_dx at (96, 32), where the shared chunk kernels do not fit: the per-element route, with
    the reference's seeding and the oracle's summed gradients."""
    import _native
    from differentiable_lqr import LqrNet, LqrNet_cost_dx
    T, B, n, m = 5, 3, 96, 32
    s = n + m
    with pytest.raises(_native.DiffMpcError):
        ctx.lqr_shared_workspace_bytes(np.float64, T, B, n, m)
    rs = np.random.RandomState(4)
    x0, f = rs.randn(B, n), 0.1 * rs.randn(T - 1, B, n)
    gx, gu = rs.randn(T, B, n), rs.randn(T, B, m)
    C = np.ascontiguousarray(np.broadcast_to(np.eye(s), (T, B, s, s)))
    c = rs.randn(T, B, s)
    net = LqrNet(T, B, n, m, seed=0)
    x, u = net.forward((x0, C, c, f))
    Fm = np.concatenate((net.A.array, net.B.array), 1)
    Fb = np.ascontiguousarray(np.broadcast_to(Fm, (T - 1, B, n, s)))
    x_o, u_o, _, _ = olqr.lqr_solve(x0, C, c, Fb, f, n, m)
    assert rel_err(np.asarray(getattr(x, "array", x)), x_o) < 1e-10
    gA, gB = net.backward_numpy(gx, gu)
    d = olqr.difflqr_backward(x0, C, c, Fb, x_o, np.asarray(getattr(u, "array", u)), gx, gu, n, m)
    gF = d[3].sum((0, 1))
    assert np.max(np.abs(np.concatenate((gA, gB), 1) - gF)) <= 1e-9 * np.max(np.abs(d[3]).sum((0, 1)))

    # The reference's seeding of LqrNet_cost_dx (C = I + 0.2 randn, not positive definite) is ill-conditioned at this
    # size: the oracle itself moves by ~4e-7 (u) when C is perturbed by one part in 1e16.  The bound is 10x that measured
    # sensitivity (at least 1e-10 / 1e-9), so it still fails on a wrong step but not on rounding.
    net2 = LqrNet_cost_dx(T, B, n, m, seed=0)
    x, u = net2.forward((x0, f))
    Cp, cp = net2.C.array, net2.c.array
    Fm = np.concatenate((net2.A.array, net2.B.array), 1)
    cb = np.ascontiguousarray(np.broadcast_to(cp, (T, B, s)))
    Fb = np.ascontiguousarray(np.broadcast_to(Fm, (T - 1, B, n, s)))

    def ref(Cm):
        Cb = np.ascontiguousarray(np.broadcast_to(Cm, (T, B, s, s)))
        xo, uo, _, _ = olqr.lqr_solve(x0, Cb, cb, Fb, f, n, m)
        return uo, olqr.difflqr_backward(x0, Cb, cb, Fb, xo, uo, gx, gu, n, m)

    u_o, d = ref(Cp)
    u_p, d_p = ref(Cp * (1 + 1e-16 * np.random.RandomState(1).randn(s, s)))
    assert rel_err(np.asarray(getattr(u, "array", u)), u_o) < max(1e-10, 10 * rel_err(u_p, u_o))
    gA, gB, gC, gc = net2.backward_numpy(gx, gu)
    for got, full, full_p in ((np.concatenate((gA, gB), 1), d[3], d_p[3]), (gC, d[1], d_p[1]), (gc, d[2], d_p[2])):
        assert got.shape == full.shape[2:]
        scale = np.max(np.abs(full).sum((0, 1)))
        sens = np.max(np.abs(full_p.sum((0, 1)) - full.sum((0, 1)))) / scale
        assert np.max(np.abs(got - full.sum((0, 1)))) <= max(1e-9, 10 * sens) * scale


# ------------------------------------------------------------------------------------------------ dispatch
def test_kernels_reached():
    """In a child process under torch.profiler: every case runs the large forward and the large reduced adjoint (the
    full adjoint at fp64 (64, 8) and below stays on lqr_dtau_kernel / adjoint_out_kernel); the largest shapes that fit
    today keep lqr_solve_kernel<..., 0, 0, 256> and their adjoint kernels and never reach the large ones."""
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "names.npz")
        env = {k: v for k, v in os.environ.items() if not k.startswith("DMPC_")}
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", path], env=env, capture_output=True,
                           text=True, timeout=1200)
        assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-4000:])
        with np.load(path, allow_pickle=False) as z:
            names = {k: list(z[k]) for k in z.files}
    for c in CASES:
        got = names[case_id(c)]
        R = CNAME[c["dt"]]
        for k in ("q", "factor", "rollout"):
            assert any("lqr_large_%s_kernel<%s>" % (k, R) in g for g in got), (case_id(c), k, got)
        # each adjoint call ran: the large kernels, or (where the per-element ones still fit) lqr_dtau + adjoint_out
        old = any("lqr_dtau_kernel<%s" % R in g for g in got) and any("adjoint_out_kernel<%s" % R in g for g in got)
        assert any("lqr_large_adj_kernel<%s>" % R in g for g in got) or old, (case_id(c), got)
        if c["T"] > 1:
            assert any("lqr_large_v_kernel<%s>" % R in g for g in got), (case_id(c), got)
    for c in KEEP:
        got = names["keep-%s-%d-%d" % (c["dt"], c["n"], c["m"])]
        R = CNAME[c["dt"]]
        assert not any("lqr_large" in g for g in got), got
        for k in ("lqr_solve_kernel<%s, 0, 0, 256>" % R, "lqr_dtau_kernel<%s, 0, 0, 64" % R, "adjoint_out_kernel<%s, 0, 0, 128" % R):
            assert any(k in g for g in got), (c, k, got)


def _child_main(path):
    import torch  # noqa: F401
    from torch.profiler import profile, ProfilerActivity
    import _native
    ctx = _native.default_context(0)
    res = {}
    jobs = [(case_id(c), problem_of(c), c) for c in CASES]
    jobs += [("keep-%s-%d-%d" % (c["dt"], c["n"], c["m"]), problem(2, 3, 2, c["n"], c["m"], dt=c["dt"]),
              dict(dt=c["dt"], strict=True, off=0, df_null=False)) for c in KEEP]
    for key, pr, c in jobs:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run(ctx, pr, c["dt"], c["strict"], c["off"], c["df_null"])
            ctx.sync()
        names = set(e.name for e in prof.events())
        try:
            for e in prof.profiler.kineto_results.events():
                names.add(e.name())
        except AttributeError:
            pass
        res[key] = np.array(sorted(k for k in names if "dmpc::" in k))
    np.savez(path, **res)


if __name__ == "__main__" and len(sys.argv) == 3 and sys.argv[1] == "--child":
    _child_main(sys.argv[2])
