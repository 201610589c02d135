"""GPU, torch-free, ~3 s: the thread-per-element LQR kernels (csrc/lqr_tpe_kernel.cuh) launched with thin warps (8 / 16 elements
per warp, DMPC_LQR_TPE_EPW=auto) against the oracle: forward + adjoint on four shapes, slices at both ends and in the middle of
the batch.  Prints EPW_CHECK PASS|FAIL.  A quick profiling-side check; the test suite covers the same shapes in
tests/test_gpu_dispatch_matrix.py (setting epw_auto)."""
import os, sys, time
os.environ.setdefault("DMPC_LQR_TPE_EPW", "auto")
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "chainer-differentiable-mpc_b200")):
    sys.path.insert(0, p)
import types
import numpy as np
sys.modules.setdefault('torch', types.ModuleType('torch'))   # oracle.linalg imports torch for the LU of PNQP only; not needed here
import _native
from _helpers import lqr_problem, rel_err
from oracle import lqr as olqr


def run_solve(ctx, pr, dtype=np.float64, save_fac=True):
    T, B, n, m = pr["C"].shape[0], pr["C"].shape[1], int(pr["n"]), int(pr["m"])
    s = n + m
    d = {k: ctx.to_device(pr[k], dtype) for k in ("x0", "C", "c")}
    F = pr["F"]
    dF = ctx.to_device(F, dtype)
    df = ctx.to_device(pr["f"], dtype)
    x = ctx.empty((T, B, n), dtype); u = ctx.empty((T, B, m), dtype)
    Ks = ctx.empty((T, B, m, n), dtype); ks = ctx.empty((T, B, m), dtype)
    fac = ctx.empty((ctx.lqr_fac_elems(T, B, n, m),), dtype)
    flags = _native.LQR_FACTOR | _native.LQR_ROLLOUT | _native.LQR_SAVE_FAC
    ctx.lqr_solve(dtype, T, B, n, m, d["x0"], d["C"], d["c"], dF, T - 1, df, x, u, Ks, ks, fac, flags)
    ctx.sync()
    return dict(x=x, u=u, Ks=Ks, ks=ks, fac=fac, C=d["C"], c=d["c"], F=dF, f=df, x0=d["x0"], T=T, B=B, n=n, m=m)


def run_adjoint(ctx, r, gx, gu, dtype=np.float64):
    T, B, n, m = r["T"], r["B"], r["n"], r["m"]
    s = n + m
    dgx = ctx.to_device(gx, dtype); dgu = ctx.to_device(gu, dtype)
    dx0 = ctx.empty((B, n), dtype); dC = ctx.empty((T, B, s, s), dtype); dc = ctx.empty((T, B, s), dtype)
    dF = ctx.empty((max(T - 1, 1), B, n, s), dtype); df = ctx.empty((max(T - 1, 1), B, n), dtype)
    ctx.lqr_adjoint(dtype, T, B, n, m, r["C"], r["c"], r["F"], r["x"], r["u"], dgx, dgu, r["Ks"], r["fac"],
                    dx0, dC, dc, dF, df, _native.ADJ_STRICT_REFERENCE)
    ctx.sync()
    return [dx0.download(), dC.download(), dc.download(), dF.download()[:T - 1], df.download()[:T - 1]]

ctx = _native.default_context(0)
worst = 0.0
for (T, B, n, m) in ((50, 4096, 4, 2), (20, 8192, 3, 1), (7, 4737, 4, 2), (6, 130, 2, 1)):
    pr = lqr_problem(B + n, T, B, n, m, with_f=True)
    rs = np.random.RandomState(4)
    gx, gu = rs.randn(T, B, n), rs.randn(T, B, m)
    r = run_solve(ctx, pr)
    out = run_adjoint(ctx, r, gx, gu)
    got = {k: r[k].download() for k in ("x", "u", "Ks", "ks")}
    w = 0.0
    for sl in (slice(0, 20), slice(B // 2 - 9, B // 2 + 9), slice(B - 19, B)):
        ox, ou, oK, ok = olqr.lqr_solve(pr["x0"][sl], pr["C"][:, sl], pr["c"][:, sl], pr["F"][:, sl], pr["f"][:, sl], n, m)
        for a, b in ((got["x"], ox), (got["u"], ou), (got["Ks"], oK), (got["ks"], ok)):
            w = max(w, rel_err(a[:, sl], b))
        want = olqr.difflqr_backward(pr["x0"][sl], pr["C"][:, sl], pr["c"][:, sl], pr["F"][:, sl], ox, ou, gx[:, sl], gu[:, sl],
                                     n, m, quirk_dC=True, quirk_df=True)
        w = max(w, rel_err(out[0][sl], want[0]))
        for a, b in zip(out[1:], want[1:]):
            w = max(w, rel_err(a[:, sl], b))
    # every element finite and the batch-wide sums reproducible: a second run must be bit-identical
    r2 = run_solve(ctx, pr)
    same = np.array_equal(r2["x"].download(), got["x"]) and np.isfinite(got["x"]).all() and all(np.isfinite(o).all() for o in out)
    print("shape", (T, B, n, m), "max_rel", w, "finite+repeatable", bool(same), flush=True)
    worst = max(worst, w)
print("EPW_CHECK", "PASS" if worst < 1e-10 else "FAIL", worst)
