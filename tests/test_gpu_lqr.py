"""GPU parity: lqr_solve / lqr_adjoint kernels (through the C ABI) vs the oracle and the golden fixtures.

Reference behaviour: lqr/lqr_recursion.py:69-209 and lqr/differentiable_lqr.py:78-142.
Tolerances (BASELINE.json north_star): 1e-10 relative in fp64, 1e-4 relative in fp32.
"""
import numpy as np
import pytest

import _native
from _helpers import load_golden, rel_err, lqr_problem
from oracle import lqr as olqr

pytestmark = pytest.mark.gpu

TOL = {np.float64: 1e-10, np.float32: 1e-4}


@pytest.fixture(scope="module")
def ctx():
    return _native.default_context(0)


def run_solve(ctx, pr, dtype=np.float64, save_fac=True):
    T, B, n, m = pr["C"].shape[0], pr["C"].shape[1], int(pr["n"]), int(pr["m"])
    s = n + m
    d = {k: ctx.to_device(pr[k], dtype) for k in ("x0", "C", "c")}
    F = pr["F"]
    dF = ctx.to_device(F if F.size else np.zeros((1, B, n, s)), dtype)
    f = pr.get("f")
    df = None if f is None else ctx.to_device(f if f.size else np.zeros((1, B, n)), dtype)
    x = ctx.empty((T, B, n), dtype); u = ctx.empty((T, B, m), dtype)
    Ks = ctx.empty((T, B, m, n), dtype); ks = ctx.empty((T, B, m), dtype)
    fac = ctx.empty((ctx.lqr_fac_elems(T, B, n, m),), dtype) if save_fac else None
    flags = _native.LQR_FACTOR | _native.LQR_ROLLOUT | (_native.LQR_SAVE_FAC if save_fac else 0)
    ctx.lqr_solve(dtype, T, B, n, m, d["x0"], d["C"], d["c"], dF, max(T - 1, F.shape[0]), df, x, u, Ks, ks, fac, flags)
    ctx.sync()
    return dict(x=x, u=u, Ks=Ks, ks=ks, fac=fac, C=d["C"], c=d["c"], F=dF, f=df, x0=d["x0"], T=T, B=B, n=n, m=m)


GOLDEN = ["boyd", "onevar", "lqr_n4m2", "lqr_n4m2_nof", "lqr_n3m1_f", "lqr_n5m3_nonsym", "lqr_n8m4", "lqr_T1"]


@pytest.mark.parametrize("name", GOLDEN)
def test_lqr_solve_golden(ctx, name):
    g = load_golden(name)
    if g["F"].shape[0] == g["C"].shape[0]:          # examples pass T rows of F (Q8)
        g["F"] = g["F"][:-1]
    r = run_solve(ctx, g)
    assert rel_err(r["x"].download(), g["x"]) < 1e-10
    assert rel_err(r["u"].download(), g["u"]) < 1e-10
    assert rel_err(r["Ks"].download(), g["Ks"]) < 1e-10
    assert rel_err(r["ks"].download(), g["ks"]) < 1e-10


SHAPES = [  # (T, B, n, m, with_f)  - specialised and runtime-shape kernels, ragged batch sizes
    (20, 64, 3, 1, True), (50, 257, 4, 2, True), (50, 33, 8, 4, True), (12, 5, 32, 8, True),
    (9, 7, 5, 3, False), (6, 3, 12, 6, True), (5, 2, 20, 10, False), (30, 1, 2, 1, True), (4, 130, 6, 1, True),
]


@pytest.mark.parametrize("T,B,n,m,with_f", SHAPES)
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_lqr_solve_random(ctx, T, B, n, m, with_f, dtype):
    pr = lqr_problem(T * 1000 + B + n, T, B, n, m, with_f=with_f)
    ox, ou, oK, ok = olqr.lqr_solve(pr["x0"], pr["C"], pr["c"], pr["F"], pr["f"], n, m)
    r = run_solve(ctx, pr, dtype)
    tol = TOL[dtype]
    assert rel_err(r["Ks"].download(), oK) < tol
    assert rel_err(r["ks"].download(), ok) < tol
    assert rel_err(r["x"].download(), ox) < tol
    assert rel_err(r["u"].download(), ou) < tol


def run_adjoint(ctx, r, gx, gu, dtype=np.float64, strict=True):
    T, B, n, m = r["T"], r["B"], r["n"], r["m"]
    s = n + m
    dgx = ctx.to_device(gx, dtype); dgu = ctx.to_device(gu, dtype)
    dx0 = ctx.empty((B, n), dtype); dC = ctx.empty((T, B, s, s), dtype); dc = ctx.empty((T, B, s), dtype)
    dF = ctx.empty((max(T - 1, 1), B, n, s), dtype); df = ctx.empty((max(T - 1, 1), B, n), dtype)
    ctx.lqr_adjoint(dtype, T, B, n, m, r["C"], r["c"], r["F"], r["x"], r["u"], dgx, dgu, r["Ks"], r["fac"],
                    dx0, dC, dc, dF, df, _native.ADJ_STRICT_REFERENCE if strict else 0)
    ctx.sync()
    return [dx0.download(), dC.download(), dc.download(), dF.download()[:T - 1], df.download()[:T - 1]]


@pytest.mark.parametrize("name", [c for c in GOLDEN if c not in ("boyd", "onevar", "lqr_T1")])
def test_lqr_adjoint_golden(ctx, name):
    g = load_golden(name)
    r = run_solve(ctx, g)
    out = run_adjoint(ctx, r, g["gx"], g["gu"])
    for a, k in zip(out, ("dx0", "dC", "dc", "dF", "df")):
        assert rel_err(a, g[k]) < 1e-10, k


@pytest.mark.parametrize("T,B,n,m,with_f", [s for s in SHAPES if s[0] > 1])
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("strict", [True, False])
def test_lqr_adjoint_random(ctx, T, B, n, m, with_f, dtype, strict):
    pr = lqr_problem(T * 77 + B + m, T, B, n, m, with_f=with_f, sym=(n % 2 == 0))
    rs = np.random.RandomState(3)
    gx, gu = rs.randn(T, B, n), rs.randn(T, B, m)
    ox, ou, _, _ = olqr.lqr_solve(pr["x0"], pr["C"], pr["c"], pr["F"], pr["f"], n, m)
    want = olqr.difflqr_backward(pr["x0"], pr["C"], pr["c"], pr["F"], ox, ou, gx, gu, n, m,
                                 quirk_dC=strict, quirk_df=strict)
    r = run_solve(ctx, pr, dtype)
    out = run_adjoint(ctx, r, gx, gu, dtype, strict)
    for a, b, k in zip(out, want, ("dx0", "dC", "dc", "dF", "df")):
        assert rel_err(a, b) < TOL[dtype] * (10 if dtype == np.float32 else 1), k


@pytest.mark.parametrize("B,n,m", [(9601, 4, 2), (19003, 3, 1)])
def test_tpe_kernels_other_launch_geometries(ctx, B, n, m):
    """lqr_tpe_kernel / lqr_dtau_tpe_kernel (s <= 6) pick their operand-ring depth and CTA size from the batch: every other
    test runs the deep-ring, one-warp-CTA form (B <= 9472).  9601 -> shallow rings, 32-thread CTAs; 19003 -> shallow rings,
    64-thread CTAs; both with a ragged last warp.  Elements are independent, so the oracle runs on two slices."""
    T = 6
    pr = lqr_problem(B + n, T, B, n, m, with_f=True)
    rs = np.random.RandomState(4)
    gx, gu = rs.randn(T, B, n), rs.randn(T, B, m)
    r = run_solve(ctx, pr)
    out = run_adjoint(ctx, r, gx, gu)
    got = {k: r[k].download() for k in ("x", "u", "Ks", "ks")}
    for sl in (slice(0, 40), slice(B - 45, B)):
        ox, ou, oK, ok = olqr.lqr_solve(pr["x0"][sl], pr["C"][:, sl], pr["c"][:, sl], pr["F"][:, sl], pr["f"][:, sl], n, m)
        for a, b, k in ((got["x"], ox, "x"), (got["u"], ou, "u"), (got["Ks"], oK, "Ks"), (got["ks"], ok, "ks")):
            assert rel_err(a[:, sl], b) < 1e-10, k
        want = olqr.difflqr_backward(pr["x0"][sl], pr["C"][:, sl], pr["c"][:, sl], pr["F"][:, sl], ox, ou, gx[:, sl], gu[:, sl],
                                     n, m, quirk_dC=True, quirk_df=True)
        assert rel_err(out[0][sl], want[0]) < 1e-10, "dx0"
        for a, b, k in zip(out[1:], want[1:], ("dC", "dc", "dF", "df")):
            assert rel_err(a[:, sl], b) < 1e-10, k


def test_factor_then_rollout_split(ctx):
    """LqrRecursion.backward() then .forward(Ks, ks) as two calls == solve_recursion()."""
    pr = lqr_problem(5, 15, 40, 4, 2)
    T, B, n, m = 15, 40, 4, 2
    r = run_solve(ctx, pr)
    x2 = ctx.empty((T, B, n)); u2 = ctx.empty((T, B, m))
    ctx.lqr_solve(np.float64, T, B, n, m, r["x0"], None, None, r["F"], T - 1, r["f"], x2, u2, r["Ks"], r["ks"], None,
                  _native.LQR_ROLLOUT)
    ctx.sync()
    assert np.array_equal(x2.download(), r["x"].download())
    assert np.array_equal(u2.download(), r["u"].download())


def test_linearity_property_full_size(ctx):
    """Size-independent property at a BASELINE-sized batch (c2: n4 m2 T50 B4096): the LQR solution
    is affine in (x0, c, f): solve(a*p1 + (1-a)*p2) == a*solve(p1) + (1-a)*solve(p2) for shared C, F."""
    T, B, n, m = 50, 4096, 4, 2
    pr = lqr_problem(11, T, B, n, m)
    rs = np.random.RandomState(12)
    pr2 = dict(pr)
    pr2["x0"] = rs.randn(B, n); pr2["c"] = rs.randn(T, B, n + m); pr2["f"] = 0.1 * rs.randn(T - 1, B, n)
    a = 0.3
    pr3 = dict(pr)
    for k in ("x0", "c", "f"):
        pr3[k] = a * pr[k] + (1 - a) * pr2[k]
    r1, r2, r3 = run_solve(ctx, pr), run_solve(ctx, pr2), run_solve(ctx, pr3)
    for k in ("x", "u"):
        mix = a * r1[k].download() + (1 - a) * r2[k].download()
        assert rel_err(r3[k].download(), mix) < 1e-9


@pytest.mark.parametrize("T,B,with_f,sym", [(1, 3, True, True), (2, 6, True, True), (3, 1, False, True), (7, 9, False, False),
                                           (16, 130, True, False)])
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_dmma_warp_kernel_edge_cases(ctx, T, B, with_f, sym, dtype):
    """n=32, m=8 runs lqr_factor_dmma_warp_kernel (one warp per element, 4 per CTA): horizon edge cases, batch sizes
    that leave warps of the last CTA idle, f=None, and a NON-symmetric C (the reference never symmetrises C, and the
    kernel's operand re-use must not assume it).  float32 = the same kernel with float tensors in HBM and in the
    staging buffers (different row pitches, copy sizes and chunk counts), fp64 arithmetic."""
    n, m = 32, 8
    pr = lqr_problem(T * 31 + B, T, B, n, m, with_f=with_f, sym=sym)
    ox, ou, oK, ok = olqr.lqr_solve(pr["x0"], pr["C"], pr["c"], pr["F"], pr["f"], n, m)
    r = run_solve(ctx, pr, dtype)
    tol = TOL[dtype]
    assert rel_err(r["Ks"].download(), oK) < tol and rel_err(r["ks"].download(), ok) < tol
    assert rel_err(r["x"].download(), ox) < tol and rel_err(r["u"].download(), ou) < tol


def test_dmma_warp_kernel_fp32_is_rounded_fp64(ctx):
    """The fp32 n=32/m=8 path computes in fp64 on float inputs: on inputs that are exactly representable in float its
    gains equal the fp64 path's gains rounded to float, and the trajectory differs only by the float rounding of the stored
    K_t, k_t that the rollout re-reads."""
    T, B, n, m = 20, 37, 32, 8
    pr = lqr_problem(991, T, B, n, m, with_f=True, sym=False)
    for k in ("x0", "C", "c", "F", "f"):
        pr[k] = pr[k].astype(np.float32).astype(np.float64)
    r64 = run_solve(ctx, pr, np.float64)
    r32 = run_solve(ctx, pr, np.float32)
    K64, K32 = r64["Ks"].download(), r32["Ks"].download()
    assert K32.dtype == np.float32
    # gains: the fp64 values rounded to float (one float ulp of slack)
    assert np.allclose(K32, K64.astype(np.float32), rtol=2.4e-7, atol=1e-12)
    assert np.allclose(r32["ks"].download(), r64["ks"].download().astype(np.float32), rtol=2.4e-7, atol=1e-12)
    assert rel_err(r32["x"].download(), r64["x"].download()) < 1e-5
    assert rel_err(r32["u"].download(), r64["u"].download()) < 1e-5
