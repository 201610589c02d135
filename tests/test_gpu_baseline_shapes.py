"""GPU parity at the BASELINE.json configurations' REAL shapes (VERDICT r1, item 1): every kernel that a headline
number is quoted on is compared with the oracle at that configuration's own (n, m, T) - not only at short horizons.

  c5  n=32 m=8 T=100   lqr_factor_dmma_warp_kernel + adjoint pair + fused reduction, fp64 1e-10 and fp32 1e-4,
                       batches with a remainder modulo the 4 warps of a CTA (7, 130)
  c2  n=4 m=2 T=50 B=4096   whole batch on the GPU, oracle on a 64-element slice (elements are independent)
  c3  n=8 m=4 T=50 B=16384  box-constrained MPC step at the calibrated +-0.8 bound, oracle on a 64-element slice,
                            PNQP masks / iteration counts / line-search alphas bit-exact
  c1  pendulum n=3 m=1 T=20 B=64 exactly as env_dx/il_env.py:48-70 wires it (both couplings)
plus the fp32 instantiations of the MPC kernels (north_star: 1e-4 relative in fp32).

Reference behaviour: lqr/lqr_recursion.py:69-200, lqr/differentiable_lqr.py:78-142, mpc/mpc_step.py:70-328,
mpc/pnqp.py:37-201, util.py:201-236, env_dx/pendulum.py:65-102.  Errors are ELEMENT-relative (tests/_helpers.rel_err).
"""
import warnings

import numpy as np
import pytest

import _native
from _helpers import rel_err, rel_err_norm, lqr_problem, psd_cost, stable_dynamics
from oracle import lqr as olqr, mpc as ompc, pnqp as opnqp, pendulum as opend, boxddp as oddp

pytestmark = pytest.mark.gpu

TOL = {np.float64: 1e-10, np.float32: 1e-4}


@pytest.fixture(scope="module")
def ctx():
    return _native.default_context(0)


def _lqr_fwd_bwd(ctx, pr, gx, gu, dtype, reduced=False):
    T, B, n, m = pr["T"], pr["B"], pr["n"], pr["m"]
    s = n + m
    d = {k: ctx.to_device(pr[k], dtype) for k in ("x0", "C", "c", "F", "f")}
    o = dict(x=ctx.empty((T, B, n), dtype), u=ctx.empty((T, B, m), dtype), Ks=ctx.empty((T, B, m, n), dtype),
             ks=ctx.empty((T, B, m), dtype), fac=ctx.empty((ctx.lqr_fac_elems(T, B, n, m),), dtype))
    ctx.lqr_solve(dtype, T, B, n, m, d["x0"], d["C"], d["c"], d["F"], T - 1, d["f"], o["x"], o["u"], o["Ks"], o["ks"],
                  o["fac"], _native.LQR_FACTOR | _native.LQR_ROLLOUT | _native.LQR_SAVE_FAC)
    dgx, dgu = ctx.to_device(gx, dtype), ctx.to_device(gu, dtype)
    g = dict(dx0=ctx.empty((B, n), dtype), dC=ctx.empty((T, B, s, s), dtype), dc=ctx.empty((T, B, s), dtype),
             dF=ctx.empty((T - 1, B, n, s), dtype), df=ctx.empty((T - 1, B, n), dtype))
    ctx.lqr_adjoint(dtype, T, B, n, m, d["C"], d["c"], d["F"], o["x"], o["u"], dgx, dgu, o["Ks"], o["fac"], g["dx0"],
                    g["dC"], g["dc"], g["dF"], g["df"], _native.ADJ_STRICT_REFERENCE)
    ctx.sync()
    out = {k: v.download() for k, v in list(o.items()) + list(g.items()) if k != "fac"}
    if reduced:
        rsz = ctx.reduced_grad_elems(n, m)
        part = ctx.empty((B, rsz), dtype); sums = ctx.empty((rsz,), dtype); wsd = ctx.empty((T, B, s), dtype)
        dx0r = ctx.empty((B, n), dtype)
        ctx.lqr_adjoint_reduced(dtype, T, B, n, m, d["C"], d["c"], d["F"], o["x"], o["u"], dgx, dgu, o["Ks"], o["fac"],
                                wsd, part, dx0r, sums, _native.ADJ_STRICT_REFERENCE)
        ctx.sync()
        out["red"] = _native.Context.split_reduced(sums.download(), n, m)
        out["dx0_red"] = dx0r.download()
    return out


# ------------------------------------------------------------------------------------------------- config 5
@pytest.mark.parametrize("B", [7, 130])
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_c5_T100_vs_oracle(ctx, B, dtype):
    """n=32, m=8, T=100 (BASELINE config 5 - the shape the headline is quoted on): x, u, Ks, ks, all five adjoint
    outputs and the fused (T,B)-sums against the oracle.  This pins the DMMA warp kernel's mbarrier phases, just-in-time
    refills, pivot keys and register aliasing over the full 100-step horizon, and its dropped K^T(Qux+Quu K) terms."""
    T, n, m = 100, 32, 8
    pr = lqr_problem(500 + B, T, B, n, m, with_f=True, sym=(B == 7))
    rs = np.random.RandomState(B)
    gx, gu = rs.randn(T, B, n), rs.randn(T, B, m)
    ox, ou, oK, ok = olqr.lqr_solve(pr["x0"], pr["C"], pr["c"], pr["F"], pr["f"], n, m)
    og = olqr.difflqr_backward(pr["x0"], pr["C"], pr["c"], pr["F"], ox, ou, gx, gu, n, m)
    r = _lqr_fwd_bwd(ctx, pr, gx, gu, dtype, reduced=True)
    tol = TOL[dtype]
    errs = {"Ks": rel_err(r["Ks"], oK), "ks": rel_err(r["ks"], ok), "x": rel_err(r["x"], ox), "u": rel_err(r["u"], ou)}
    for k, w in zip(("dx0", "dC", "dc", "dF", "df"), og):
        errs[k] = rel_err(r[k], w)
    sums = (og[1].sum(axis=(0, 1)), og[2].sum(axis=(0, 1)), og[3].sum(axis=(0, 1)), og[4].sum(axis=(0, 1)))
    for k, a, w in zip(("sum_dC", "sum_dc", "sum_dF", "sum_df"), r["red"], sums):
        # a sum of T*B signed terms: normalise by the sum of magnitudes scale, i.e. tensor-wide
        errs[k] = float(np.max(np.abs(a.astype(np.float64) - w))) / float(np.max(np.abs(w)))
    errs["dx0_red"] = rel_err(r["dx0_red"], og[0])
    bad = {k: v for k, v in errs.items() if not v < tol * (10 if (dtype == np.float32 and k.startswith("sum")) else 1)}
    assert not bad, (bad, errs)


# ------------------------------------------------------------------------------------------------- config 2
def test_c2_full_batch_slice_vs_oracle(ctx):
    """n=4, m=2, T=50, B=4096 (BASELINE config 2) fwd+bwd on the GPU at the full batch; the oracle solves a strided
    64-element slice of the same inputs (batch elements are independent in LQR)."""
    T, B, n, m = 50, 4096, 4, 2
    pr = lqr_problem(2024, T, B, n, m)
    rs = np.random.RandomState(7)
    gx, gu = rs.randn(T, B, n), rs.randn(T, B, m)
    r = _lqr_fwd_bwd(ctx, pr, gx, gu, np.float64)
    sl = np.arange(5, B, 64)
    sub = lambda a: None if a is None else np.ascontiguousarray(a[:, sl])
    ox, ou, oK, ok = olqr.lqr_solve(pr["x0"][sl], sub(pr["C"]), sub(pr["c"]), sub(pr["F"]), sub(pr["f"]), n, m)
    og = olqr.difflqr_backward(pr["x0"][sl], sub(pr["C"]), sub(pr["c"]), sub(pr["F"]), ox, ou, sub(gx), sub(gu), n, m)
    assert rel_err(r["Ks"][:, sl], oK) < 1e-10 and rel_err(r["ks"][:, sl], ok) < 1e-10
    assert rel_err(r["x"][:, sl], ox) < 1e-10 and rel_err(r["u"][:, sl], ou) < 1e-10
    assert rel_err(r["dx0"][sl], og[0]) < 1e-10
    for k, w in zip(("dC", "dc", "dF", "df"), og[1:]):
        assert rel_err(r[k][:, sl], w) < 1e-10, k


# ------------------------------------------------------------------------------------------------- config 3
def _mpc_problem(seed, T, B, n, m, bound):
    rs = np.random.RandomState(seed)
    s = n + m
    A = np.eye(n) + 0.2 * rs.randn(B, n, n)
    rho = np.max(np.abs(np.linalg.eigvals(A)), axis=1)
    A *= np.minimum(1.0, 0.95 / rho)[:, None, None]
    Fb = np.concatenate((A, rs.randn(B, n, m)), axis=2)
    F = np.ascontiguousarray(np.broadcast_to(Fb[None], (T - 1, B, n, s)))
    L = 0.3 * rs.randn(B, s, s)
    C = np.ascontiguousarray(np.broadcast_to((L @ L.transpose(0, 2, 1) + np.eye(s))[None], (T, B, s, s)))
    c = rs.randn(T, B, s)
    f = 0.1 * rs.randn(T - 1, B, n)
    x0 = rs.randn(B, n)
    u = np.clip(0.2 * rs.randn(T, B, m), -bound, bound)
    lo = np.full((T, B, m), -bound); hi = np.full((T, B, m), bound)
    return dict(C=C, c=c, F=F, f=f, x0=x0, u_nom=u, lower=lo, upper=hi, n=n, m=m)


def _run_mpc(ctx, g, coupling, dtype=np.float64, dynamics=_native.DYN_LINEAR, dyn_params=None, decay=0.2):
    n, m = int(g["n"]), int(g["m"])
    T, B = g["C"].shape[:2]
    C = ctx.to_device(g["C"], dtype); c = ctx.to_device(g["c"], dtype); F = ctx.to_device(g["F"], dtype)
    f = ctx.to_device(g["f"], dtype) if g.get("f") is not None else None
    xn = ctx.to_device(g["x_nom"], dtype); un = ctx.to_device(g["u_nom"], dtype)
    lo = ctx.to_device(g["lower"], dtype); hi = ctx.to_device(g["upper"], dtype)
    o = dict(x=ctx.empty((T, B, n), dtype), u=ctx.empty((T, B, m), dtype), Ks=ctx.empty((T, B, m, n), dtype),
             ks=ctx.empty((T, B, m), dtype), u_first=ctx.empty((T, B, m), dtype), objs=ctx.empty((T, B), dtype),
             costs=ctx.empty((B,), dtype), old=ctx.empty((B,), dtype), alphas=ctx.empty((B,), dtype),
             n_qp=ctx.empty((T, B), np.int32), free=ctx.empty((T, B, m), np.uint8), n_ls=ctx.empty((B,), np.int32),
             flags=ctx.empty((B,), np.int32))
    lin = dynamics == _native.DYN_LINEAR
    ctx.mpc_step_forward(dtype, T, B, n, m, C, c, F, g["F"].shape[0], f, xn, un, lo, hi, C, c, dynamics,
                         F if lin else None, f if lin else None, dyn_params, decay, 64, True, coupling, o["x"], o["u"],
                         o["Ks"], o["ks"], o["u_first"], o["objs"], o["costs"], o["old"], o["alphas"], o["n_qp"],
                         o["free"], o["n_ls"], o["flags"])
    ctx.sync()
    return {k: v.download() for k, v in o.items()}


def test_c3_mpc_step_full_batch_slice_vs_oracle(ctx):
    """n=8, m=4, T=50, B=16384 (BASELINE config 3) at the calibrated +-0.8 bound (about 30 % of the timesteps end with
    a clamped control): one box-constrained MPC step on the whole batch, the oracle on a 64-element slice in the same
    (element) coupling.  PNQP active sets, iteration counts and line-search alphas bit-exact; values 1e-10."""
    T, B, n, m, bound = 50, 16384, 8, 4, 0.8
    g = _mpc_problem(303, T, B, n, m, bound)
    xd = ctx.empty((T, B, n))
    ctx.get_traj(np.float64, T, B, n, m, _native.DYN_LINEAR, ctx.to_device(g["x0"]), ctx.to_device(g["u_nom"]),
                 ctx.to_device(g["F"]), ctx.to_device(g["f"]), None, xd)
    ctx.sync()
    g["x_nom"] = xd.download()
    r = _run_mpc(ctx, g, _native.COUPLING_ELEMENT)
    clamped = ((r["u"] <= -bound + 1e-8) | (r["u"] >= bound - 1e-8)).any(axis=2).mean()
    assert 0.15 < clamped < 0.5, clamped
    assert not r["flags"].any()
    sl = np.arange(3, B, 256)
    sub = lambda a: np.ascontiguousarray(a[:, sl])
    x_nom_o = ompc.get_traj(g["x0"][sl], sub(g["u_nom"]), ("linear", sub(g["F"]), sub(g["f"])))
    assert rel_err(sub(g["x_nom"]), x_nom_o) < 1e-12
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ox, ou, fo, aux = ompc.step_forward(sub(g["C"]), sub(g["c"]), sub(g["F"]), sub(g["f"]), sub(g["x_nom"]),
                                            sub(g["u_nom"]), sub(g["lower"]), sub(g["upper"]), (sub(g["C"]), sub(g["c"])),
                                            ("linear", sub(g["F"]), sub(g["f"])), 0.2, 10, n, m, need_expand=True,
                                            coupling="element")
    assert np.array_equal(r["n_qp"][:, sl], aux["n_qp"])
    assert np.array_equal(r["free"][:, sl].astype(float), aux["free"])
    assert np.array_equal(r["alphas"][sl], fo.alphas)
    assert rel_err(r["Ks"][:, sl], aux["Ks"]) < 1e-10 and rel_err(r["ks"][:, sl], aux["ks"]) < 1e-10
    assert rel_err(r["x"][:, sl], ox) < 1e-10 and rel_err(r["u"][:, sl], ou) < 1e-10
    assert rel_err(r["costs"][sl], fo.costs) < 1e-10


# ------------------------------------------------------------------------------------------------- config 1
def _pendulum_c1(B=64, T=20, seed=0):
    """env_dx/il_env.py:48-70: th ~ U(-pi/2, pi/2), dth ~ U(-1, 1), x = (cos th, sin th, dth); true cost
    q = [1, 1, 0.1, 0.001], p = [-1, 0, 0, 0] (env_dx/pendulum.py:122-145); bounds +-2; u_init = 0."""
    rs = np.random.RandomState(seed)
    th = rs.uniform(-np.pi / 2, np.pi / 2, size=B)
    dth = rs.uniform(-1.0, 1.0, size=B)
    x0 = np.stack((np.cos(th), np.sin(th), dth), axis=1)
    q = np.array([1.0, 1.0, 0.1, 0.001]); p = np.array([-1.0, 0.0, 0.0, 0.0])
    C = np.ascontiguousarray(np.broadcast_to(np.diag(q)[None, None], (T, B, 4, 4)))
    c = np.ascontiguousarray(np.broadcast_to(p[None, None], (T, B, 4)))
    return x0, C, c


@pytest.mark.parametrize("coupling", ["batch", "element"])
@pytest.mark.parametrize("u_scale", [0.0, 1.5])
def test_c1_pendulum_mpc_step_vs_oracle(ctx, coupling, u_scale):
    """BASELINE config 1: pendulum n=3, m=1, T=20, B=64, one MPC step (PNQP per timestep + line search through the true
    pendulum dynamics) from u = 0 (the first BoxDDP iteration of IL_Env.mpc) and from a saturating nominal."""
    T, B = 20, 64
    x0, C, c = _pendulum_c1(B, T)
    rs = np.random.RandomState(11)
    u_nom = np.clip(u_scale * rs.randn(T, B, 1), -2.0, 2.0)
    x_nom = ompc.get_traj(x0, u_nom, ("pendulum", (10.0, 1.0, 1.0)))
    F, f = opend.linearize(x0, u_nom)
    lo = np.full((T, B, 1), -2.0); hi = np.full((T, B, 1), 2.0)
    g = dict(C=C, c=c, F=F, f=f, x_nom=x_nom, u_nom=u_nom, lower=lo, upper=hi, n=3, m=1)
    r = _run_mpc(ctx, g, _native.COUPLING_BATCH if coupling == "batch" else _native.COUPLING_ELEMENT,
                 dynamics=_native.DYN_PENDULUM, dyn_params=(10.0, 1.0, 1.0))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ox, ou, fo, aux = ompc.step_forward(C, c, F, f, x_nom, u_nom, lo, hi, (C, c), ("pendulum", (10.0, 1.0, 1.0)),
                                            0.2, 5, 3, 1, need_expand=True, coupling=coupling)
    assert np.array_equal(r["n_qp"], aux["n_qp"])
    assert np.array_equal(r["free"].astype(float), aux["free"])
    assert np.array_equal(r["alphas"], fo.alphas)
    assert rel_err(r["Ks"], aux["Ks"]) < 1e-10 and rel_err(r["ks"], aux["ks"]) < 1e-10
    assert rel_err(r["x"], ox) < 1e-10 and rel_err(r["u"], ou) < 1e-10
    assert rel_err(r["costs"], fo.costs) < 1e-10 and rel_err(r["objs"], fo.objs) < 1e-10


# ------------------------------------------------------------------------------------------------- fp32 MPC kernels
def _f32(a):
    return np.asarray(a, dtype=np.float32).astype(np.float64)


@pytest.mark.parametrize("m,B", [(1, 300), (4, 500), (8, 129)])
def test_pnqp_fp32_vs_oracle(ctx, m, B):
    """pnqp_kernel<float>: inputs exactly representable in float; elements whose fp64 oracle run is well separated from a
    decision threshold must reproduce its active set; x within 1e-4 (the algorithm's own stopping tolerance is 1e-4)."""
    rs = np.random.RandomState(200 + m)
    L = rs.randn(B, m, m)
    H = _f32(L @ L.transpose(0, 2, 1) + 0.5 * np.eye(m))
    q = _f32(3 * rs.randn(B, m)); lo = _f32(-rs.rand(B, m)); hi = _f32(rs.rand(B, m))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ox, _, ofree, oit = opnqp.pnqp(H, q, lo, hi, coupling="element")
    d = [ctx.to_device(a, np.float32) for a in (H, q, lo, hi)]
    x = ctx.empty((B, m), np.float32); LU = ctx.empty((B, m, m), np.float32); piv = ctx.empty((B, m), np.int32)
    free = ctx.empty((B, m), np.float32); it = ctx.empty((B,), np.int32); fl = ctx.empty((B,), np.int32)
    ctx.pnqp(np.float32, B, m, d[0], d[1], d[2], d[3], None, x, LU, piv, free, it, fl, 20, _native.COUPLING_ELEMENT)
    ctx.sync()
    x, free, it = x.download(), free.download(), it.download()
    # the Newton step must drop below 1e-4 (pnqp.py:139-140): on an ill-conditioned H that is below float rounding of
    # the step itself, so a few elements hit the 20-iteration cap in float arithmetic (the reference in float32 would too)
    capped = fl.download() != 0
    assert x.dtype == np.float32 and capped.mean() < 0.03, capped.mean()
    same = (free == ofree).all(axis=1) & ~capped
    assert same.mean() > 0.95, same.mean()           # float rounding may flip a decision sitting on a threshold
    # PNQP stops when |dx| < 1e-4 and returns x before that last step: 2e-4 absolute is the algorithm's own resolution
    assert np.max(np.abs(x[same] - ox[same])) < 2e-4
    # KKT at the float solution
    gvec = np.einsum("bij,bj->bi", H, x.astype(np.float64)) + q
    interior = (x > lo) & (x < hi) & ~capped[:, None]
    assert np.max(np.abs(gvec[interior])) < 5e-3


@pytest.mark.parametrize("T,B,n,m,bound", [(20, 64, 3, 1, 0.3), (50, 40, 4, 2, 0.4), (50, 37, 8, 4, 0.8)])
def test_mpc_step_forward_fp32_vs_oracle(ctx, T, B, n, m, bound):
    """mpc_forward_kernel<float> + traj_kernel<float>: float inputs, compared with the fp64 oracle on the same
    (float-representable) inputs.  Discrete decisions must agree on all but threshold-sitting elements; where they
    agree the trajectory is within 1e-4 relative."""
    g = _mpc_problem(T + n, T, B, n, m, bound)
    for k in ("C", "c", "F", "f", "x0", "u_nom", "lower", "upper"):
        g[k] = _f32(g[k])
    xd = ctx.empty((T, B, n), np.float32)
    ctx.get_traj(np.float32, T, B, n, m, _native.DYN_LINEAR, ctx.to_device(g["x0"], np.float32),
                 ctx.to_device(g["u_nom"], np.float32), ctx.to_device(g["F"], np.float32),
                 ctx.to_device(g["f"], np.float32), None, xd)
    ctx.sync()
    x_nom32 = xd.download()
    x_nom = ompc.get_traj(g["x0"], g["u_nom"], ("linear", g["F"], g["f"]))
    assert x_nom32.dtype == np.float32 and rel_err(x_nom32, x_nom) < 1e-4
    g["x_nom"] = x_nom32.astype(np.float64)
    r = _run_mpc(ctx, g, _native.COUPLING_ELEMENT, dtype=np.float32)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ox, ou, fo, aux = ompc.step_forward(g["C"], g["c"], g["F"], g["f"], g["x_nom"], g["u_nom"], g["lower"], g["upper"],
                                            (g["C"], g["c"]), ("linear", g["F"], g["f"]), 0.2, 10, n, m, need_expand=True,
                                            coupling="element")
    assert r["x"].dtype == np.float32
    same = (r["free"].astype(float) == aux["free"]).all(axis=(0, 2)) & (r["alphas"].astype(np.float64) == _f32(fo.alphas))
    assert same.mean() >= 0.9, same.mean()
    # PNQP returns k_t before its last sub-threshold step (|dx| < 1e-4, Q4): in float arithmetic WHICH iterate that is
    # differs from the fp64 run, so k_t - and through it x, u - carry up to ~1e-4 of absolute slack that no float
    # kernel can remove; 1e-3 of the trajectory scale is asserted (the costs, which are stationary in k, agree to 1e-4)
    assert rel_err_norm(r["x"][:, same], ox[:, same]) < 1e-3 and rel_err_norm(r["u"][:, same], ou[:, same]) < 1e-3
    assert rel_err_norm(r["costs"][same], fo.costs[same]) < 1e-4


def test_pendulum_traj_and_boxddp_fp32(ctx):
    """traj_kernel<float> with the pendulum + its linearisation, and the whole device-resident BoxDDP loop in fp32 on the
    il_env wiring: converges and lands on the fp64 oracle's solution to the solver's own tolerance (eps = 1e-3)."""
    T, B = 20, 64
    x0, C, c = _pendulum_c1(B, T, seed=3)
    rs = np.random.RandomState(4)
    u = _f32(np.clip(rs.randn(T, B, 1), -2, 2))
    x0 = _f32(x0)
    want = ompc.get_traj(x0, u, ("pendulum", (10.0, 1.0, 1.0)))
    wF, wf = opend.linearize(x0, u)
    x = ctx.empty((T, B, 3), np.float32); Fo = ctx.empty((T - 1, B, 3, 4), np.float32); fo = ctx.empty((T - 1, B, 3), np.float32)
    ctx.get_traj(np.float32, T, B, 3, 1, _native.DYN_PENDULUM, ctx.to_device(x0, np.float32), ctx.to_device(u, np.float32),
                 None, None, (10.0, 1.0, 1.0), x, Fo, fo)
    ctx.sync()
    assert rel_err(x.download(), want) < 1e-4
    assert rel_err(Fo.download(), wF, floor_frac=0.1) < 1e-4 and rel_err(fo.download(), wf, floor_frac=0.1) < 2e-4
    # BoxDDP fp32 (C ABI), u_init = 0, bounds +-2, eps 1e-3, decay 0.2 (env_dx/pendulum.py:58-63)
    f32 = np.float32
    lo = ctx.to_device(np.full((T, B, 1), -2.0), f32); hi = ctx.to_device(np.full((T, B, 1), 2.0), f32)
    xb = ctx.empty((T, B, 3), f32); ub = ctx.empty((T, B, 1), f32); cb = ctx.empty((B,), f32); dub = ctx.empty((B,), f32)
    dul = ctx.empty((B,), f32); Fl = ctx.empty((T - 1, B, 3, 4), f32); fl = ctx.empty((T - 1, B, 3), f32)
    n_iter, status, flags = ctx.boxddp_solve(f32, T, B, 3, 1, ctx.to_device(x0, f32), ctx.to_device(C, f32),
                                             ctx.to_device(c, f32), lo, hi, _native.DYN_PENDULUM, None, T - 1, None,
                                             (10.0, 1.0, 1.0), ctx.zeros((T, B, 1), f32), 1e-3, 1e-4, 0.2, 5, 60, 64,
                                             _native.COUPLING_BATCH, xb, ub, cb, dub, dul, Fl, fl)
    # In float arithmetic the batch-global exit max(full_du_norm) < 1e-3 (box_ddp.py:223) sits on the noise floor of
    # PNQP's own 1e-4 stopping threshold, so the loop may run to max_iter; what is asserted is where it lands.
    assert status in (_native.BOXDDP_CONVERGED, _native.BOXDDP_NOT_IMPROVED, _native.BOXDDP_MAX_ITER), status
    assert n_iter >= 10
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):
            o = oddp.box_ddp(x0, (C, c), ("pendulum", (10.0, 1.0, 1.0)), T, -2.0, 2.0, 3, 1, u_init=None, eps=1e-3,
                             not_improved_lim=5, ls_decay=0.2, max_ls_iter=5, best_cost_eps=1e-4, max_iter=500)
    # two local solvers stopped at eps = 1e-3 in different precisions: compare costs (what the solver minimises)
    cg = cb.download().astype(np.float64)
    assert np.all(np.isfinite(cg))
    assert np.median(np.abs(cg - o["costs"]) / np.maximum(1.0, np.abs(o["costs"]))) < 1e-3
    assert np.max(np.abs(ub.download())) <= 2.0 + 1e-6
