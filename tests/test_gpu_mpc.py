"""GPU parity: PNQP, MPC step forward/backward, LQR_active and trajectory kernels (through the C ABI)
vs the oracle and the golden fixtures produced from the unmodified reference
(mpc/pnqp.py, mpc/mpc_step.py, mpc/active_constrained_lqr.py, util.get_traj, env_dx/pendulum.py).

fp64: values within 1e-10 relative (fixtures use the fp64-clean LU shim, SURVEY.md H1);
active-set masks, iteration counts and line-search step selections bit-exact.
"""
import warnings

import numpy as np
import pytest

import _native
from _helpers import load_golden, rel_err, psd_cost, stable_dynamics
from oracle import pnqp as opnqp, mpc as ompc, pendulum as opend

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    return _native.default_context(0)


# ------------------------------------------------------------------------------------------- PNQP
def run_pnqp(ctx, H, q, lo, hi, xi=None, coupling=_native.COUPLING_ELEMENT, dtype=np.float64):
    B, m = q.shape
    d = [ctx.to_device(a, dtype) for a in (H, q, lo, hi)]
    dxi = None if xi is None else ctx.to_device(xi, dtype)
    x = ctx.empty((B, m), dtype); LU = ctx.empty((B, m, m), dtype); piv = ctx.empty((B, m), np.int32)
    free = ctx.empty((B, m), dtype); it = ctx.empty((B,), np.int32); fl = ctx.empty((B,), np.int32)
    ctx.pnqp(dtype, B, m, d[0], d[1], d[2], d[3], dxi, x, LU, piv, free, it, fl, 20, coupling)
    ctx.sync()
    return x.download(), LU.download(), piv.download(), free.download(), it.download(), fl.download()


PNQP_CASES = ["pnqp_kat", "pnqp_d4", "pnqp_d4_warm", "pnqp_d1", "pnqp_d8_loose", "pnqp_d3"]


@pytest.mark.parametrize("name", PNQP_CASES)
def test_pnqp_element_golden(ctx, name):
    g = load_golden(name)
    x, LU, piv, free, it, fl = run_pnqp(ctx, g["H"], g["q"], g["lower"], g["upper"], g.get("x_init"))
    assert rel_err(x, g["x_elem"]) < 1e-10
    assert np.array_equal(free, g["free_elem"])          # active-set masks bit-exact
    assert np.array_equal(it, g["it_elem"])
    assert not fl.any()
    if "kat" in g:   # experiment_mpc/Projected_Newton_Quadratic_Programming.py:67-68 (4 printed digits)
        assert np.allclose(x, g["kat"], atol=5e-5)


@pytest.mark.parametrize("name", PNQP_CASES)
def test_pnqp_batch_golden(ctx, name):
    g = load_golden(name)
    x, LU, piv, free, it, fl = run_pnqp(ctx, g["H"], g["q"], g["lower"], g["upper"], g.get("x_init"),
                                        coupling=_native.COUPLING_BATCH)
    assert rel_err(x, g["x"]) < 1e-10
    assert np.array_equal(free, g["free"])
    assert (it == int(g["it"])).all()
    if g["H"].shape[1] > 1:
        assert rel_err(LU, g["LU"]) < 1e-10 and np.array_equal(piv, g["piv"])
    else:
        assert rel_err(LU, g["Hf"]) < 1e-10


@pytest.mark.parametrize("m,B", [(1, 300), (2, 257), (4, 1000), (6, 64), (8, 129), (12, 33), (20, 40), (32, 17)])
def test_pnqp_random_vs_oracle(ctx, m, B):
    rs = np.random.RandomState(100 + m)
    L = rs.randn(B, m, m)
    H = L @ L.transpose(0, 2, 1) + 0.5 * np.eye(m)
    q = 3 * rs.randn(B, m)
    lo = -rs.rand(B, m); hi = rs.rand(B, m)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ox, _, ofree, oit = opnqp.pnqp(H, q, lo, hi, coupling="element")
    x, LU, piv, free, it, fl = run_pnqp(ctx, H, q, lo, hi)
    assert np.array_equal(free, ofree)
    assert np.array_equal(it, oit)
    assert rel_err(x, ox) < 1e-10
    # KKT property (size-independent): projected gradient vanishes at the solution
    gvec = np.einsum("bij,bj->bi", H, x) + q
    interior = (x > lo) & (x < hi)
    assert np.max(np.abs(gvec[interior])) < 1e-3
    assert (gvec[x == lo] >= -1e-3).all() and (gvec[x == hi] <= 1e-3).all()


# ------------------------------------------------------------------------------------------- MPC step
def mpc_inputs_from_golden(g):
    n, m = int(g["n"]), int(g["m"])
    T, B = g["C"].shape[:2]
    return T, B, n, m


def run_mpc_forward(ctx, g, coupling, dtype=np.float64, dynamics=_native.DYN_LINEAR, dyn_params=None):
    T, B, n, m = mpc_inputs_from_golden(g)
    s = n + m
    C = ctx.to_device(g["C"], dtype); c = ctx.to_device(g["c"], dtype); F = ctx.to_device(g["F"], dtype)
    f = ctx.to_device(g["f"], dtype) if "f" in g else None
    xn = ctx.to_device(g["x_nom"], dtype); un = ctx.to_device(g["u_nom"], dtype)
    lo = ctx.to_device(g["lower"], dtype); hi = ctx.to_device(g["upper"], dtype)
    o = dict(x=ctx.empty((T, B, n), dtype), u=ctx.empty((T, B, m), dtype), Ks=ctx.empty((T, B, m, n), dtype),
             ks=ctx.empty((T, B, m), dtype), u_first=ctx.empty((T, B, m), dtype), objs=ctx.empty((T, B), dtype),
             costs=ctx.empty((B,), dtype), old=ctx.empty((B,), dtype), alphas=ctx.empty((B,), dtype),
             n_qp=ctx.empty((T, B), np.int32), free=ctx.empty((T, B, m), np.uint8), n_ls=ctx.empty((B,), np.int32),
             flags=ctx.empty((B,), np.int32))
    ctx.mpc_step_forward(dtype, T, B, n, m, C, c, F, g["F"].shape[0], f, xn, un, lo, hi, C, c, dynamics, F, f,
                         dyn_params, 0.2, 64, True, coupling, o["x"], o["u"], o["Ks"], o["ks"], o["u_first"],
                         o["objs"], o["costs"], o["old"], o["alphas"], o["n_qp"], o["free"], o["n_ls"], o["flags"])
    ctx.sync()
    return {k: v.download() for k, v in o.items()}, dict(C=C, c=c, F=F, f=f, lo=lo, hi=hi)


MPC_CASES = ["mpc_n3m2", "mpc_n3m1", "mpc_n8m4", "mpc_n4m2_loose"]


@pytest.mark.parametrize("name", MPC_CASES)
@pytest.mark.parametrize("coupling", ["element", "batch"])
def test_mpc_step_forward_golden(ctx, name, coupling):
    g = load_golden(name + "_" + coupling)
    T, B, n, m = mpc_inputs_from_golden(g)
    r, _ = run_mpc_forward(ctx, g, _native.COUPLING_BATCH if coupling == "batch" else _native.COUPLING_ELEMENT)
    assert np.array_equal(r["free"].astype(float), g["free"])       # active sets bit-exact
    assert np.array_equal(r["alphas"], g["alphas"])                  # line-search step selection bit-exact
    assert rel_err(r["Ks"], g["Ks"]) < 1e-10 and rel_err(r["ks"], g["ks"]) < 1e-10
    assert rel_err(r["x"], g["x"]) < 1e-10 and rel_err(r["u"], g["u"]) < 1e-10
    assert rel_err(r["costs"], g["costs"]) < 1e-10 and rel_err(r["objs"], g["objs"]) < 1e-10
    assert not r["flags"].any()
    if coupling == "batch":
        assert int(r["n_qp"].max(axis=1).sum()) == int(g["n_total_qp_iter"])
        du = g["u_nom"] - r["u_first"]     # mpc_step.py:261-263 scrambled norm, done by the facade
        full = np.sqrt(np.sum(np.transpose(du, (0, 2, 1)).reshape(B, T * m) ** 2, axis=1))
        assert rel_err(full, g["full_du_norm"]) < 1e-10
    else:
        assert np.array_equal(r["n_qp"].sum(axis=0), g["n_total_qp_iter_elem"])


@pytest.mark.parametrize("name", MPC_CASES)
def test_mpc_step_backward_golden(ctx, name):
    g = load_golden(name + "_batch")
    T, B, n, m = mpc_inputs_from_golden(g)
    s = n + m
    dt = np.float64
    C = ctx.to_device(g["C"]); c = ctx.to_device(g["c"]); F = ctx.to_device(g["F"])
    x = ctx.to_device(g["x"]); u = ctx.to_device(g["u"]); lo = ctx.to_device(g["lower"]); hi = ctx.to_device(g["upper"])
    gx = ctx.to_device(g["gx"]); gu = ctx.to_device(g["gu"])
    FT = g["F"].shape[0]
    wsK = ctx.empty((T, B, m, n)); wsk = ctx.empty((T, B, m)); wsd = ctx.empty((T, B, s)); act = ctx.empty((T, B, m), np.uint8)
    dx0 = ctx.empty((B, n)); dC = ctx.empty((T, B, s, s)); dc = ctx.empty((T, B, s)); dF = ctx.empty((FT, B, n, s))
    df = ctx.empty((T - 1, B, n)) if "df" in g else None
    ctx.mpc_step_backward(dt, T, B, n, m, C, c, F, FT, x, u, lo, hi, gx, gu, wsK, wsk, wsd, act, dx0, dC, dc, dF, df)
    ctx.sync()
    assert rel_err(dx0.download(), g["dx0"]) < 1e-10
    assert rel_err(dC.download(), g["dC"]) < 1e-10
    assert rel_err(dc.download(), g["dc"]) < 1e-10
    assert rel_err(dF.download(), g["dF"]) < 1e-10
    if df is not None:
        assert rel_err(df.download(), g["df"]) < 1e-10
    want_act = (np.abs(g["u"] - g["lower"]) <= 1e-8) | (np.abs(g["u"] - g["upper"]) <= 1e-8)
    assert np.array_equal(act.download().astype(bool), want_act)


@pytest.mark.parametrize("T,B,n,m,bound", [(20, 64, 3, 1, 0.3), (50, 40, 4, 2, 0.4), (50, 37, 8, 4, 0.3),
                                            (12, 9, 5, 3, 0.5), (8, 3, 10, 5, 0.4), (10, 2, 32, 8, 0.5)])
def test_mpc_step_forward_random_vs_oracle(ctx, T, B, n, m, bound):
    rs = np.random.RandomState(T + B + n)
    s = n + m
    C, c = psd_cost(rs, T, B, s)
    F = stable_dynamics(rs, T, B, n, m, per_t=False)
    f = 0.1 * rs.randn(T - 1, B, n)
    x0 = rs.randn(B, n)
    u_nom = np.clip(0.2 * rs.randn(T, B, m), -bound, bound)
    lo = np.full((T, B, m), -bound); hi = np.full((T, B, m), bound)
    x_nom = ompc.get_traj(x0, u_nom, ("linear", F, f))
    g = dict(C=C, c=c, F=F, f=f, x_nom=x_nom, u_nom=u_nom, lower=lo, upper=hi, n=n, m=m)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ox, ou, fo, aux = ompc.step_forward(C, c, F, f, x_nom, u_nom, lo, hi, (C, c), ("linear", F, f), 0.2, 10, n, m,
                                            need_expand=True, coupling="element")
    r, _ = run_mpc_forward(ctx, g, _native.COUPLING_ELEMENT)
    # elements whose PNQP iteration counts agree are non-degenerate: demand bit-exact discrete decisions there
    same = np.array_equal(r["n_qp"], aux["n_qp"])
    assert same, "PNQP iteration counts differ"
    assert np.array_equal(r["free"].astype(float), aux["free"])
    assert np.array_equal(r["alphas"], fo.alphas)
    assert rel_err(r["x"], ox) < 1e-9 and rel_err(r["u"], ou) < 1e-9
    assert rel_err(r["costs"], fo.costs) < 1e-10


@pytest.mark.parametrize("T,B,n,m", [(12, 21, 6, 3), (16, 70, 4, 2), (20, 35, 3, 1), (9, 5, 2, 1)])
def test_lqr_active_vs_oracle(ctx, T, B, n, m):
    """(6,3): group kernel; (4,2), (3,1), (2,1): thread-per-element kernel (lqr_tpe_kernel.cuh), masked rows included."""
    rs = np.random.RandomState(5)
    C, c = psd_cost(rs, T, B, n + m)
    F = stable_dynamics(rs, T, B, n, m)
    x0 = rs.randn(B, n)
    active = rs.rand(T, B, m) < 0.4
    ox, ou = ompc.lqr_active(x0, C, c, F, None, active, n, m)
    d = [ctx.to_device(a) for a in (x0, C, c, F)]
    da = ctx.to_device(active.astype(np.uint8))
    x = ctx.empty((T, B, n)); u = ctx.empty((T, B, m)); Ks = ctx.empty((T, B, m, n)); ks = ctx.empty((T, B, m))
    ctx.lqr_active_solve(np.float64, T, B, n, m, d[0], d[1], d[2], d[3], T - 1, None, da, x, u, Ks, ks)
    ctx.sync()
    assert rel_err(x.download(), ox) < 1e-10 and rel_err(u.download(), ou) < 1e-10
    assert (u.download()[active] == 0).all()


# ------------------------------------------------------------------------------------------- trajectories
def test_get_traj_linear_and_pendulum(ctx):
    rs = np.random.RandomState(9)
    T, B, n, m = 15, 70, 5, 2
    F = stable_dynamics(rs, T, B, n, m); f = 0.1 * rs.randn(T - 1, B, n)
    x0 = rs.randn(B, n); u = rs.randn(T, B, m)
    want = ompc.get_traj(x0, u, ("linear", F, f))
    x = ctx.empty((T, B, n))
    ctx.get_traj(np.float64, T, B, n, m, _native.DYN_LINEAR, ctx.to_device(x0), ctx.to_device(u), ctx.to_device(F),
                 ctx.to_device(f), None, x)
    ctx.sync()
    assert rel_err(x.download(), want) < 1e-12
    # pendulum (env_dx/pendulum.py:65-102) + analytic linearisation: the reference's parameters, (g, m, l, dt,
    # max_torque) none at its default (the controls reach 7: the torque clip at 1.5 and at 2.0 are both active), and
    # dt <= 0 / max_torque <= 0, which mean the defaults 0.05 / 2.0
    g = load_golden("pendulum_step")
    B = g["x"].shape[0]
    T = 6
    u = np.repeat(g["u"][None], T, axis=0) * np.linspace(0.2, 1.0, T)[:, None, None]
    assert ((np.abs(u) > 1.5) & (np.abs(u) < 2.0)).any()
    for dev, par, dt, maxu in (((10.0, 1.0, 1.0), (10.0, 1.0, 1.0), 0.05, 2.0),
                               ((9.5, 1.3, 0.8, 0.03, 1.5), (9.5, 1.3, 0.8), 0.03, 1.5),
                               ((9.5, 1.3, 0.8, 0.0, -1.0), (9.5, 1.3, 0.8), 0.05, 2.0)):
        want = ompc.get_traj(g["x"], u, ("pendulum", par, dt, maxu))
        wF, wf = opend.linearize(g["x"], u, par, dt, maxu)
        x = ctx.empty((T, B, 3)); Fo = ctx.empty((T - 1, B, 3, 4)); fo = ctx.empty((T - 1, B, 3))
        ctx.get_traj(np.float64, T, B, 3, 1, _native.DYN_PENDULUM, ctx.to_device(g["x"]), ctx.to_device(u), None, None,
                     dev, x, Fo, fo)
        ctx.sync()
        assert rel_err(x.download()[1], want[1]) < 1e-13, dev
        assert rel_err(x.download(), want) < 1e-12, dev
        assert rel_err(Fo.download(), wF) < 1e-12 and rel_err(fo.download(), wf) < 1e-11, dev


def test_bad_bounds_are_reported_through_the_c_abi(ctx):
    """lower > upper: the reference asserts (pnqp.py:64, mpc_step.py:139).  The stream-ordered C-ABI calls flag the
    element (DMPC_FLAG_BAD_BOUNDS in d_flags); dmpc_boxddp_solve, which reads its loop record anyway, returns
    DMPC_ERR_BAD_BOUNDS (surfaced as AssertionError by the ctypes layer, like the reference)."""
    rs = np.random.RandomState(3)
    B, m = 9, 3
    L = rs.randn(B, m, m)
    H = L @ L.transpose(0, 2, 1) + np.eye(m)
    q = rs.randn(B, m); lo = -np.ones((B, m)); hi = np.ones((B, m))
    lo[4, 1], hi[4, 1] = 0.5, -0.5
    *_, fl = run_pnqp(ctx, H, q, lo, hi)
    assert (fl[4] & _native.FLAG_BAD_BOUNDS) and not (np.delete(fl, 4) & _native.FLAG_BAD_BOUNDS).any()
    # MPC step (group kernel, n=4 m=2) and the thread-per-element kernel (n=3 m=1)
    for n, m in ((4, 2), (3, 1)):
        T, B = 6, 10
        s = n + m
        C, c = psd_cost(rs, T, B, s)
        F = stable_dynamics(rs, T, B, n, m, per_t=False)
        u = np.zeros((T, B, m)); x0 = rs.randn(B, n)
        lo = np.full((T, B, m), -0.5); hi = np.full((T, B, m), 0.5)
        lo[2, 7, 0], hi[2, 7, 0] = 0.3, -0.3
        g = dict(C=C, c=c, F=F, f=None, x_nom=ompc.get_traj(x0, u, ("linear", F, None)), u_nom=u, lower=lo, upper=hi, n=n, m=m)
        g.pop("f")
        r, d = run_mpc_forward(ctx, g, _native.COUPLING_ELEMENT)
        assert r["flags"][7] & _native.FLAG_BAD_BOUNDS and not (np.delete(r["flags"], 7) & _native.FLAG_BAD_BOUNDS).any()
    # BoxDDP: status code
    T, B, n, m = 6, 10, 3, 1
    dlo, dhi = ctx.to_device(lo), ctx.to_device(hi)
    o = [ctx.empty((T, B, n)), ctx.empty((T, B, m)), ctx.empty((B,)), ctx.empty((B,)), ctx.empty((B,))]
    with pytest.raises(AssertionError):
        ctx.boxddp_solve(np.float64, T, B, n, m, ctx.to_device(x0), ctx.to_device(C), ctx.to_device(c), dlo, dhi,
                         _native.DYN_LINEAR, ctx.to_device(F), T - 1, None, None, ctx.zeros((T, B, m)), 1e-6, 1e-4, 0.2, 5, 5, 64,
                         _native.COUPLING_ELEMENT, *o)


@pytest.mark.parametrize("n,m,B,T", [(8, 4, 100, 20), (4, 2, 700, 12), (3, 2, 300, 10), (3, 1, 2000, 20), (3, 1, 700, 20)])
def test_batch_coupling_across_a_cluster(ctx, n, m, B, T):
    """coupling = BATCH with more elements than one CTA holds: the batch is spread over the CTAs of one thread-block
    cluster and PNQP's batch-global decisions (pnqp.py:139-144, 172-187) are OR-reduced through distributed shared memory
    (csrc/common.cuh batch_or).  Against the oracle in the same (whole-batch) coupling: PNQP iteration counts, active sets
    and line-search alphas bit-exact, values 1e-10."""
    rs = np.random.RandomState(B + n)
    s = n + m
    bound = 0.4
    C, c = psd_cost(rs, T, B, s)
    F = stable_dynamics(rs, T, B, n, m, per_t=False)
    f = 0.1 * rs.randn(T - 1, B, n)
    x0 = rs.randn(B, n)
    u_nom = np.clip(0.2 * rs.randn(T, B, m), -bound, bound)
    lo = np.full((T, B, m), -bound); hi = np.full((T, B, m), bound)
    x_nom = ompc.get_traj(x0, u_nom, ("linear", F, f))
    g = dict(C=C, c=c, F=F, f=f, x_nom=x_nom, u_nom=u_nom, lower=lo, upper=hi, n=n, m=m)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ox, ou, fo, aux = ompc.step_forward(C, c, F, f, x_nom, u_nom, lo, hi, (C, c), ("linear", F, f), 0.2, 10, n, m,
                                            need_expand=True, coupling="batch")
    r, _ = run_mpc_forward(ctx, g, _native.COUPLING_BATCH)
    assert np.array_equal(r["n_qp"], aux["n_qp"])
    assert np.array_equal(r["free"].astype(float), aux["free"])
    assert np.array_equal(r["alphas"], fo.alphas)
    assert rel_err(r["Ks"], aux["Ks"]) < 1e-10 and rel_err(r["ks"], aux["ks"]) < 1e-10
    assert rel_err(r["x"], ox) < 1e-10 and rel_err(r["u"], ou) < 1e-10
    assert rel_err(r["costs"], fo.costs) < 1e-10
    assert not r["flags"].any()


def test_pnqp_batch_coupling_across_a_cluster(ctx):
    rs = np.random.RandomState(77)
    B, m = 2000, 4                      # 2000 x 4 lanes: ~14 CTAs of one cluster (112 registers -> 576 threads per CTA)
    L = rs.randn(B, m, m)
    H = L @ L.transpose(0, 2, 1) + 0.5 * np.eye(m)
    q = 3 * rs.randn(B, m); lo = -rs.rand(B, m); hi = rs.rand(B, m)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ox, _, ofree, oit = opnqp.pnqp(H, q, lo, hi, coupling="batch")
    x, LU, piv, free, it, fl = run_pnqp(ctx, H, q, lo, hi, coupling=_native.COUPLING_BATCH)
    assert np.array_equal(free, ofree) and (it == int(oit)).all()
    assert rel_err(x, ox) < 1e-10
