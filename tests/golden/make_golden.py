#!/usr/bin/env python
"""Generate tests/golden/*.npz from the UNMODIFIED reference and pin the oracle to it.

Needs a checkout of the original chainer-differentiable-mpc:
    DIFFMPC_REFERENCE=<checkout> python tests/golden/make_golden.py

For every case the reference modules (imported unmodified under
tests/_chainer_stub, see _ref_loader.py) and the numpy oracle (oracle/) are run
on the same seeded inputs; the script asserts that they agree (bit-for-bit up
to BLAS summation order, tolerance 1e-12 relative) and stores inputs + reference
outputs as fixtures.  Cases whose name ends in `_fp32lu` use the literal
reference (float32 torch.lu_solve, util.py:522-526); all others use the
fp64-clean shim (SURVEY.md H1) that the 1e-10 parity target is defined against.
"""
import os
import sys
import types
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
import _ref_loader  # noqa: E402

warnings.filterwarnings("ignore")


def close(a, b, tol=1e-12, what=""):
    a = np.asarray(a, dtype=float)
    b = np.asarray(b, dtype=float)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    if a.size == 0:
        return
    scale = max(1.0, float(np.max(np.abs(b))))
    err = float(np.max(np.abs(a - b))) / scale
    assert err <= tol, "%s: oracle vs reference rel err %.3e > %.1e" % (what, err, tol)


def stable_dynamics(rs, B, n, m, T, rho=0.95, per_t=False):
    A = np.eye(n) + 0.2 * rs.randn(B, n, n)
    for b in range(B):
        r = np.max(np.abs(np.linalg.eigvals(A[b])))
        if r > rho:
            A[b] *= rho / r
    Bm = rs.randn(B, n, m)
    F = np.concatenate((A, Bm), axis=2)
    F = np.repeat(F[None], T - 1, axis=0).copy()
    if per_t:
        F += 0.01 * rs.randn(*F.shape)
    return F


def psd_cost(rs, T, B, s, sym=True):
    L = rs.randn(T, B, s, s) * 0.3
    C = L @ np.transpose(L, (0, 1, 3, 2)) + np.eye(s)
    if not sym:
        C = C + 0.05 * rs.randn(T, B, s, s)
    c = rs.randn(T, B, s)
    return C, c


def main(lu_modes=(False, True)):
    out = {}
    _ref_loader.load(lu_fp32=False)
    import chainer
    V = chainer.Variable
    from oracle import lqr as olqr, pnqp as opnqp, mpc as ompc, boxddp as obox, pendulum as opend

    # ------------------------------------------------------------ LQR goldens
    mods = _ref_loader.load(lu_fp32=False)
    LqrRecursion = mods["lqr_recursion"].LqrRecursion
    DiffLqr = mods["differentiable_lqr"].DiffLqr

    def ref_lqr(x0, C, c, F, f, T, n, m):
        r = LqrRecursion(V(x0), V(C), V(c), V(F), None if f is None else V(f), T, n, m)
        Ks, ks = r.backward()
        x, u = r.forward(Ks, ks)
        return x.array, u.array, np.stack([k.array for k in Ks]), np.stack([k.array for k in ks])

    # Boyd EE363 example (examples/Boyd_lqr.py:24-37)
    T, n, m = 51, 3, 1
    F = np.repeat(np.array([[1.0, 0, 0, 1], [1, 1.0, 0, 0], [0, 1, 1, 0]])[None, None], T, axis=0)
    c = np.zeros((T, 1, 4))
    C = np.repeat(np.diag([0, 0, 1.0, 1.0])[None, None], T, axis=0)
    C[T - 1, 0, 3, 3] = 1e-14
    x0 = np.array([[0.5428, 0.7633, 0.3504]])
    x, u, Ks, ks = ref_lqr(x0, C, c, F, None, T, n, m)
    ox, ou, oK, ok_ = olqr.lqr_solve(x0, C, c, F, None, n, m)
    close(ox, x, what="boyd x"); close(ou, u, what="boyd u"); close(oK, Ks, what="boyd K")
    # printed digits of examples/Boyd_lqr.ipynb:508-558, 668-768
    assert np.allclose(Ks[0, 0, 0], [-1.86152282, -1.34921019, -0.35888729], atol=5e-9)
    assert np.allclose(Ks[47, 0, 0], [-1.5, -1.5, -0.5], atol=5e-9)
    out["boyd"] = dict(x0=x0, C=C, c=c, F=F, x=x, u=u, Ks=Ks, ks=ks, n=n, m=m)

    # one-variable example (examples/LQR_recursion_solver_one_variable.py:24-32)
    T, n, m = 20, 2, 1
    F = np.repeat(np.array([[1.0, 1.0, 0], [0, 1.0, 1.0]])[None, None], T, axis=0)
    c = np.zeros((T, 1, 3))
    C = np.repeat(np.diag([1.0, 0, 10])[None, None], T, axis=0)
    x0 = np.array([[1.0, 0.0]])
    x, u, Ks, ks = ref_lqr(x0, C, c, F, None, T, n, m)
    ox, ou, oK, ok_ = olqr.lqr_solve(x0, C, c, F, None, n, m)
    close(ox, x, what="onevar x"); close(oK, Ks, what="onevar K")
    out["onevar"] = dict(x0=x0, C=C, c=c, F=F, x=x, u=u, Ks=Ks, ks=ks, n=n, m=m)

    # random multi-input LQR (F.batch_inv branch), with and without f, non-symmetric C (Q10)
    for name, (T, B, n, m, with_f, sym) in {
        "lqr_n4m2": (12, 5, 4, 2, True, True),
        "lqr_n4m2_nof": (12, 5, 4, 2, False, True),
        "lqr_n3m1_f": (7, 4, 3, 1, True, True),
        "lqr_n5m3_nonsym": (9, 3, 5, 3, True, False),
        "lqr_n8m4": (10, 3, 8, 4, True, True),
        "lqr_T1": (1, 3, 3, 2, False, True),
    }.items():
        rs = np.random.RandomState(abs(hash(name)) % 2 ** 31 if False else sum(map(ord, name)))
        s = n + m
        C, c = psd_cost(rs, T, B, s, sym)
        F = stable_dynamics(rs, B, n, m, max(T, 2), per_t=True)[:T - 1] if T > 1 else np.zeros((0, B, n, s))
        f = 0.1 * rs.randn(max(T - 1, 0), B, n) if with_f else None
        x0 = rs.randn(B, n)
        x, u, Ks, ks = ref_lqr(x0, C, c, F, f, T, n, m)
        ox, ou, oK, ok_ = olqr.lqr_solve(x0, C, c, F, f, n, m)
        close(ox, x, what=name + " x"); close(ou, u, what=name + " u")
        close(oK, Ks, what=name + " K"); close(ok_, ks, what=name + " k")
        d = dict(x0=x0, C=C, c=c, F=F, x=x, u=u, Ks=Ks, ks=ks, n=n, m=m)
        if f is not None:
            d["f"] = f
        # DiffLqr.backward on the same problem
        if T > 1:
            gx = rs.randn(T, B, n)
            gu = rs.randn(T, B, m)
            node = DiffLqr(T, B, n, m)
            node.apply((x0, C, c, F, f))
            g = node.backward((0, 1, 2, 3, 4), (V(gx), V(gu)))
            g = [np.asarray(v.array) for v in g]
            og = olqr.difflqr_backward(x0, C, c, F, x, u, gx, gu, n, m)
            for a, b, nm in zip(og, g, ("dx0", "dC", "dc", "dF", "df")):
                close(a, b, what=name + " " + nm)
            d.update(gx=gx, gu=gu, dx0=g[0], dC=g[1], dc=g[2], dF=g[3], df=g[4])
        out[name] = d

    # ------------------------------------------------------------ PNQP
    H = np.array([[[7.9325, 4.9520, 1.0314, 0.2282], [4.9520, 8.7746, 1.7916, 3.3622],
                   [1.0314, 1.7916, 4.2824, -2.5979], [0.2282, 3.3622, -2.5979, 6.7064]],
                  [[3.4423, -1.9137, -0.9978, -4.4905], [-1.9137, 6.7254, 3.3720, 1.7444],
                   [-0.9978, 3.3720, 3.5695, -0.9766], [-4.4905, 1.7444, -0.9766, 13.0806]]])
    q = np.array([[-0.8277, 8.5116, -12.1597, 17.9497], [-3.5764, -5.3455, -3.2465, 4.3960]])
    lo = np.array([[-0.2843, -0.0063, -0.1808, -0.6669], [-0.1359, -0.3629, -0.2125, -0.0121]])
    hi = np.array([[0.1345, 0.0307, 0.0277, 0.9418], [0.6205, 0.2703, 0.4023, 0.2560]])
    kat = np.array([[0.1239, -0.0063, 0.0277, -0.6669], [0.6205, 0.2703, 0.4023, -0.0121]])

    def rand_qp(rs, B, d, scale=1.0):
        L = rs.randn(B, d, d)
        H = L @ np.transpose(L, (0, 2, 1)) + 0.5 * np.eye(d)
        q = 3.0 * rs.randn(B, d)
        lo = -scale * rs.rand(B, d)
        hi = scale * rs.rand(B, d)
        return H, q, lo, hi

    for fp32 in lu_modes:
        mods = _ref_loader.load(lu_fp32=fp32)
        PNQP = mods["pnqp"].PNQP
        sfx = "_fp32lu" if fp32 else ""
        cases = {"pnqp_kat": (H, q, lo, hi, None)}
        rs = np.random.RandomState(7)
        cases["pnqp_d4"] = rand_qp(rs, 16, 4) + (None,)
        cases["pnqp_d4_warm"] = rand_qp(rs, 16, 4) + (0.3 * rs.randn(16, 4),)
        cases["pnqp_d1"] = rand_qp(rs, 16, 1) + (None,)
        cases["pnqp_d8_loose"] = rand_qp(rs, 8, 8, scale=5.0) + (None,)
        cases["pnqp_d3"] = rand_qp(rs, 11, 3, scale=0.7) + (None,)
        for name, (H_, q_, lo_, hi_, xi) in cases.items():
            rx, rfac, rfree, ri = PNQP(V(H_), V(q_), V(lo_), V(hi_), x_init=xi)
            ox, ofac, ofree, oi = opnqp.pnqp(H_, q_, lo_, hi_, x_init=xi, lu_fp32=fp32, coupling="batch")
            close(ox, rx, tol=1e-12 if not fp32 else 1e-6, what=name + sfx + " x")
            assert np.array_equal(ofree, rfree), name
            assert oi == ri, (name, oi, ri)
            d = dict(H=H_, q=q_, lower=lo_, upper=hi_, x=rx, free=rfree, it=ri)
            if xi is not None:
                d["x_init"] = xi
            if H_.shape[1] == 1:
                d["Hf"] = rfac
                close(ofac, rfac, what=name + " Hf")
            else:
                d["LU"], d["piv"] = rfac
                close(ofac[0], rfac[0], tol=1e-12, what=name + " LU")
                assert np.array_equal(ofac[1], rfac[1])
            # per-element coupling == reference at n_batch 1
            ex = []
            for b in range(H_.shape[0]):
                sl = slice(b, b + 1)
                r1 = PNQP(V(H_[sl]), V(q_[sl]), V(lo_[sl]), V(hi_[sl]),
                          x_init=None if xi is None else xi[sl])
                ex.append((r1[0], r1[2], r1[3]))
            d["x_elem"] = np.concatenate([e[0] for e in ex])
            d["free_elem"] = np.concatenate([e[1] for e in ex])
            d["it_elem"] = np.array([e[2] for e in ex])
            oe = opnqp.pnqp(H_, q_, lo_, hi_, x_init=xi, lu_fp32=fp32, coupling="element")
            close(oe[0], d["x_elem"], tol=1e-12 if not fp32 else 1e-6, what=name + " elem x")
            assert np.array_equal(oe[2], d["free_elem"]) and np.array_equal(oe[3], d["it_elem"])
            out[name + sfx] = d
        if not fp32:
            assert np.allclose(out["pnqp_kat"]["x"], kat, atol=5e-5)   # 4 printed digits
            out["pnqp_kat"]["kat"] = kat

    # ------------------------------------------------------------ MPC step fwd/bwd, BoxDDP (LinDx)
    for fp32 in lu_modes:
        mods = _ref_loader.load(lu_fp32=fp32)
        util = mods["util"]
        MPCstep = mods["mpc_step"].MPCstep
        BoxDDP = mods["box_ddp"].BoxDDP
        sfx = "_fp32lu" if fp32 else ""
        tol = 1e-11 if not fp32 else 2e-5
        for name, (T, B, n, m, bound, with_f) in {
            "mpc_n3m2": (6, 4, 3, 2, 0.4, True),
            "mpc_n3m1": (8, 5, 3, 1, 0.3, False),
            "mpc_n8m4": (10, 3, 8, 4, 0.35, True),
            "mpc_n4m2_loose": (7, 4, 4, 2, 50.0, True),
        }.items():
            rs = np.random.RandomState(sum(map(ord, name)))
            s = n + m
            C, c = psd_cost(rs, T, B, s)
            F = stable_dynamics(rs, B, n, m, T)
            f = 0.1 * rs.randn(T - 1, B, n) if with_f else None
            x0 = rs.randn(B, n)
            u_nom = np.clip(0.2 * rs.randn(T, B, m), -bound, bound)
            lo = np.full((T, B, m), -bound)
            hi = np.full((T, B, m), bound)
            dyn = ("linear", F, f)
            x_nom = ompc.get_traj(x0, u_nom, dyn)
            for coupling in ("batch", "element"):
                def run_ref(sl):
                    fs = None if f is None else f[:, sl]
                    st = MPCstep(controls=u_nom[:, sl], T=T, u_upper=hi[:, sl], u_lower=lo[:, sl],
                                 n_batch=x0[sl].shape[0], n_state=n, n_ctrl=m,
                                 current_states=x_nom[:, sl],
                                 true_cost=util.QuadCost(C[:, sl], c[:, sl]),
                                 true_dynamics=util.LinDx(F[:, sl], fs), ls_decay=0.2,
                                 max_ls_iter=10, need_expand=True)
                    xo, uo = st.apply((x0[sl], C[:, sl], c[:, sl], F[:, sl], fs))
                    return st, xo.array, uo.array
                if coupling == "batch":
                    st, rx, ru = run_ref(slice(0, B))
                    rcost = st.for_out.costs
                    robjs = st.for_out.objs
                    extra = dict(full_du_norm=st.for_out.full_du_norm, alpha_du_norm=st.for_out.alpha_du_norm,
                                 mean_alphas=st.for_out.mean_alphas, n_total_qp_iter=st.back_out.n_total_qp_iter)
                else:
                    parts = [run_ref(slice(b, b + 1)) for b in range(B)]
                    rx = np.concatenate([p[1] for p in parts], axis=1)
                    ru = np.concatenate([p[2] for p in parts], axis=1)
                    rcost = np.concatenate([p[0].for_out.costs for p in parts])
                    robjs = np.concatenate([p[0].for_out.objs for p in parts], axis=1)
                    extra = dict(n_total_qp_iter_elem=np.array([p[0].back_out.n_total_qp_iter for p in parts]))
                ox, ou, fo, aux = ompc.step_forward(C, c, F, f, x_nom, u_nom, lo, hi, (C, c), dyn, 0.2, 10,
                                                    n, m, need_expand=True, lu_fp32=fp32, coupling=coupling)
                close(ox, rx, tol=tol, what=name + sfx + coupling + " x")
                close(ou, ru, tol=tol, what=name + sfx + coupling + " u")
                close(fo.costs, rcost, tol=tol, what=name + " costs")
                close(fo.objs, robjs, tol=tol, what=name + " objs")
                if coupling == "batch":
                    close(fo.full_du_norm, extra["full_du_norm"], tol=tol, what="full_du")
                    close(fo.alpha_du_norm, extra["alpha_du_norm"], tol=tol, what="alpha_du")
                    assert int(aux["n_qp"].max(axis=1).sum()) == extra["n_total_qp_iter"]
                else:
                    assert np.array_equal(aux["n_qp"].sum(axis=0), extra["n_total_qp_iter_elem"])
                d = dict(C=C, c=c, F=F, x0=x0, x_nom=x_nom, u_nom=u_nom, lower=lo, upper=hi,
                         x=rx, u=ru, costs=rcost, objs=robjs, n=n, m=m, alphas=fo.alphas, free=aux["free"],
                         Ks=aux["Ks"], ks=aux["ks"])
                d.update(extra)
                if f is not None:
                    d["f"] = f
                # adjoint through the returned point (reference: no_op_forward step's backward)
                if coupling == "batch":
                    gx = rs.randn(T, B, n)
                    gu = rs.randn(T, B, m)
                    st2 = MPCstep(controls=ru, T=T, u_upper=hi, u_lower=lo, n_batch=B, n_state=n, n_ctrl=m,
                                  current_states=rx, true_cost=util.QuadCost(C, c),
                                  true_dynamics=util.LinDx(F, f), ls_decay=0.2, max_ls_iter=10,
                                  need_expand=True, no_op_forward=True)
                    st2.apply((x0, C, c, F, f))
                    g = st2.backward((0, 1, 2, 3, 4), (V(gx), V(gu)))
                    g = [None if v.array is None else np.asarray(v.array) for v in g]
                    og = ompc.step_backward(C, c, F, f, rx, ru, lo, hi, gx, gu, n, m, lu_fp32=fp32)
                    for a, b_, nm in zip(og, g, ("dx0", "dC", "dc", "dF", "df")):
                        if b_ is None:
                            assert a is None
                            continue
                        close(a, b_, tol=tol, what=name + " bwd " + nm)
                    d.update(gx=gx, gu=gu, dx0=g[0], dC=g[1], dc=g[2], dF=g[3])
                    if g[4] is not None:
                        d["df"] = g[4]
                    d["active_frac"] = np.mean((np.abs(ru - lo) <= 1e-8) | (np.abs(ru - hi) <= 1e-8))
                out[name + "_" + coupling + sfx] = d

        # BoxDDP with QuadCost + LinDx (box_ddp.py:93-291)
        for name, (T, B, n, m, bound) in {"ddp_n3m2": (6, 4, 3, 2, 0.5), "ddp_n3m1": (8, 6, 3, 1, 0.3)}.items():
            rs = np.random.RandomState(sum(map(ord, name)))
            s = n + m
            C, c = psd_cost(rs, T, B, s)
            F = stable_dynamics(rs, B, n, m, T)
            f = 0.1 * rs.randn(T - 1, B, n)
            x0 = rs.randn(B, n)
            import io, contextlib
            buf = io.StringIO()
            with contextlib.redirect_stdout(buf):
                solver = BoxDDP(T=T, u_lower=-bound, u_upper=bound, n_batch=B, n_state=n, n_ctrl=m,
                                u_init=None, eps=1e-7, max_iter=30, line_search_decay=0.2,
                                max_line_search_iter=10)
                rx, ru, rcosts = solver((x0, util.QuadCost(V(C), V(c)), util.LinDx(V(F), V(f))))
            o = obox.box_ddp(x0, (C, c), ("linear", F, f), T, -bound, bound, n, m, eps=1e-7, max_iter=30,
                             lu_fp32=fp32, coupling="batch")
            close(o["x"], rx.array, tol=tol * 10, what=name + " ddp x")
            close(o["u"], ru.array, tol=tol * 10, what=name + " ddp u")
            close(o["costs"], np.asarray(rcosts), tol=tol * 10, what=name + " ddp costs")
            out[name + sfx] = dict(C=C, c=c, F=F, f=f, x0=x0, bound=bound, x=rx.array, u=ru.array,
                                   costs=np.asarray(rcosts), n=n, m=m, log=buf.getvalue().strip(),
                                   n_iter=o["n_iter"])

    # ------------------------------------------------------------ pendulum (PendulumDx.forward + BoxDDP)
    mods = _ref_loader.load(lu_fp32=False)
    for modname in ("matplotlib", "matplotlib.pyplot"):
        if modname not in sys.modules:
            mm = types.ModuleType(modname)
            mm.use = lambda *a, **k: None
            mm.style = types.SimpleNamespace(use=lambda *a, **k: None)
            sys.modules[modname] = mm
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.path.insert(0, os.path.join(_ref_loader.REF, "env_dx"))
    import pendulum as ref_pend
    dx = ref_pend.PendulumDx()
    rs = np.random.RandomState(0)
    th = rs.rand(64) * np.pi - np.pi / 2
    thd = rs.rand(64) * 2 - 1
    xin = np.stack((np.cos(th), np.sin(th), thd), axis=1)
    uin = 3.0 * rs.randn(64, 1)
    ref_next = dx(V(xin), V(uin)).array
    close(opend.step(xin, uin), ref_next, what="pendulum step")
    # Jacobian by central differences of the reference step
    xn, R, S = opend.jacobian(xin, uin)
    eps = 1e-6
    for j in range(3):
        e = np.zeros(3); e[j] = eps
        fd = (dx(V(xin + e), V(uin)).array - dx(V(xin - e), V(uin)).array) / (2 * eps)
        assert np.max(np.abs(fd - R[:, :, j])) < 1e-7
    fd = (dx(V(xin), V(uin + eps)).array - dx(V(xin), V(uin - eps)).array) / (2 * eps)
    assert np.max(np.abs(fd - S[:, :, 0])) < 1e-7
    out["pendulum_step"] = dict(x=xin, u=uin, xn=ref_next, R=R, S=S)

    # BoxDDP on the pendulum exactly as IL_Env.mpc wires it (il_env.py:104-158), with the
    # analytic linearisation patched in for approximate.linearize_dynamics (no chainer.grad).
    box_mod = mods["box_ddp"]

    def lin_patch(x, u, dynamics):
        Fl, fl = opend.linearize(np.asarray(x[0].array), np.asarray(u.array))
        return V(Fl), V(fl)
    box_mod.linearize_dynamics = lin_patch
    q_true, p_true = dx.get_true_obj()
    T, B = 20, 16
    rs = np.random.RandomState(0)
    th = rs.rand(B) * np.pi - np.pi / 2
    thd = rs.rand(B) * 2 - 1
    xinit = np.stack((np.cos(th), np.sin(th), thd), axis=1)
    Q = np.repeat(np.repeat(np.diag(q_true)[None, None], T, 0), B, 1)
    p = np.repeat(np.repeat(p_true[None, None], T, 0), B, 1)
    import io, contextlib
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        solver = box_mod.BoxDDP(T=T, u_lower=dx.lower, u_upper=dx.upper, n_batch=B, n_state=3, n_ctrl=1,
                                u_init=None, eps=dx.mpc_eps, max_iter=500, verbose=False,
                                exit_unconverged=False, detach_unconverged=True,
                                line_search_decay=dx.linesearch_decay,
                                max_line_search_iter=dx.max_linesearch_iter, update_dynamics=True)
        rx, ru, rc = solver((xinit, mods["util"].QuadCost(V(Q), V(p)), dx))
    o = obox.box_ddp(xinit, (Q, p), ("pendulum", (10.0, 1.0, 1.0)), T, dx.lower, dx.upper, 3, 1,
                     eps=dx.mpc_eps, max_iter=500, ls_decay=dx.linesearch_decay,
                     max_ls_iter=dx.max_linesearch_iter, coupling="batch")
    close(o["x"], rx.array, tol=1e-9, what="pendulum ddp x")
    close(o["u"], ru.array, tol=1e-9, what="pendulum ddp u")
    out["pendulum_ddp"] = dict(x0=xinit, Q=Q, p=p, x=rx.array, u=ru.array, costs=np.asarray(rc),
                               log=buf.getvalue().strip(), n_iter=o["n_iter"],
                               clamped_frac=np.mean(np.abs(np.abs(ru.array) - 2.0) < 1e-8))

    # ------------------------------------------------------------ LQRnet training trace (KAT chain)
    # examples/LQRnet.ipynb cells 2-10 -> stored output :184-203 (6 printed digits)
    trace = [(0, 0.661925, 4.774785), (10, 0.294314, 4.722322), (20, 0.229643, 4.779115),
             (30, 0.176507, 4.801983), (40, 0.161523, 4.819201), (50, 0.219494, 4.833848),
             (60, 0.148188, 4.845135), (70, 0.134515, 4.835713), (80, 0.164870, 4.823391),
             (90, 0.197836, 4.798079), (100, 0.133565, 4.785647), (110, 0.146801, 4.759894),
             (120, 0.146065, 4.724303), (130, 0.166107, 4.678963), (140, 0.145697, 4.630056),
             (150, 0.146848, 4.585837), (160, 0.155886, 4.535748), (170, 0.146954, 4.473944),
             (180, 0.140506, 4.407619), (190, 0.137744, 4.346956)]
    out["lqrnet_trace"] = dict(trace=np.array(trace))

    for name, d in out.items():
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **{k: np.asarray(v) for k, v in d.items()})
    print("wrote %d fixtures to %s" % (len(out), HERE))
    for k in sorted(out):
        extra = ""
        if "active_frac" in out[k]:
            extra = " active_frac=%.2f" % out[k]["active_frac"]
        if "log" in out[k]:
            extra += " log=%r n_iter=%s" % (out[k]["log"][-40:], out[k].get("n_iter"))
        print("  ", k, extra)


if __name__ == "__main__":
    main()
