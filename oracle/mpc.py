"""Oracle: one box-DDP / iLQR step and its adjoint (test infrastructure).

backward_rec   follows mpc/mpc_step.py:70-173
forward_rec    follows mpc/mpc_step.py:175-286 (incl. the batch-scrambled du norms, :261-263)
step_forward   follows mpc/mpc_step.py:288-328
lqr_active     follows mpc/active_constrained_lqr.py:67-193
step_backward  follows mpc/mpc_step.py:330-460

`dynamics` is ('linear', F, f) or ('pendulum', params[, dt, max_torque]) (PendulumDx: params = (g, m, l) or the
non-`simple` (g, m, l, d, b); dt / max_torque default to 0.05 / 2.0); `cost` is (C, c) (QuadCost).
"""
from collections import namedtuple

import numpy as np

from .linalg import bmv, bger, bquad, bdot, clamp, lu_factor, lu_solve
from .pnqp import pnqp
from . import pendulum as _pend

ForOut = namedtuple("ForOut", "objs full_du_norm alpha_du_norm mean_alphas costs alphas u_first n_ls")


def dyn_step(dynamics, t, x, u):
    if dynamics[0] == "linear":
        _, F, f = dynamics
        xn = bmv(F[t], np.concatenate((x, u), axis=1))
        if f is not None:
            xn = xn + f[t]
        return xn
    return _pend.step(x, u, *dynamics[1:])


def traj_cost(x, u, cost):
    """util.py:162-198 with x given."""
    C, c = cost
    T = u.shape[0]
    objs = []
    for t in range(T):
        tau = np.concatenate((x[t], u[t]), axis=1)
        objs.append(0.5 * bquad(tau, C[t]) + bdot(tau, c[t]))
    return np.sum(np.stack(objs), axis=0)


def get_traj(x0, u, dynamics):
    """util.py:201-236."""
    T = u.shape[0]
    xs = [x0]
    for t in range(T - 1):
        xs.append(dyn_step(dynamics, t, xs[t], u[t]))
    return np.stack(xs)


def _scrambled_norm(du, B, T, m):
    """mpc_step.py:261-263 / :275-277: transpose(0,2,1) then reshape(B, T*m) mixes
    batch elements (SURVEY.md H2-iv); kept bit-faithful."""
    d = np.transpose(du, (0, 2, 1)).reshape(B, T * m)
    return np.sqrt(np.sum(d ** 2, axis=1))


def backward_rec(C, c, F, f, u_nom, u_lower, u_upper, n, m, lu_fp32=False, coupling="batch"):
    T, B = C.shape[0], C.shape[1]
    if F.shape[0] == T:
        F = F[:T - 1]
    Ks = np.zeros((T, B, m, n))
    ks = np.zeros((T, B, m))
    n_qp = np.zeros((T, B), dtype=np.int64)
    free_all = np.zeros((T, B, m))
    V = v = None
    prev_k = None
    for t in range(T - 1, -1, -1):
        if t == T - 1:
            Q, q = C[t], c[t]
        else:
            Ft = F[t]
            FtT = np.transpose(Ft, (0, 2, 1))
            Q = C[t] + FtT @ V @ Ft
            if f is None:
                q = c[t] + bmv(FtT, v)
            else:
                q = c[t] + bmv(FtT @ V, f[t]) + bmv(FtT, v)
        Qxx, Qxu = Q[:, :n, :n], Q[:, :n, n:]
        Qux, Quu = Q[:, n:, :n], Q[:, n:, n:]
        qx, qu = q[:, :n], q[:, n:]
        lb = u_lower[t] - u_nom[t]                                   # :136-138
        ub = u_upper[t] - u_nom[t]
        k, fac, free, it = pnqp(Quu, qu, lb, ub, x_init=prev_k, n_iter=20,
                                lu_fp32=lu_fp32, coupling=coupling)  # :141-142
        n_qp[t] = 1 + it
        free_all[t] = free
        prev_k = k
        Qux_m = Qux.copy()
        Qux_m[np.repeat((1.0 - free)[:, :, None], n, axis=2).astype(bool)] = 0.0   # :147-150
        if m == 1:
            K = -((1.0 / fac) * Qux_m)                               # :152-154
        else:
            K = -lu_solve(fac, Qux_m, fp32=lu_fp32)                  # :155-157
        KT = np.transpose(K, (0, 2, 1))
        Ks[t], ks[t] = K, k
        V = Qxx + Qxu @ K + KT @ Qux + KT @ Quu @ K                  # :165 (unmasked Quu,Qux)
        v = qx + bmv(Qxu, k) + bmv(KT, qu) + bmv(KT @ Quu, k)        # :166
    return Ks, ks, n_qp, free_all


def ls_pass(Ks, ks, x_nom, u_nom, u_lower, u_upper, cost, dynamics, alphas):
    """One line-search pass of forward_rec (mpc_step.py:198-253) at the per-element step lengths alphas[B]:
    returns (new_x, new_u, objs[T,B], cost[B])."""
    T = u_nom.shape[0]
    C, c = cost
    new_x = [x_nom[0]]
    new_u = []
    dx = [np.zeros_like(x_nom[0])]
    objs = []
    for t in range(T):
        nu = bmv(Ks[t], dx[t]) + u_nom[t]
        nu = nu + alphas[:, None] * ks[t]                             # :213-219 (diagflat(alphas) @ kt)
        nu = clamp(nu, u_lower[t], u_upper[t])
        new_u.append(nu)
        tau = np.concatenate((new_x[t], nu), axis=1)
        if t < T - 1:
            xn = dyn_step(dynamics, t, new_x[t], nu)
            new_x.append(xn)
            dx.append(xn - x_nom[t + 1])
        objs.append(0.5 * bquad(tau, C[t]) + bdot(tau, c[t]))         # :251
    objs = np.stack(objs)
    return np.stack(new_x), np.stack(new_u), objs, np.sum(objs, axis=0)


def forward_rec(Ks, ks, x_nom, u_nom, u_lower, u_upper, cost, dynamics, ls_decay, max_ls_iter,
                max_trials=200):
    T, B, m = u_nom.shape
    alphas = np.ones(B, dtype=u_nom.dtype)
    old_cost = traj_cost(x_nom, u_nom, cost)                          # :191
    cur = None
    n_iter = 0
    full_du_norm = None
    u_first = None
    while (n_iter < max_ls_iter and cur is None) or (cur is not None and (cur > old_cost).any()):   # :196 (Q5)
        new_x, new_u, objs, cur = ls_pass(Ks, ks, x_nom, u_nom, u_lower, u_upper, cost, dynamics, alphas)
        if full_du_norm is None:
            u_first = new_u.copy()
            full_du_norm = _scrambled_norm(u_nom - new_u, B, T, m)
        alphas[cur > old_cost] *= ls_decay
        n_iter += 1
        if n_iter >= max_trials:
            break
    alpha_du_norm = _scrambled_norm(u_nom - new_u, B, T, m)
    return new_x, new_u, ForOut(objs, full_du_norm, alpha_du_norm, np.mean(alphas), cur, alphas,
                                u_first, n_iter)


def step_forward(C, c, F, f, x_nom, u_nom, u_lower, u_upper, cost, dynamics, ls_decay, max_ls_iter,
                 n, m, need_expand=True, lu_fp32=False, coupling="batch", max_trials=200):
    """mpc_step.py:288-328.  coupling='element' runs the reference control flow with
    n_batch == 1 on every element (SURVEY.md H2) and re-assembles the batch.  max_trials caps the
    line-search passes (forward_rec); n_ls = passes run (per element under 'element')."""
    T, B = C.shape[0], C.shape[1]
    if coupling == "element" and B > 1:
        outs = []
        for b in range(B):
            sl = slice(b, b + 1)
            dyn_b = dynamics
            if dynamics[0] == "linear":
                dyn_b = ("linear", dynamics[1][:, sl], None if dynamics[2] is None else dynamics[2][:, sl])
            outs.append(step_forward(C[:, sl], c[:, sl], F[:, sl], None if f is None else f[:, sl],
                                     x_nom[:, sl], u_nom[:, sl], u_lower[:, sl], u_upper[:, sl],
                                     (cost[0][:, sl], cost[1][:, sl]), dyn_b, ls_decay, max_ls_iter,
                                     n, m, need_expand, lu_fp32, "batch", max_trials))
        x = np.concatenate([o[0] for o in outs], axis=1)
        u = np.concatenate([o[1] for o in outs], axis=1)
        u_first = np.concatenate([o[2].u_first for o in outs], axis=1)
        alphas = np.concatenate([o[2].alphas for o in outs])
        fo = ForOut(np.concatenate([o[2].objs for o in outs], axis=1),
                    _scrambled_norm(u_nom - u_first, B, T, m),
                    _scrambled_norm(u_nom - u, B, T, m),
                    np.mean(alphas),
                    np.concatenate([o[2].costs for o in outs]), alphas, u_first,
                    np.array([o[2].n_ls for o in outs]))
        aux = dict(Ks=np.concatenate([o[3]["Ks"] for o in outs], axis=1),
                   ks=np.concatenate([o[3]["ks"] for o in outs], axis=1),
                   n_qp=np.concatenate([o[3]["n_qp"] for o in outs], axis=1),
                   free=np.concatenate([o[3]["free"] for o in outs], axis=1))
        return x, u, fo, aux
    if need_expand:                                                    # :305-317
        c_hat = np.stack([bmv(C[t], np.concatenate((x_nom[t], u_nom[t]), axis=1)) + c[t] for t in range(T)])
        f_hat = None
    else:
        c_hat, f_hat = c, f
    Ks, ks, n_qp, free = backward_rec(C, c_hat, F, f_hat, u_nom, u_lower, u_upper, n, m, lu_fp32, "batch")
    x, u, fo = forward_rec(Ks, ks, x_nom, u_nom, u_lower, u_upper, cost, dynamics, ls_decay, max_ls_iter,
                           max_trials)
    return x, u, fo, dict(Ks=Ks, ks=ks, n_qp=n_qp, free=free)


def lqr_active(x0, C, c, F, f, active, n, m, lu_fp32=False):
    """active_constrained_lqr.py:67-193.  active[T,B,m] bool."""
    T, B = C.shape[0], C.shape[1]
    Ks = np.zeros((T, B, m, n))
    ks = np.zeros((T, B, m))
    V = v = None
    for t in range(T - 1, -1, -1):
        if t == T - 1:
            Q, q = C[t], c[t]
        else:
            Ft = F[t]
            FtT = np.transpose(Ft, (0, 2, 1))
            Q = C[t] + FtT @ V @ Ft
            if f is None:
                q = c[t] + bmv(FtT, v)
            else:
                q = c[t] + bmv(FtT @ V, f[t]) + bmv(FtT, v)
        Qxx, Qxu = Q[:, :n, :n], Q[:, :n, n:]
        Qux, Quu = Q[:, n:, :n], Q[:, n:, n:]
        qx, qu = q[:, :n], q[:, n:]
        idx = active[t]
        qu_m = qu.copy()
        qu_m[idx] = 0.0                                                # :113-114
        Quu_m = Quu.copy()
        notI = 1.0 - idx.astype(float)
        Quu_m[(1 - bger(notI, notI)).astype(bool)] = 0.0               # :116-119
        ar = np.arange(m)
        diag_mask = np.zeros((B, m, m), dtype=bool)
        diag_mask[:, ar, ar] = idx
        Quu_m[diag_mask] += 1e-8                                       # :121-122
        Qux_m = Qux.copy()
        Qux_m[np.repeat(idx[:, :, None], n, axis=2)] = 0.0             # :124-126
        if m == 1:
            K = -(1.0 / Quu_m) * Qux_m
            k = -(1.0 / Quu_m[:, :, 0]) * qu_m
        else:
            fac = lu_factor(Quu_m)
            K = -lu_solve(fac, Qux_m, fp32=lu_fp32)
            k = -lu_solve(fac, qu_m, fp32=lu_fp32)
        KT = np.transpose(K, (0, 2, 1))
        Ks[t], ks[t] = K, k
        V = Qxx + Qxu @ K + KT @ Qux + (KT @ Quu) @ K                   # :143-144
        v = qx + bmv(Qxu, k) + bmv(KT, qu) + bmv(KT @ Quu, k)
    from .lqr import rollout
    x, u = rollout(x0, Ks, ks, F, f, zero_mask=active)
    return x, u


def step_backward(C, c, F, f, x, u, u_lower, u_upper, dl_dx, dl_du, n, m, lu_fp32=False):
    """mpc_step.py:330-460.  F may have T or T-1 rows (Q8); returns
    (dx0, dC, dc, dF[like F], df[T-1,B,n] or None when f is None)."""
    T, B = C.shape[0], C.shape[1]
    if dl_dx is None:
        dl_dx = np.zeros((T, B, n))
    if dl_du is None:
        dl_du = np.zeros((T, B, m))
    d_taus = np.concatenate((dl_dx, dl_du), axis=2)
    active = (np.abs(u - u_lower) <= 1e-8) | (np.abs(u - u_upper) <= 1e-8)     # :363-364
    dx, du = lqr_active(np.zeros((B, n)), C, -d_taus, F, None, active, n, m, lu_fp32)   # :374-376
    dxu = np.concatenate((dx, du), axis=2)
    xu = np.concatenate((x, u), axis=2)
    dC = np.zeros_like(C)
    for t in range(T):
        dC[t] = -0.5 * (bger(dxu[t], xu[t]) + bger(xu[t], dxu[t]))              # :387
    dc = -dxu
    lams = np.zeros((T, B, n))
    prev = None
    for t in range(T - 1, -1, -1):                                              # :395-406
        lam = bmv(C[t, :, :n, :n], x[t]) + bmv(C[t, :, :n, n:], u[t]) + c[t, :, :n]
        if prev is not None:
            lam = lam + bmv(np.transpose(F[t, :, :, :n], (0, 2, 1)), prev)
        lams[t] = lam
        prev = lam
    dlams = np.zeros_like(lams)
    prev = None
    for t in range(T - 1, -1, -1):                                              # :414-425
        dl = bmv(C[t, :, :n, :n], dx[t]) + bmv(C[t, :, :n, n:], du[t]) - d_taus[t, :, :n]
        if prev is not None:
            dl = dl + bmv(np.transpose(F[t, :, :, :n], (0, 2, 1)), prev)
        dlams[t] = dl
        prev = dl
    dF = np.zeros_like(F)
    for t in range(T - 1):                                                      # :429-436
        dF[t] = -(bger(dlams[t + 1], xu[t]) + bger(lams[t + 1], dxu[t]))
    df = None if f is None else -dlams[1:]                                      # :437-444
    return -dlams[0], dC, dc, dF, df
