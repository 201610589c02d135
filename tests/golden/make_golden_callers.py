#!/usr/bin/env python
"""Fixtures from the reference's own CALLERS of the hot path, run unmodified (build container only):

  il_env_mpc.npz   env_dx/il_env.py  IL_Env.mpc  - (a) data-generation call (il_env.py:94: true q, p, u_init=None,
                   update_dynamics=True) and (b) training call (il_exp.py:249 via pendulum_net.py:34-38: learner q, p,
                   warm-started u_init, update_dynamics=False) at B=64, plus the backward of the final MPCstep for
                   loss = mean((u - u_expert)^2) (il_exp.py:260-275) reduced to the gradients of q and p.
  mpcnet_dx.npz    mpc/mpc_net.py  MpcNet_dx.forward (experiment_mpc/MpcNet.py:44-104 wiring: T=5, n=3, m=3, B=128,
                   bounds +-10) plus the backward reduced to the gradients of A and B.

Chainer 6.3.0 is not installable here, so the reference files run under tests/_chainer_stub (forward only);
approximate.linearize_dynamics (n_state chainer.grad calls per step) is replaced by the analytic pendulum
linearisation of oracle/pendulum.py exactly as tests/golden/make_golden.py does (SURVEY.md H3), and the literal
float32 lu_solve is replaced by the fp64-clean shim (SURVEY.md H1).

    DIFFMPC_REFERENCE=<checkout of the original chainer-differentiable-mpc> python tests/golden/make_golden_callers.py
"""
import contextlib
import io
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


def main():
    mods = _ref_loader.load(lu_fp32=False)
    import chainer
    V = chainer.Variable
    from oracle import pendulum as opend
    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.animation"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["matplotlib"].use = lambda *a, **k: None
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.modules["matplotlib.pyplot"].style = types.SimpleNamespace(use=lambda *a, **k: None)
    sys.path.insert(0, os.path.join(_ref_loader.REF, "env_dx"))
    import il_env as ref_il_env
    box_mod = mods["box_ddp"]
    assert ref_il_env.BoxDDP is box_mod.BoxDDP

    def lin_patch(x, u, dynamics):
        Fl, fl = opend.linearize(np.asarray(x[0].array), np.asarray(u.array))
        return V(Fl), V(fl)
    box_mod.linearize_dynamics = lin_patch

    created = []
    RefStep = box_mod.MPCstep

    class RecordingStep(RefStep):
        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            created.append(self)
    box_mod.MPCstep = RecordingStep

    out = {}
    # ------------------------------------------------------------------ IL_Env.mpc
    env = ref_il_env.IL_Env("pendulum", lqr_iter=500, mpc_T=20)
    np.random.seed(0)
    B, T = 64, 20
    xinit = env.sample_xinit(n_batch=B)                              # il_env.py:48-70
    q_true, p_true = env.true_dx.get_true_obj()
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        xa, ua = env.mpc(env.true_dx, xinit, V(q_true), V(p_true), update_dynamics=True)     # il_env.py:94
    log_a = buf.getvalue().strip().splitlines()[-1]
    n_iter_a = len(created) - 1
    # learner call (pendulum_net.py:34-38): q = sigmoid(logit), p = sqrt(q) * learn_p; warm start = expert + noise
    rs = np.random.RandomState(1)
    q_l = 1.0 / (1.0 + np.exp(-0.3 * rs.randn(4)))                    # learn_q_logit = 0.3 randn
    p_l = np.sqrt(q_l) * (0.5 * rs.randn(4))
    warm = np.clip(ua.array + 0.3 * rs.randn(T, B, 1), -2.0, 2.0)
    del created[:]
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        xb, ub = env.mpc(env.true_dx, xinit, V(q_l), V(p_l), u_init=warm.copy())             # update_dynamics=False
    log_b = buf.getvalue().strip().splitlines()[-1]
    n_iter_b = len(created) - 1
    final = created[-1]
    gu = 2.0 * (ub.array - ua.array) / ub.array.size                 # d mean((u - u_expert)^2) / du
    g = final.backward((0, 1, 2, 3, 4), (None, V(gu)))
    dC, dc = g[1].array, g[2].array
    out["il_env_mpc"] = dict(
        xinit=xinit, q_true=q_true, p_true=p_true, xa=xa.array, ua=ua.array, log_a=log_a, n_iter_a=n_iter_a,
        q_l=q_l, p_l=p_l, warm=warm, xb=xb.array, ub=ub.array, log_b=log_b, n_iter_b=n_iter_b,
        gu=gu, dq=np.einsum("tbii->i", dC), dp=dc.sum(axis=(0, 1)), dx0=g[0].array,
        clamped_frac_a=np.mean(np.abs(np.abs(ua.array) - 2.0) < 1e-8))

    # ------------------------------------------------------------------ MpcNet_dx
    box_mod.MPCstep = RecordingStep
    sys.path.insert(0, os.path.join(_ref_loader.REF, "mpc"))
    import mpc_net as ref_mpc_net
    util = mods["util"]
    T, n, m, B = 5, 3, 3, 128
    s = n + m
    np.random.seed(42)                                               # experiment_mpc/MpcNet.py:48-57
    Q = np.eye(s); p = np.random.randn(s)
    C = util.expand_time_batch(V(Q), T, B); c = util.expand_time_batch(V(p), T, B)
    lo = util.expand_time_batch(-10.0 * np.ones(m), T, B); hi = util.expand_time_batch(10.0 * np.ones(m), T, B)
    del created[:]
    net = ref_mpc_net.MpcNet_dx(T, lo, hi, B, n, m, 1, u_init=None, max_iter=10, verbose=False)
    x_init = np.random.randn(B, n)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        x, u, costs = net((V(x_init), util.QuadCost(C, c)))
    final = created[-1]
    rs = np.random.RandomState(3)
    gx = rs.randn(T, B, n) / (T * B * n); gu = rs.randn(T, B, m) / (T * B * m)
    g = final.backward((0, 1, 2, 3, 4), (V(gx), V(gu)))
    dF = g[3].array
    out["mpcnet_dx"] = dict(Q=Q, p=p, A=net.A.array, B=net.B.array, x_init=x_init, x=x.array, u=u.array,
                            costs=np.asarray(costs), log=buf.getvalue().strip().splitlines()[-1],
                            n_iter=len(created) - 1, gx=gx, gu=gu, dAB=dF.sum(axis=(0, 1)), dx0=g[0].array)

    for name, d in out.items():
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **{k: np.asarray(v) for k, v in d.items()})
        print(name, {k: (np.asarray(v).shape if np.asarray(v).ndim else np.asarray(v).item()) for k, v in d.items()})


if __name__ == "__main__":
    main()
