"""How the reference's imitation-learning environment calls the solver (env_dx/il_env.py:104-158), restated in a few
lines for runs without the original project at hand: the cost vectors q, p become chainer Variables broadcast to
[T, B, 4, 4] / [T, B, 4] with util.chainer_diag + F.expand_dims + F.repeat, the solver is BoxDDP with the pendulum's own
settings and float bounds, and the dynamics object is passed as is.  TEST INFRASTRUCTURE: tests/callers/run_callers.py uses
the reference's unmodified il_env.py instead when DIFFMPC_REFERENCE names a checkout of it."""
from box_ddp import BoxDDP
from chainer import functions as F
from util import QuadCost, chainer_diag


class IL_Env:
    def __init__(self, env, lqr_iter=500, mpc_T=20, dx_factory=None):
        assert env == "pendulum"
        self.true_dx = dx_factory()
        self.lqr_iter, self.mpc_T = lqr_iter, mpc_T

    def mpc(self, dx, xinit, q, p, u_init=None, eps_override=None, lqr_iter_override=None, update_dynamics=False):
        B, T, d = xinit.shape[0], self.mpc_T, self.true_dx
        Q = F.repeat(F.repeat(F.expand_dims(F.expand_dims(chainer_diag(q), axis=0), axis=0), T, axis=0), B, axis=1)
        pp = F.repeat(F.repeat(F.expand_dims(F.expand_dims(p, axis=0), axis=0), T, axis=0), B, axis=1)
        solver = BoxDDP(T=T, u_lower=d.lower, u_upper=d.upper, n_batch=B, n_state=d.n_state, n_ctrl=d.n_ctrl,
                        u_init=u_init, eps=eps_override or d.mpc_eps, max_iter=lqr_iter_override or self.lqr_iter,
                        verbose=False, exit_unconverged=False, detach_unconverged=True,
                        line_search_decay=d.linesearch_decay, max_line_search_iter=d.max_linesearch_iter,
                        update_dynamics=update_dynamics)
        x_mpc, u_mpc, _ = solver((xinit, QuadCost(Q, pp), dx))
        return x_mpc, u_mpc
