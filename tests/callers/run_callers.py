#!/usr/bin/env python
"""Child process of tests/test_gpu_reference_callers.py: runs the reference's CALLERS of the hot path on this package
under the forward-only Chainer stub and writes their results to an .npz.

    python tests/callers/run_callers.py OUT.npz

sys.path order = [chainer stub, package dirs, (reference env_dx / mpc dirs when DIFFMPC_REFERENCE names a checkout of
the original chainer-differentiable-mpc)], so `box_ddp`, `mpc_step`, `util`, ... resolve to THIS package while `il_env`,
`pendulum`, `mpc_net` are the reference's unmodified files when that checkout is given and tests/callers' restatement /
the package's own classes otherwise.  The fixtures it is compared with come from the unmodified reference
(tests/golden/make_golden_callers.py).
"""
import contextlib
import io
import os
import sys
import types
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
PKG = os.path.join(ROOT, "chainer-differentiable-mpc_b200")
REF = os.environ.get("DIFFMPC_REFERENCE", "")
USE_REF = bool(REF) and os.path.isdir(os.path.join(REF, "env_dx")) and os.environ.get("DIFFMPC_NO_REFERENCE") != "1"

sys.path[:0] = [os.path.join(TESTS, "_chainer_stub"), PKG, os.path.join(PKG, "lqr"), os.path.join(PKG, "mpc"),
                os.path.join(PKG, "env_dx"), TESTS, HERE]
for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.animation"):
    sys.modules.setdefault(name, types.ModuleType(name))
sys.modules["matplotlib"].use = lambda *a, **k: None
sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
sys.modules["matplotlib.pyplot"].style = types.SimpleNamespace(use=lambda *a, **k: None)
warnings.filterwarnings("ignore")

import chainer  # noqa: E402  (the stub)
import box_ddp  # noqa: E402  (this package)
assert box_ddp.__file__.startswith(PKG), box_ddp.__file__
V = chainer.Variable


def main(out_path):
    from _helpers import load_golden
    res = {"used_reference_callers": USE_REF}
    created = []
    Step = box_ddp.MPCstep

    class RecordingStep(Step):
        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            created.append(self)
    box_ddp.MPCstep = RecordingStep
    solvers = []                                         # BoxDDP instances are local to the callers: record them
    _fwd = box_ddp.BoxDDP.forward

    def recording_forward(self, inputs):
        solvers.append(self)
        return _fwd(self, inputs)
    box_ddp.BoxDDP.forward = recording_forward

    # ---------------------------------------------------------------- IL_Env.mpc (il_env.py:104-158, il_exp.py:249)
    g = load_golden("il_env_mpc")
    if USE_REF:
        sys.path.append(os.path.join(REF, "env_dx"))
        import il_env                                    # the reference's file, unmodified
        assert il_env.__file__.startswith(REF) and il_env.BoxDDP is box_ddp.BoxDDP
        env = il_env.IL_Env("pendulum", lqr_iter=500, mpc_T=20)
        assert type(env.true_dx).__module__ == "pendulum"            # the reference's chainer.Link PendulumDx
    else:
        import il_env_wiring
        from pendulum_dx import PendulumDx
        env = il_env_wiring.IL_Env("pendulum", lqr_iter=500, mpc_T=20, dx_factory=PendulumDx)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        xa, ua = env.mpc(env.true_dx, g["xinit"], V(g["q_true"]), V(g["p_true"]), update_dynamics=True)
    res.update(xa=xa.array, ua=ua.array, log_a=buf.getvalue().strip().splitlines()[-1], n_iter_a=solvers[-1].info["n_iter"])
    del created[:]
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        xb, ub = env.mpc(env.true_dx, g["xinit"], V(g["q_l"]), V(g["p_l"]), u_init=g["warm"].copy())
    res.update(xb=xb.array, ub=ub.array, log_b=buf.getvalue().strip().splitlines()[-1], n_iter_b=solvers[-1].info["n_iter"])
    final = created[-1]
    grads = final.backward((0, 1, 2, 3, 4), (None, V(g["gu"])))       # the FunctionNode protocol, full [T,B,...] tensors
    dC, dc = np.asarray(grads[1].array), np.asarray(grads[2].array)
    red = final.backward_reduced_numpy(None, g["gu"])                 # fused (T,B)-sum
    res.update(dq=np.einsum("tbii->i", dC), dp=dc.sum(axis=(0, 1)), dx0=np.asarray(grads[0].array),
               dq_red=np.diag(red[1]).copy(), dp_red=red[2])

    # ---------------------------------------------------------------- MpcNet_dx (mpc_net.py:20-87, MpcNet.py:44-104)
    g = load_golden("mpcnet_dx")
    import util
    if USE_REF:                                          # the reference's file by path (the package has an mpc_net.py too)
        import importlib.util
        spec = importlib.util.spec_from_file_location("ref_mpc_net", os.path.join(REF, "mpc", "mpc_net.py"))
        mpc_net = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mpc_net)
        assert mpc_net.BoxDDP is box_ddp.BoxDDP
    else:
        import mpc_net
    res["mpc_net_file"] = mpc_net.__file__
    T, B = g["x"].shape[:2]
    n, m = g["A"].shape[0], g["B"].shape[1]
    C = util.expand_time_batch(V(g["Q"]), T, B); c = util.expand_time_batch(V(g["p"]), T, B)
    lo = util.expand_time_batch(-10.0 * np.ones(m), T, B); hi = util.expand_time_batch(10.0 * np.ones(m), T, B)
    del created[:]
    net = mpc_net.MpcNet_dx(T, lo, hi, B, n, m, 1, u_init=None, max_iter=10, verbose=False)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        x, u, costs = net((V(g["x_init"]), util.QuadCost(C, c)))
    final = created[-1]
    grads = final.backward((0, 1, 2, 3, 4), (V(g["gx"]), V(g["gu"])))
    red = final.backward_reduced_numpy(g["gx"], g["gu"])
    res.update(net_A=np.asarray(net.A.array), net_B=np.asarray(net.B.array), net_x=x.array, net_u=u.array,
               net_costs=np.asarray(costs), net_log=buf.getvalue().strip().splitlines()[-1], net_n_iter=solvers[-1].info["n_iter"],
               net_dAB=np.asarray(grads[3].array).sum(axis=(0, 1)), net_dAB_red=red[3], net_dx0=np.asarray(grads[0].array))
    np.savez(out_path, **{k: np.asarray(v) for k, v in res.items()})


if __name__ == "__main__":
    main(sys.argv[1])
