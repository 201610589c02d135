"""CPU (build container): the reference's own caller modules import UNMODIFIED against this package and reach the native
boundary - north_star "drops into env_dx/il_exp.py unchanged" (VERDICT r1 N1).

env_dx/il_env.py:15-20 does `from box_ddp import BoxDDP`, `from pendulum import PendulumDx`, `from util import QuadCost,
chainer_diag`; mpc/mpc_net.py:15-18 does `from box_ddp import BoxDDP`, `from util import expand_time_batch, LinDx`;
experiment_mpc/MpcNet.py:36 needs `util.bmv`, `util.expand_batch`.  With the package directories ahead of the reference's
on sys.path those names must resolve to this package; calling IL_Env.mpc must then fail LOUDLY at dmpc_create (there is no
GPU here and no CPU fallback).  The GPU-side run of the same callers is tests/test_gpu_reference_callers.py.
The reference's files are not part of this repository: the test runs when DIFFMPC_REFERENCE names a checkout of the
original chainer-differentiable-mpc and is skipped otherwise."""
import os
import subprocess
import sys

import pytest

REF = os.environ.get("DIFFMPC_REFERENCE", "")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CODE = r'''
import os, sys, types
ROOT = %r; REF = %r
PKG = os.path.join(ROOT, "chainer-differentiable-mpc_b200")
sys.path[:0] = [os.path.join(ROOT, "tests", "_chainer_stub"), PKG, os.path.join(PKG, "lqr"), os.path.join(PKG, "mpc"), os.path.join(PKG, "env_dx")]
for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.animation"):
    sys.modules[name] = types.ModuleType(name)
sys.modules["matplotlib"].use = lambda *a, **k: None
sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
sys.modules["matplotlib.pyplot"].style = types.SimpleNamespace(use=lambda *a, **k: None)
sys.path += [os.path.join(REF, "env_dx")]
import importlib.util
import numpy as np, chainer
import il_env, util, box_ddp, _native
spec = importlib.util.spec_from_file_location("ref_mpc_net", os.path.join(REF, "mpc", "mpc_net.py"))   # the package has its
mpc_net = importlib.util.module_from_spec(spec); spec.loader.exec_module(mpc_net)                     # own mpc_net.py too
assert il_env.__file__.startswith(REF) and mpc_net.__file__.startswith(REF)
assert util.__file__.startswith(PKG) and box_ddp.__file__.startswith(PKG)
assert il_env.BoxDDP is box_ddp.BoxDDP and mpc_net.BoxDDP is box_ddp.BoxDDP
for name in ("QuadCost", "LinDx", "chainer_diag", "to_xp", "table_log", "get_array_module", "clamp", "xpclamp", "get_cost",
             "xpget_cost", "get_traj", "xpget_traj", "bmv", "xpbmv", "bger", "xpbger", "bquad", "xpbquad",
             "expand_time_batch", "expand_batch", "xpexpand_batch", "bdot", "xpbdot"):
    assert hasattr(util, name), name
rs = np.random.RandomState(0)
a, x, y = rs.randn(5, 3, 4), rs.randn(5, 4), rs.randn(5, 4)
V = chainer.Variable
assert np.allclose(util.bmv(V(a), V(x)).array, np.einsum("bij,bj->bi", a, x))
assert np.allclose(util.bger(V(x), V(y)).array, np.einsum("bi,bj->bij", x, y))
assert np.allclose(util.bdot(V(x), V(y)).array, np.einsum("bi,bi->b", x, y))
Q = rs.randn(5, 4, 4)
assert np.allclose(util.bquad(V(x), V(Q)).array, np.einsum("bi,bij,bj->b", x, Q, x))
assert np.array_equal(util.chainer_diag(V(np.array([1.0, 2.0, 3.0]))).array, np.diag([1.0, 2.0, 3.0]))
assert util.expand_batch(V(x[0]), 7).shape == (7, 4) and util.expand_time_batch(V(x[0]), 3, 7).shape == (3, 7, 4)
assert np.array_equal(util.clamp(V(x), V(-0.5 * np.ones_like(x)), V(0.5 * np.ones_like(x))).array, np.clip(x, -0.5, 0.5))
env = il_env.IL_Env("pendulum", lqr_iter=500, mpc_T=20)
assert type(env.true_dx).__module__ == "pendulum"
import mpc_step
assert mpc_step.is_pendulum(env.true_dx) and mpc_step.pendulum_params(env.true_dx) == (10.0, 1.0, 1.0, 0.05, 2.0)
class PendulumDx:          # an unrelated class that merely shares the name must not be dispatched to the device pendulum
    pass
assert not mpc_step.is_pendulum(PendulumDx())
q, p = env.true_dx.get_true_obj()
try:
    env.mpc(env.true_dx, env.sample_xinit(4), V(q), V(p), update_dynamics=True)
except _native.DiffMpcError as e:
    assert "no CUDA device" in str(e) or "CPU fallback" in str(e), str(e)
    print("LOUD-FAILURE-OK")
else:
    import torch
    assert torch.cuda.is_available(), "IL_Env.mpc returned without a GPU: a CPU fallback exists"
    print("RAN-ON-GPU")
lo = util.expand_time_batch(-np.ones(2), 4, 3); hi = util.expand_time_batch(np.ones(2), 4, 3)
net = mpc_net.MpcNet_dx(4, lo, hi, 3, 3, 2, 1, u_init=None)
assert net.mpc_layer.__class__ is box_ddp.BoxDDP
print("IMPORT-OK")
'''


@pytest.mark.skipif(not (REF and os.path.isdir(os.path.join(REF, "env_dx"))),
                    reason="needs the original chainer-differentiable-mpc: set DIFFMPC_REFERENCE to its checkout")
def test_reference_il_env_and_mpc_net_import_against_package():
    r = subprocess.run([sys.executable, "-c", CODE % (ROOT, REF)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "IMPORT-OK" in r.stdout and ("LOUD-FAILURE-OK" in r.stdout or "RAN-ON-GPU" in r.stdout), r.stdout


def test_package_links_without_chainer():
    """LqrNet / LqrNet_cost_dx / MpcNet_dx are importable and constructible without Chainer (numpy mode) and seed their
    parameters as the reference does (differentiable_lqr.py:167-171, mpc_net.py:57-64)."""
    import numpy as np
    code = r'''
import os, sys
ROOT = %r
PKG = os.path.join(ROOT, "chainer-differentiable-mpc_b200")
sys.path[:0] = [PKG, os.path.join(PKG, "lqr"), os.path.join(PKG, "mpc")]
import numpy as np
import differentiable_lqr as dl, _native
for cls in (dl.LqrNet, dl.LqrNet_cost_dx):
    try:
        cls(5, 8, 3, 1, 1)
    except _native.DiffMpcError:
        pass        # DiffLqr grabs a device context: loud failure without a GPU is the contract
np.random.seed(1); A = np.eye(3) + 0.2 * np.random.randn(3, 3); B = np.random.randn(3, 2)
import mpc_net
net = mpc_net.MpcNet_dx(4, -np.ones((4, 6, 2)), np.ones((4, 6, 2)), 6, 3, 2, 1, u_init=None)
assert np.array_equal(net.A.array, A) and np.array_equal(net.B.array, B)
print("OK")
''' % ROOT
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr
