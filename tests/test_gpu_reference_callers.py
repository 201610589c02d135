"""GPU: the reference's CALLERS of the hot path running on this package (VERDICT r1 N1 / f4).

tests/callers/run_callers.py (a child process with the forward-only Chainer stub first on sys.path) drives
  * IL_Env.mpc exactly as env_dx/il_env.py:94 (data generation) and env_dx/il_exp.py:249 (training step, warm start,
    update_dynamics=False) do, B=64 - through the reference's own unmodified il_env.py + pendulum.py when DIFFMPC_REFERENCE
    names a checkout of it, through the few-line restatement tests/callers/il_env_wiring.py otherwise - and the backward of the final
    MPCstep for the imitation loss, reduced to d loss / d q, d loss / d p;
  * MpcNet_dx.forward + backward as experiment_mpc/MpcNet.py:44-104 wires it.
Results are compared with fixtures produced by the UNMODIFIED reference (tests/golden/make_golden_callers.py).

test_boxddp_pendulum_teacher_forced demonstrates (instead of asserting) DESIGN.md section 6: on every iLQR iteration the
CUDA step and the oracle step FROM THE SAME ITERATE agree bit-exactly on PNQP iteration counts and active sets, and on
the line-search alpha of every element whose alpha=1 cost differs from the old cost by more than rounding; where the
decisions agree the new iterate agrees to 1e-10."""
import os
import subprocess
import sys
import tempfile
import warnings

import numpy as np
import pytest

import _native
from _helpers import load_golden, rel_err
from oracle import mpc as ompc, pendulum as opend

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def callers():
    with tempfile.TemporaryDirectory() as td:
        out = os.path.join(td, "callers.npz")
        r = subprocess.run([sys.executable, os.path.join(HERE, "callers", "run_callers.py"), out], capture_output=True,
                           text=True, timeout=900)
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
        d = np.load(out, allow_pickle=False)
        return {k: d[k] for k in d.files}


def test_il_env_mpc_data_generation_call(callers):
    """il_env.py:94: true q, p; u_init=None; update_dynamics=True.  66 % of the controls sit on the +-2 bounds."""
    g = load_golden("il_env_mpc")
    assert str(callers["log_a"]) == str(g["log_a"]) == "Converged"
    assert int(callers["n_iter_a"]) == int(g["n_iter_a"])
    # eps = 1e-3 solver on a non-linear system: elements that are already converged take rounding-level line-search
    # decisions (demonstrated by test_boxddp_pendulum_teacher_forced); the trajectories agree far below eps
    assert np.max(np.abs(callers["ua"] - g["ua"])) < 1e-5 and np.max(np.abs(callers["xa"] - g["xa"])) < 1e-5
    assert abs(np.mean(np.abs(np.abs(callers["ua"]) - 2.0) < 1e-8) - float(g["clamped_frac_a"])) < 0.01


def test_il_env_mpc_training_call_and_gradients(callers):
    """il_exp.py:249-275: learner q, p; warm-started u_init; update_dynamics=False; d mean((u-u_expert)^2) / d(q, p)."""
    g = load_golden("il_env_mpc")
    assert str(callers["log_b"]) == str(g["log_b"])
    assert int(callers["n_iter_b"]) == int(g["n_iter_b"])
    # 18 warm-started iterations of an eps = 1e-3 solver; the rounding-level line-search decisions on already converged
    # elements (test_boxddp_pendulum_teacher_forced) leave the two runs 1e-4-close, a tenth of the solver's own tolerance
    assert np.max(np.abs(callers["ub"] - g["ub"])) < 2e-4 and np.max(np.abs(callers["xb"] - g["xb"])) < 2e-4
    # gradients: the reference's backward at the reference's point vs ours at ours (points differ by < 2e-4)
    scale = max(np.max(np.abs(g["dq"])), np.max(np.abs(g["dp"])))
    assert np.max(np.abs(callers["dq"] - g["dq"])) < 2e-3 * scale and np.max(np.abs(callers["dp"] - g["dp"])) < 2e-3 * scale
    # full-tensor backward and fused (T,B)-sum backward are the same numbers
    assert np.max(np.abs(callers["dq_red"] - callers["dq"])) < 1e-12 * max(1.0, scale)
    assert np.max(np.abs(callers["dp_red"] - callers["dp"])) < 1e-12 * max(1.0, scale)


def test_mpcnet_dx_forward_backward(callers):
    """mpc_net.py:72-87 with the seeding of :57-64; LinDx dynamics from the learned A, B; gradients reach A, B through dF."""
    g = load_golden("mpcnet_dx")
    assert np.array_equal(callers["net_A"], g["A"]) and np.array_equal(callers["net_B"], g["B"])
    assert str(callers["net_log"]) == str(g["log"]) and int(callers["net_n_iter"]) == int(g["n_iter"])
    assert rel_err(callers["net_x"], g["x"]) < 1e-9 and rel_err(callers["net_u"], g["u"]) < 1e-9
    assert rel_err(callers["net_costs"], g["costs"]) < 1e-9
    assert rel_err(callers["net_dx0"], g["dx0"]) < 1e-8
    sc = np.max(np.abs(g["dAB"]))
    assert np.max(np.abs(callers["net_dAB"] - g["dAB"])) < 1e-8 * sc
    assert np.max(np.abs(callers["net_dAB_red"] - g["dAB"])) < 1e-8 * sc


def test_boxddp_pendulum_teacher_forced():
    """BoxDDP on the pendulum (IL_Env.mpc wiring, B=64), iteration by iteration: the CUDA step and the oracle step are run
    from the SAME nominal trajectory (the CUDA path's iterate).  Asserted per iteration:
      * PNQP iteration counts and active sets bit-exact for every element;
      * alpha bit-exact for every element that is not degenerate, where degenerate means: the oracle's own decision hangs
        on the rounding of a T-term sum (|cost(alpha=1) - old_cost| <= 32 eps sum_t |obj_t|);
      * on elements with equal alpha: new x, u within 1e-10 (element-relative), costs 1e-10.
    and over the whole run: some element is degenerate at some iteration only once the solver is converging (so the
    1e-5 end-to-end tolerance of the caller tests is the degenerate decisions' doing, not arithmetic drift)."""
    ctx = _native.default_context(0)
    g = load_golden("il_env_mpc")
    T, B, n, m = 20, 64, 3, 1
    x0 = g["xinit"]
    q, p = g["q_true"], g["p_true"]
    C = np.ascontiguousarray(np.broadcast_to(np.diag(q)[None, None], (T, B, 4, 4)))
    c = np.ascontiguousarray(np.broadcast_to(p[None, None], (T, B, 4)))
    lo = np.full((T, B, m), -2.0); hi = np.full((T, B, m), 2.0)
    par = (10.0, 1.0, 1.0, 0.05, 2.0)
    dC, dc, dlo, dhi, dx0 = (ctx.to_device(a) for a in (C, c, lo, hi, x0))
    u = np.zeros((T, B, m))
    eps64 = np.finfo(np.float64).eps
    n_degenerate, n_checked, converged_at = 0, 0, None
    for it in range(40):
        du = ctx.to_device(u)
        xn = ctx.empty((T, B, n)); Fo = ctx.empty((T - 1, B, 3, 4)); fo = ctx.empty((T - 1, B, 3))
        ctx.get_traj(np.float64, T, B, n, m, _native.DYN_PENDULUM, dx0, du, None, None, par, xn, Fo, fo)
        o = dict(x=ctx.empty((T, B, n)), u=ctx.empty((T, B, m)), Ks=ctx.empty((T, B, m, n)), ks=ctx.empty((T, B, m)),
                 uf=ctx.empty((T, B, m)), objs=ctx.empty((T, B)), costs=ctx.empty((B,)), old=ctx.empty((B,)),
                 al=ctx.empty((B,)), nqp=ctx.empty((T, B), np.int32), fr=ctx.empty((T, B, m), np.uint8),
                 nls=ctx.empty((B,), np.int32), fl=ctx.empty((B,), np.int32))
        ctx.mpc_step_forward(np.float64, T, B, n, m, dC, dc, Fo, T - 1, fo, xn, du, dlo, dhi, dC, dc, _native.DYN_PENDULUM,
                             None, None, par, 0.2, 64, True, _native.COUPLING_BATCH, o["x"], o["u"], o["Ks"], o["ks"],
                             o["uf"], o["objs"], o["costs"], o["old"], o["al"], o["nqp"], o["fr"], o["nls"], o["fl"])
        ctx.sync()
        r = {k: v.download() for k, v in o.items()}
        x_nom, F, f = xn.download(), Fo.download(), fo.download()
        # oracle from the same iterate (nominal trajectory and linearisation recomputed by the oracle itself)
        ox_nom = ompc.get_traj(x0, u, ("pendulum", (10.0, 1.0, 1.0)))
        oF, of = opend.linearize(x0, u)
        assert rel_err(x_nom, ox_nom) < 1e-11 and rel_err(F, oF) < 1e-10
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ox, ou, fo_, aux = ompc.step_forward(C, c, F, f, x_nom, u, lo, hi, (C, c), ("pendulum", (10.0, 1.0, 1.0)),
                                                 0.2, 5, n, m, need_expand=True, coupling="batch")
        assert np.array_equal(r["nqp"], aux["n_qp"]), it
        assert np.array_equal(r["fr"].astype(float), aux["free"]), it
        old = ompc.traj_cost(x_nom, u, (C, c))
        # alpha = 1 trial cost of the oracle: re-run its forward pass at alpha = 1
        _, _, f1 = ompc.forward_rec(aux["Ks"], aux["ks"], x_nom, u, lo, hi, (C, c), ("pendulum", (10.0, 1.0, 1.0)), 1.0, 1,
                                    max_trials=1)
        degenerate = np.abs(f1.costs - old) <= 32 * eps64 * np.sum(np.abs(f1.objs), axis=0)
        same_alpha = r["al"] == fo_.alphas
        assert (same_alpha | degenerate).all(), (it, np.where(~(same_alpha | degenerate))[0])
        n_degenerate += int((~same_alpha).sum()); n_checked += B
        if same_alpha.any():
            assert rel_err(r["x"][:, same_alpha], ox[:, same_alpha]) < 1e-10
            assert rel_err(r["u"][:, same_alpha], ou[:, same_alpha]) < 1e-10
            assert rel_err(r["costs"][same_alpha], fo_.costs[same_alpha]) < 1e-10
        if (~same_alpha).any():
            # a degenerate element's step is tiny: either decision moves u by less than 1e-5
            assert np.max(np.abs(r["u"][:, ~same_alpha] - ou[:, ~same_alpha])) < 1e-5, it
        full = np.sqrt(np.sum(np.transpose(u - r["uf"], (0, 2, 1)).reshape(B, T * m) ** 2, axis=1))
        u = r["u"]
        if full.max() < 1e-3:
            converged_at = it + 1
            break
    assert converged_at is not None and converged_at <= 20
    # n_degenerate / n_checked decisions differed, every one of them on an element that had already converged
    print("teacher-forced BoxDDP: %d of %d line-search decisions differ, all degenerate" % (n_degenerate, n_checked))
