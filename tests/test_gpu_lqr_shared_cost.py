"""GPU: LQR batches that share c as well as C_t and F_t (DMPC_SHARE_C: dmpc_lqr_solve_shared_ex /
dmpc_lqr_adjoint_shared_ex, DiffLqrShared with c [T,s]), and the two model links built on them, LqrNet and
LqrNet_cost_dx.

The oracle runs the reference recursions (oracle/lqr.py) on the broadcast tensors.  Per-element outputs are compared at
rel_err 1e-10 in fp64 (fp32: 1e-4 / 1e-3 on fp32-rounded inputs).  dC and dF keep the bounds of test_gpu_lqr_shared.py;
each entry of the summed dc[T,s] must lie within 1e-10 (fp32: 2e-5) times sum_b |dtau| of the oracle's sum, and every
case shows from the oracle that this bound fails when element B-1 is left out.

With f None the forward is the B = 1 Riccati sweep (run on the shared c) plus lqr_shared_rollout_kernel; with f given it
is lqr_shared_fwd_kernel's vector sweep on the stride-0 c.  Which kernels ran is read from a torch.profiler trace taken in
a child process, as test_gpu_lqr_shared.py does.
"""
import ctypes
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

if __name__ == "__main__":                   # the child process of test_kernels_reached: the paths conftest.py would set
    _root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    _pkg = os.path.join(_root, "chainer-differentiable-mpc_b200")
    sys.path[:0] = [os.path.dirname(os.path.abspath(__file__)), _root, _pkg, os.path.join(_pkg, "lqr")]

from _helpers import load_golden, rel_err  # noqa: E402
from oracle import lqr as olqr  # noqa: E402
from test_gpu_lqr_shared import assert_sum, oracle, shared_problem  # noqa: E402

pytestmark = pytest.mark.gpu

F64, F32 = "f64", "f32"
NP = {F64: np.float64, F32: np.float32}
CNAME = {F64: "double", F32: "float"}
SHARE_C = 1


def tol(dt, grad=False):
    return 1e-10 if dt == F64 else (1e-3 if grad else 1e-4)


def sum_tol(dt):
    return 1e-10 if dt == F64 else 2e-5


def agree_tol(T):
    """share = C against the broadcast-c entry, fp64.  With f None the two take k_t from different kernels (the B = 1
    sweep, the chunk kernel's vector sweep), equal to the last bits; the rollout and the adjoint carry that difference
    through T steps, so the bound is 1e-12 up to T = 20 and grows with T beyond (measured: 1.6e-12 at T = 100)."""
    return 1e-12 * max(1.0, T / 20.0)


# ------------------------------------------------------------------------------------------------ problems
def cost_problem(seed, T, B, n, m, F_T, with_f, pivot, dt):
    """shared_problem with c replaced by one [T,s] block; pr["c"] is its broadcast [T,B,s] (what the oracle and the
    existing entry take), pr["cs"] the block."""
    pr = shared_problem(seed, T, B, n, m, F_T, with_f, pivot, dt)
    cs = np.random.RandomState(seed + 1).randn(T, n + m)
    if dt == F32:
        cs = cs.astype(np.float32).astype(np.float64)
    pr["cs"] = cs
    pr["c"] = np.ascontiguousarray(np.broadcast_to(cs[:, None], (T, B, n + m)))
    return pr


def dc_sum(o):
    """The oracle's sum_b dtau and its bound sum_b |dtau|."""
    return o["dc"].sum(1), np.abs(o["dc"]).sum(1)


def assert_dc_bound_is_sharp(o, eps):
    B = o["dc"].shape[1]
    _, bound = dc_sum(o)
    assert np.max(np.abs(o["dc"][:, B - 1]) / (eps * bound + 1e-300)) > 1.0


# ------------------------------------------------------------------------------------------------ device calls
class Bufs:
    """Device tensors `off` elements past the start of a torch allocation; outputs start as NaN."""

    def __init__(self, off=0):
        import torch
        self.torch, self.off, self.keep = torch, off, []

    def _t(self, dt):
        return {np.dtype(np.float64): self.torch.float64, np.dtype(np.float32): self.torch.float32,
                np.dtype(np.uint8): self.torch.uint8}[np.dtype(dt)]

    def put(self, a, dt):
        a = np.ascontiguousarray(a, dtype=dt)
        t = self.torch.zeros(a.size + self.off, dtype=self._t(dt), device="cuda")
        t[self.off:].copy_(self.torch.from_numpy(a.reshape(-1)))
        self.keep.append(t)
        return t.data_ptr() + self.off * t.element_size()

    def empty(self, shape, dt):
        size = int(np.prod(shape))
        fill = float("nan") if np.dtype(dt).kind == "f" else 0
        t = self.torch.full((size + self.off,), fill, dtype=self._t(dt), device="cuda")
        self.keep.append(t)
        return (t, shape)

    def ptr(self, b):
        return b[0].data_ptr() + self.off * b[0].element_size()

    def get(self, b):
        return b[0][self.off:].cpu().numpy().reshape(b[1])


def run(ctx, pr, dt, strict, share, off=0, gx_null=False, gu_null=False, repeat=False):
    """Forward + adjoint through the C ABI.  share = SHARE_C: c [T,s] through the _ex calls; share = None: the existing
    entry points on the broadcast c [T,B,s]."""
    import torch
    T, B, n, m, F_T = pr["T"], pr["B"], pr["n"], pr["m"], pr["F_T"]
    s, R = n + m, NP[dt]
    bf = Bufs(off)
    c_in = pr["cs"] if share else pr["c"]
    x0, C, c, F = bf.put(pr["x0"], R), bf.put(pr["C"], R), bf.put(c_in, R), bf.put(pr["F"], R) if F_T else None
    f = bf.put(pr["f"], R) if pr["f"] is not None else None
    gx = None if gx_null else bf.put(pr["gx"], R)
    gu = None if gu_null else bf.put(pr["gu"], R)
    nb = ctx.lqr_shared_workspace_bytes(R, T, B, n, m, share)
    ws = bf.empty((nb,), np.uint8)
    o = {k: bf.empty(v, R) for k, v in dict(x=(T, B, n), u=(T, B, m), dx0=(B, n), dC=(T, s, s),
                                             dc=(T, s) if share else (T, B, s), dF=(F_T, n, s),
                                             df=(max(T - 1, 0), B, n)).items()}
    P = {k: bf.ptr(v) for k, v in o.items()}
    torch.cuda.synchronize()
    flags = 1 if strict else 0
    have_df = pr["f"] is not None and T > 1

    def call():
        ctx.lqr_solve_shared(R, T, B, n, m, x0, C, c, F, F_T, f, P["x"], P["u"], bf.ptr(ws), nb, share=share)
        ctx.lqr_adjoint_shared(R, T, B, n, m, C, c, F, F_T, P["x"], P["u"], gx, gu, bf.ptr(ws), P["dx0"], P["dC"],
                               P["dc"], P["dF"] if F_T else None, P["df"] if have_df else None, flags, ws_bytes=nb,
                               share=share)
        ctx.sync()
        return {k: bf.get(v) for k, v in o.items()}

    out = call()
    if repeat:
        out["again"] = call()
    return out


def check(pr, dt, strict, out, gx_null=False, gu_null=False):
    o = oracle(pr, strict, gx_null, gu_null)
    T = pr["T"]
    for k in ("x", "u"):
        assert rel_err(out[k], o[k]) < tol(dt), k
    assert rel_err(out["dx0"], o["dx0"]) < tol(dt, True), "dx0"
    if pr["f"] is not None and T > 1:
        assert rel_err(out["df"], o["df"]) < tol(dt, True), "df"
    want, bound = dc_sum(o)
    assert_sum(out["dc"], want, bound, sum_tol(dt), "dc")
    assert_sum(out["dC"], o["dC"], o["bC"], sum_tol(dt), "dC")
    assert_sum(out["dF"], o["dF"], o["bF"], sum_tol(dt), "dF")
    if pr["F_T"] == T:
        assert np.all(out["dF"][T - 1] == 0)
    assert_dc_bound_is_sharp(o, sum_tol(dt))
    return o


# ------------------------------------------------------------------------------------------------ cases
# (n, m) -> kernel of the B = 1 matrix sweep (the families test_gpu_lqr_shared.py reaches)
SWEEP = {(2, 1): "lqr_tpe_kernel<{R}, 2, 1,", (3, 1): "lqr_tpe_kernel<{R}, 3, 1,", (4, 2): "lqr_tpe_kernel<{R}, 4, 2,",
         (8, 4): "lqr_solve_kernel<{R}, 8, 4, 16>", (32, 8): "lqr_factor_dmma_warp_kernel<4, {R}>",
         (5, 1): "lqr_solve_kernel<{R}, 0, 0, 8>", (3, 9): "lqr_solve_kernel<{R}, 0, 0, 16>",
         (12, 10): "lqr_solve_kernel<{R}, 0, 0, 32>", (40, 24): "lqr_solve_kernel<{R}, 0, 0, 256>"}


def case(n, m, T=17, B=37, dt=F64, F_T=None, with_f=True, strict=True, pivot=None, off=0, gx_null=False, gu_null=False):
    return dict(n=n, m=m, T=T, B=B, dt=dt, F_T=T - 1 if F_T is None else F_T, with_f=with_f, strict=strict,
                pivot=(m >= 2) if pivot is None else pivot, off=off, gx_null=gx_null, gu_null=gu_null)


CASES = ([case(n, m, dt=dt, with_f=wf) for (n, m) in SWEEP for dt in (F64, F32) for wf in (False, True)] +
         [case(32, 8, T=100, B=300, F_T=100, with_f=False),         # config-5 horizon, F with T rows, rollout-only
          case(32, 8, T=100, B=300, F_T=100),
          case(32, 8, T=100, B=300, with_f=False, strict=False, dt=F32),
          case(32, 8, T=1, B=5, F_T=1, with_f=False), case(32, 8, T=2, B=64, with_f=False, strict=False),
          case(32, 8, T=17, B=1, with_f=False), case(32, 8, T=17, B=1),
          case(3, 1, T=1, B=3, F_T=0, with_f=False), case(3, 1, T=2, B=2, F_T=2),
          case(4, 2, T=5, B=9473, with_f=False),                     # NB = 64, one-element last chunk
          case(8, 4, T=5, B=4737, strict=False),                     # NB = 32
          case(8, 4, T=5, B=4737, with_f=False),
          case(12, 10, T=9, B=2369, with_f=False),                   # NB = 16
          case(5, 1, T=9, B=2351),                                   # NB = 8 (B < 16 * 148), ragged
          case(3, 9, T=9, B=200, strict=False, gx_null=True), case(5, 1, T=9, B=50, gu_null=True, with_f=False),
          case(32, 8, off=1, with_f=False), case(32, 8, off=1), case(3, 9, off=1, dt=F32, with_f=False),
          case(40, 24, T=6, B=9, off=1)])


def case_id(c):
    return "{dt}-n{n}m{m}-T{T}-B{B}-FT{F_T}{f}{s}{p}{o}{gx}{gu}".format(
        f="-f" if c["with_f"] else "", s="-strict" if c["strict"] else "", p="-piv" if c["pivot"] else "",
        o="-off1" if c["off"] else "", gx="-gxnull" if c["gx_null"] else "", gu="-gunull" if c["gu_null"] else "", **c)


def problem_of(c):
    seed = (c["n"] * 131 + c["m"] * 17 + c["T"] * 7 + c["B"] + 5) % 100000
    return cost_problem(seed, c["T"], c["B"], c["n"], c["m"], c["F_T"], c["with_f"], c["pivot"], c["dt"])


def expected_kernels(c):
    """(kernels that must run, kernels that must not)."""
    R = CNAME[c["dt"]]
    sweep = SWEEP[(c["n"], c["m"])]
    if c["off"] and (c["n"], c["m"]) == (32, 8):     # C, F not 16-byte aligned: the DMMA sweep hands over to the group kernel
        sweep = "lqr_solve_kernel<{R}, 32, 8, 256>"
    fwd, other = ("fwd", "rollout") if c["with_f"] else ("rollout", "fwd")
    want = [sweep.format(R=R)] + ["lqr_shared_%s_kernel<%s>" % (k, R) for k in (fwd, "adj", "reduce")]
    return want, ["lqr_shared_%s_kernel<%s>" % (other, R)]


@pytest.fixture(scope="module")
def ctx():
    import _native
    return _native.default_context(0)


@pytest.mark.parametrize("c", CASES, ids=case_id)
def test_oracle_parity(ctx, c):
    pr = problem_of(c)
    out = run(ctx, pr, c["dt"], c["strict"], SHARE_C, c["off"], c["gx_null"], c["gu_null"], repeat=True)
    check(pr, c["dt"], c["strict"], out, c["gx_null"], c["gu_null"])
    for k, v in out["again"].items():                               # a repeated call returns the same bits
        assert np.array_equal(v, out[k], equal_nan=True), k


@pytest.mark.parametrize("c", [c for c in CASES if c["dt"] == F64], ids=case_id)
def test_agrees_with_broadcast_c(ctx, c):
    """share = C against the existing entry fed the broadcast c [T,B,s] on the same problem.  The two compute k_t in
    different kernels when f is None (the sweep vs the chunk kernel), so they agree to agree_tol(T), not in every bit."""
    pr = problem_of(c)
    a = run(ctx, pr, c["dt"], c["strict"], SHARE_C, c["off"], c["gx_null"], c["gu_null"])
    b = run(ctx, pr, c["dt"], c["strict"], None, c["off"], c["gx_null"], c["gu_null"])
    errs = {k: rel_err(a[k], b[k]) for k in ("x", "u", "dx0", "dC", "dF")}
    errs["dc"] = rel_err(a["dc"], b["dc"].sum(1))
    if pr["f"] is not None and pr["T"] > 1:
        errs["df"] = rel_err(a["df"], b["df"])
    assert max(errs.values()) <= agree_tol(pr["T"]), errs


def test_cases_cover_every_sweep_family():
    """CPU-side bookkeeping of CASES: every sweep family in both dtypes and both forward forms, m > n, F with T rows,
    T = 1, 2, 17 and 100, B = 1, strict and not, NULL gx and gu, misaligned pointers."""
    for R in (F64, F32):
        for wf in (False, True):
            assert {(c["n"], c["m"]) for c in CASES if c["dt"] == R and c["with_f"] == wf} == set(SWEEP)
    assert any(c["m"] > c["n"] for c in CASES) and any(c["F_T"] == c["T"] for c in CASES)
    assert {1, 2, 17, 100} <= {c["T"] for c in CASES} and 1 in {c["B"] for c in CASES}
    assert any(not c["strict"] for c in CASES) and any(c["gx_null"] for c in CASES) and any(c["gu_null"] for c in CASES)
    assert any(c["off"] and c["with_f"] for c in CASES) and any(c["off"] and not c["with_f"] for c in CASES)


def test_kernels_reached():
    """Every case in a child process under torch.profiler: its sweep kernel, the forward form its f selects (and not
    the other one), the adjoint and the reduction ran."""
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "names.npz")
        env = {k: v for k, v in os.environ.items() if not k.startswith("DMPC_")}
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", path], env=env, capture_output=True,
                           text=True, timeout=900)
        assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-4000:])
        with np.load(path, allow_pickle=False) as z:
            names = {k: list(z[k]) for k in z.files}
    seen = set()
    for c in CASES:
        got = names[case_id(c)]
        want, not_want = expected_kernels(c)
        for e in want:
            assert any(e in k for k in got), (case_id(c), e, got)
        for e in not_want:
            assert not any(e in k for k in got), (case_id(c), e, got)
        seen |= set(got)
    for R in CNAME.values():
        for k in ("fwd", "rollout", "adj", "reduce"):
            assert any("lqr_shared_%s_kernel<%s>" % (k, R) in s for s in seen)


# ------------------------------------------------------------------------------------------------ links
def test_lqrnet_training_trace():
    """The LQRnet notebook (tests/golden/lqrnet_trace.npz: 190 RMSprop updates on net.A, net.B, seed=2) through
    LqrNet.forward / backward_numpy: C = I is the same for every element, so the link runs on DiffLqrShared."""
    from differentiable_lqr import LqrNet
    from lqr_recursion import LqrRecursion
    want = {int(r[0]): (r[1], r[2]) for r in load_golden("lqrnet_trace")["trace"]}
    T, n, m, B = 5, 3, 1, 128
    s = n + m
    np.random.seed(42)
    p = np.random.randn(s)
    A = np.eye(n) + 0.2 * np.random.randn(n, n)
    Bm = np.random.randn(n, m)
    expF = np.broadcast_to(np.concatenate((A, Bm), 1), (T - 1, B, n, s)).copy()
    Cb = np.broadcast_to(np.eye(s), (T, B, s, s)).copy()
    c = np.broadcast_to(p, (T, B, s)).copy()
    net = LqrNet(T, B, n, m, 2)
    msA, msB = np.zeros((n, n)), np.zeros((n, m))
    checked = 0
    for i in range(191):
        x0 = np.random.randn(B, n)
        xt, ut = [np.asarray(getattr(v, "array", v)) for v in LqrRecursion(x0, Cb, c, expF, None, T, n, m).solve_recursion()]
        xp_, up_ = [np.asarray(getattr(v, "array", v)) for v in net.forward((x0, Cb, c, None))]
        assert net._used_shared
        loss = np.mean((ut - up_) ** 2) + np.mean((xt - xp_) ** 2)
        gA, gB = net.backward_numpy(-2 * (xt - xp_) / xp_.size, -2 * (ut - up_) / up_.size)
        for P, G, ms in ((net.A.array, gA, msA), (net.B.array, gB, msB)):
            ms *= 0.99
            ms += 0.01 * G * G
            P -= 1e-2 * G / (np.sqrt(ms) + 1e-8)
        ml = np.mean((net.A.array - A) ** 2) + np.mean((net.B.array - Bm) ** 2)
        if i in want:
            assert abs(loss - want[i][0]) < 1e-6 and abs(ml - want[i][1]) < 1e-6, (i, loss, ml)
            checked += 1
    assert checked == len(want)


def _link_ab(net):
    return np.concatenate((np.asarray(net.A.array), np.asarray(net.B.array)), 1)


def _lqrnet_oracle(net, x0, C, c, f, gx, gu):
    """The reference recursions on a link's tensors, C [T,B,s,s] per element: (x, u, dF summed over t and b, and the
    sum of |dF_{t,b}| as its scale)."""
    T, B, n, m = net.T, net.n_batch, net.n_state, net.n_ctrl
    F = np.broadcast_to(_link_ab(net), (T - 1, B, n, n + m)).copy()
    x, u, _, _ = olqr.lqr_solve(x0, C, c, F, f, n, m)
    dF = olqr.difflqr_backward(x0, C, c, F, x, u, gx, gu, n, m, True, True)[3]
    return x, u, dF.sum((0, 1)), np.abs(dF).sum((0, 1))


def _cost_oracle(net, x0, f, gx, gu):
    """oracle() of test_gpu_lqr_shared on LqrNet_cost_dx's parameters broadcast over [T, B] (C [T,s,s] shared)."""
    T, B, n, m = net.T, net.n_batch, net.n_state, net.n_ctrl
    s = n + m
    pr = dict(T=T, B=B, n=n, m=m, F_T=T - 1, C=np.broadcast_to(np.asarray(net.C.array), (T, s, s)).copy(),
              F=np.broadcast_to(_link_ab(net), (T - 1, n, s)).copy(),
              c=np.broadcast_to(np.asarray(net.c.array), (T, B, s)).copy(), x0=x0, f=f, gx=gx, gu=gu)
    return oracle(pr, True)


def test_lqrnet_selects_by_input(ctx):
    """LqrNet picks DiffLqrShared for a plain C that does not vary over the batch (stride 0 or a copy) and keeps DiffLqr
    for a C that varies per element; every route matches the oracle, and the two shared inputs give the same bits."""
    from differentiable_lqr import LqrNet
    T, B, n, m = 6, 40, 4, 2
    s = n + m
    pr = shared_problem(21, T, B, n, m, T - 1)
    net = LqrNet(T, B, n, m, 3)
    Cv = np.ascontiguousarray(np.broadcast_to(pr["C"][:, None], (T, B, s, s))).copy()
    Cv[:, 7] += 0.05 * np.eye(s)                                     # one element differs: per-element route
    stride0 = np.broadcast_to(pr["C"][:, None], (T, B, s, s))
    results = {}
    for name, C, shared in (("varies", Cv, False), ("stride0", stride0, True), ("copy", np.ascontiguousarray(stride0), True)):
        x, u = [np.asarray(getattr(v, "array", v)) for v in net.forward((pr["x0"], C, pr["c"], pr["f"]))]
        assert net._used_shared == shared, name
        gA, gB = net.backward_numpy(pr["gx"], pr["gu"])
        ox, ou, dF, scale = _lqrnet_oracle(net, pr["x0"], np.ascontiguousarray(C), pr["c"], pr["f"], pr["gx"], pr["gu"])
        assert rel_err(x, ox) < 1e-10 and rel_err(u, ou) < 1e-10, name
        assert_sum(np.concatenate((gA, gB), 1), dF, scale, 1e-10, name)
        results[name] = (x, u, gA, gB)
    for a, b in zip(results["stride0"], results["copy"]):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("with_f", [False, True])
def test_lqrnet_cost_dx_matches_oracle(ctx, with_f):
    """LqrNet_cost_dx.forward / backward_numpy against the oracle on the broadcast tensors: per-element x, u; the
    (T,B)-summed dA, dB, dC and dc within the sum bounds, each shown to fail without element B-1."""
    from differentiable_lqr import LqrNet_cost_dx
    T, B, n, m = 9, 70, 4, 2
    s = n + m
    net = LqrNet_cost_dx(T, B, n, m, 4)
    rs = np.random.RandomState(8)
    x0, gx, gu = rs.randn(B, n), rs.randn(T, B, n), rs.randn(T, B, m)
    f = 0.1 * rs.randn(T - 1, B, n) if with_f else None
    x, u = [np.asarray(getattr(v, "array", v)) for v in net.forward((x0, f))]
    gA, gB, gC, gc = net.backward_numpy(gx, gu)
    assert gA.shape == (n, n) and gB.shape == (n, m) and gC.shape == (s, s) and gc.shape == (s,)
    o = _cost_oracle(net, x0, f, gx, gu)
    assert rel_err(x, o["x"]) < 1e-10 and rel_err(u, o["u"]) < 1e-10
    assert_sum(np.concatenate((gA, gB), 1), o["dF"].sum(0), o["bF"].sum(0), 1e-10, "dF")
    assert_sum(gC, o["dC"].sum(0), o["bC"].sum(0), 1e-10, "dC")
    assert_sum(gc, o["dc"].sum((0, 1)), np.abs(o["dc"]).sum((0, 1)), 1e-10, "dc")
    lim = lambda b: 1e-10 * b + 1e-300
    assert np.max(np.abs(o["dc"][:, B - 1].sum(0)) / lim(np.abs(o["dc"]).sum((0, 1)))) > 1.0
    assert np.max(np.abs(o["dC_full"][:, B - 1].sum(0)) / lim(o["bC"].sum(0))) > 1.0
    assert np.max(np.abs(o["dF_full"][:, B - 1].sum(0)) / lim(o["bF"].sum(0))) > 1.0


@pytest.mark.parametrize("F_T,with_f", [(4, True), (5, False)])
def test_facade_gradient_shapes_shared_c(F_T, with_f):
    """DiffLqrShared with c [T,s]: the FunctionNode backward returns dc [T,s] (summed over the batch)."""
    from differentiable_lqr import DiffLqrShared
    T, B, n, m = 5, 7, 4, 2
    s = n + m
    pr = cost_problem(3, T, B, n, m, F_T, with_f, True, F64)
    node = DiffLqrShared(T, B, n, m, strict_reference=False)
    x, u = node.apply((pr["x0"], pr["C"], pr["cs"], pr["F"], pr["f"]))
    x, u = np.asarray(getattr(x, "array", x)), np.asarray(getattr(u, "array", u))
    g = node.backward((0, 1, 2, 3, 4), (pr["gx"], pr["gu"]))
    g = [None if v is None else np.asarray(getattr(v, "array", v)) for v in g]
    assert g[0].shape == (B, n) and g[1].shape == (T, s, s) and g[2].shape == (T, s) and g[3].shape == (F_T, n, s)
    assert (g[4] is None) == (not with_f) and (g[4] is None or g[4].shape == (T - 1, B, n))
    o = oracle(pr, False)
    assert rel_err(x, o["x"]) < 1e-10 and rel_err(g[0], o["dx0"]) < 1e-10
    want, bound = dc_sum(o)
    assert_sum(g[2], want, bound, 1e-10, "dc")
    assert_sum(g[1], o["dC"], o["bC"], 1e-10, "dC")
    assert_sum(g[3], o["dF"], o["bF"], 1e-10, "dF")
    # the same node, fed c [T,B,s] next, returns dc [T,B,s] again
    node.apply((pr["x0"], pr["C"], pr["c"], pr["F"], pr["f"]))
    g2 = node.backward((0, 1, 2, 3, 4), (pr["gx"], pr["gu"]))
    assert np.asarray(getattr(g2[2], "array", g2[2])).shape == (T, B, s)


def test_capacity_lqrnet_cost_dx_full_config5_batch(ctx):
    """LqrNet_cost_dx at config 5 (n = 32, m = 8, T = 100), B = 65536, fp64, in one call.  64 sampled elements match
    the oracle (x, u, dx0); the summed gradients equal the sum of two half-batch links within the sum bounds, taken over
    the whole batch from tau and dtau (dtau from the per-element shared entry on the broadcast c)."""
    import torch
    from differentiable_lqr import LqrNet_cost_dx
    T, B, n, m = 100, 65536, 32, 8
    s = n + m
    g = torch.Generator(device="cuda").manual_seed(4)
    rn = lambda *shape: torch.randn(*shape, generator=g, device="cuda", dtype=torch.float64)
    x0, gx, gu = rn(B, n).cpu().numpy(), rn(T, B, n).cpu().numpy(), rn(T, B, m).cpu().numpy()
    net = LqrNet_cost_dx(T, B, n, m, 6)
    # a stable A and a well-conditioned C: at n = 32 the seeded I + 0.2 randn would let x grow over 100 steps
    A = np.eye(n) + 0.1 / np.sqrt(n) * np.random.RandomState(1).randn(n, n)
    net.A.array[...] = A * (0.9 / np.max(np.abs(np.linalg.eigvals(A))))
    net.C.array[...] = np.eye(s) + 0.05 * np.random.RandomState(2).randn(s, s)
    x, u = [np.asarray(getattr(v, "array", v)) for v in net.forward((x0, None))]
    grads = [a.copy() for a in net.backward_numpy(gx, gu)]
    dx0 = net.lqr_layer.backward_numpy(gx, gu)[0]
    again = net.backward_numpy(gx, gu)
    for a, b in zip(grads, again):                                   # deterministic
        assert np.array_equal(a, b)
    idx = np.sort(np.random.RandomState(5).choice(B, 64, replace=False))
    idx[-1] = B - 1
    Cm, cv = np.asarray(net.C.array), np.asarray(net.c.array)
    AB = _link_ab(net)
    pr = dict(T=T, B=64, n=n, m=m, F_T=T - 1, C=np.broadcast_to(Cm, (T, s, s)).copy(),
              F=np.broadcast_to(AB, (T - 1, n, s)).copy(), c=np.broadcast_to(cv, (T, 64, s)).copy(), x0=x0[idx], f=None,
              gx=gx[:, idx], gu=gu[:, idx])
    o = oracle(pr, True)
    assert rel_err(x[:, idx], o["x"]) < 1e-10 and rel_err(u[:, idx], o["u"]) < 1e-10
    assert rel_err(dx0[idx], o["dx0"]) < 1e-10
    # sum bounds over the whole batch, on the device: dtau from the existing entry on the broadcast c
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    Cd, Fd, cb = dev(pr["C"]), dev(pr["F"]), dev(cv).expand(T, B, s).contiguous()
    xd, ud, gxd, gud, x0d = dev(x), dev(u), dev(gx), dev(gu), dev(x0)
    nb = ctx.lqr_shared_workspace_bytes(np.float64, T, B, n, m)
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    xb, ub, dtau = torch.empty_like(xd), torch.empty_like(ud), torch.empty(T, B, s, dtype=torch.float64, device="cuda")
    dxb, dCb, dFb = torch.empty_like(x0d), torch.empty(T, s, s, dtype=torch.float64, device="cuda"), torch.empty(T - 1, n, s, dtype=torch.float64, device="cuda")
    P = lambda t: t.data_ptr()
    ctx.lqr_solve_shared(np.float64, T, B, n, m, P(x0d), P(Cd), P(cb), P(Fd), T - 1, None, P(xb), P(ub), P(ws), nb)
    ctx.lqr_adjoint_shared(np.float64, T, B, n, m, P(Cd), P(cb), P(Fd), T - 1, P(xb), P(ub), P(gxd), P(gud), P(ws),
                           P(dxb), P(dCb), P(dtau), P(dFb), None, 1, ws_bytes=nb)
    ctx.sync()
    del ws
    assert rel_err(xb.cpu().numpy(), x) <= agree_tol(T) and rel_err(dxb.cpu().numpy(), dx0) <= agree_tol(T)
    tau = torch.cat((xd, ud), 2)
    a = torch.einsum("tbi,tbj->ij", dtau.abs(), tau.abs())
    bC = (0.5 * a + a.T).cpu().numpy()
    bc = dtau.abs().sum((0, 1)).cpu().numpy()
    lam = torch.zeros(T, B, n, dtype=torch.float64, device="cuda"); dlam = torch.zeros_like(lam)
    for t in range(T - 1, -1, -1):
        lam[t] = tau[t] @ Cd[t][:n].T + cb[t][:, :n]
        dlam[t] = dtau[t] @ Cd[t][:n].T + gxd[t]
        if t < T - 1:
            lam[t] += lam[t + 1] @ Fd[t][:, :n]
            dlam[t] += dlam[t + 1] @ Fd[t][:, :n]
    bF = (torch.einsum("tbi,tbj->ij", dlam[1:].abs(), tau[:-1].abs()) +
          torch.einsum("tbi,tbj->ij", lam[1:].abs(), dtau[:-1].abs())).cpu().numpy()
    del xd, ud, gxd, gud, tau, dtau, lam, dlam, cb, xb, ub
    halves = []
    for lo, hi in ((0, B // 2), (B // 2, B)):
        h = LqrNet_cost_dx(T, hi - lo, n, m, 6)
        for nm in ("A", "B", "C", "c"):
            getattr(h, nm).array[...] = getattr(net, nm).array
        h.forward((x0[lo:hi], None))
        halves.append([a.copy() for a in h.backward_numpy(gx[:, lo:hi], gu[:, lo:hi])])
        del h
    hs = [a + b for a, b in zip(*halves)]
    assert_sum(np.concatenate(grads[:2], 1), np.concatenate(hs[:2], 1), bF, 1e-10, "dF")
    assert_sum(grads[2], hs[2], bC, 1e-10, "dC")
    assert_sum(grads[3], hs[3], bc, 1e-10, "dc")


# ------------------------------------------------------------------------------------------------ errors
def test_errors(ctx):
    lib, h = ctx.lib, ctx.h
    T, B, n, m = 4, 3, 3, 2
    sz = ctypes.c_size_t(0)
    assert lib.dmpc_lqr_shared_workspace_bytes_ex(0, T, B, n, m, 2, ctypes.byref(sz)) == 5
    assert lib.dmpc_lqr_shared_workspace_bytes_ex(0, T, B, n, m, 1, None) == 1
    assert lib.dmpc_lqr_shared_workspace_bytes_ex(0, T, B, n, m, 0, ctypes.byref(sz)) == 0
    nb0 = sz.value
    plain = ctypes.c_size_t(0)
    assert lib.dmpc_lqr_shared_workspace_bytes(0, T, B, n, m, ctypes.byref(plain)) == 0 and plain.value == nb0
    assert lib.dmpc_lqr_shared_workspace_bytes_ex(0, T, B, n, m, 1, ctypes.byref(sz)) == 0
    nb = sz.value
    assert nb > nb0
    ws = ctx.empty((nb,), np.uint8)
    bufs = [ctx.empty((4096,), np.float64) for _ in range(12)]
    p = [b.ptr for b in bufs]

    def solve(**k):
        return lib.dmpc_lqr_solve_shared_ex(k.get("h", h), 0, T, B, n, m, k.get("x0", p[0]), p[1], k.get("c", p[2]), p[3],
                                            T - 1, None, k.get("x", p[4]), p[5], ws.ptr, k.get("nb", nb),
                                            k.get("share", 1), None)

    def adj(**k):
        return lib.dmpc_lqr_adjoint_shared_ex(k.get("h", h), 0, T, B, n, m, p[1], k.get("c", p[2]), p[3], T - 1, p[4],
                                              p[5], None, None, ws.ptr, k.get("nb", nb), p[6], k.get("dC", p[7]),
                                              k.get("dc", p[8]), p[9], None, 1, k.get("share", 1), None)
    assert solve() == 0 and adj() == 0
    assert adj(dc=None) == 0                                         # dc is nullable with DMPC_SHARE_C
    assert solve(share=0) == 0 and adj(share=0) == 0
    assert adj(share=0, dc=None) == 6                                # ... and required without it
    assert solve(share=2) == 5 and adj(share=3) == 5                 # unknown bits
    assert solve(nb=nb0) == 1 and adj(nb=nb0) == 1                   # a share = 0 workspace is too small
    assert solve(x0=None) == 6 and solve(c=None) == 6 and solve(x=None) == 6
    assert adj(c=None) == 6 and adj(dC=None) == 6
    assert solve(h=None) == 6 and adj(h=None) == 6
    ctx.sync()
    for b in bufs:
        b.free()
    ws.free()
    from differentiable_lqr import DiffLqrShared
    pr = cost_problem(1, T, B, n, m, T - 1, True, False, F64)
    node = DiffLqrShared(T, B, n, m)
    with pytest.raises(AssertionError, match="c dim"):
        node.apply_numpy(pr["x0"], pr["C"], pr["cs"][:, :n], pr["F"], pr["f"])
    with pytest.raises(AssertionError, match="c dim"):
        node.apply_numpy(pr["x0"], pr["C"], pr["cs"][:2], pr["F"], pr["f"])


def _child_main(path):
    import torch  # noqa: F401
    from torch.profiler import profile, ProfilerActivity
    import _native
    ctx = _native.default_context(0)
    res = {}
    for c in CASES:
        pr = problem_of(c)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run(ctx, pr, c["dt"], c["strict"], SHARE_C, c["off"], c["gx_null"], c["gu_null"])
            ctx.sync()
        names = set()
        for e in prof.events():
            names.add(e.name)
        try:
            for e in prof.profiler.kineto_results.events():
                names.add(e.name())
        except AttributeError:
            pass
        res[case_id(c)] = np.array(sorted(k for k in names if "dmpc::" in k))
    np.savez(path, **res)


if __name__ == "__main__" and len(sys.argv) == 3 and sys.argv[1] == "--child":
    _child_main(sys.argv[2])
