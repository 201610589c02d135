"""GPU: LQR batches that share C_t and F_t (dmpc_lqr_solve_shared / dmpc_lqr_adjoint_shared, DiffLqrShared).

The oracle runs the reference recursions (oracle/lqr.py) on the broadcast tensors and sums dC and dF over the batch.
Per-element outputs are compared at rel_err 1e-10 in fp64 (fp32: the suite's 1e-4 / 1e-3 on fp32-rounded inputs); each
entry of dC and dF must lie within 1e-10 (fp32: 2e-5) times sum_b |term| of the oracle's sum, and every case shows from
the oracle that this bound fails when element B-1 or the last step is left out.

Which kernels a case reaches is read from a torch.profiler trace taken in a child process (in a process that has run other
GPU work, the profiler has been seen to return traces without the library's kernels).  The B = 1 matrix sweep selects
the thread-per-element kernels for (2,1), (3,1), (4,2), the specialised group kernel for (8,4), the DMMA warp kernel for
(32,8), and the runtime-shape group kernels with G = 8, 16, 32, 256 otherwise (m > n included); every case then runs
the fwd / adj / reduce kernels of its dtype.  The chunk size NB (64, 32, 16 or 8 elements per CTA) follows B and the
shape; the ragged cases end in a one-element chunk.
"""
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

pytestmark = pytest.mark.gpu

F64, F32 = "f64", "f32"
NP = {F64: np.float64, F32: np.float32}
CNAME = {F64: "double", F32: "float"}


def tol(dt, grad=False):
    return 1e-10 if dt == F64 else (1e-3 if grad else 1e-4)


def sum_tol(dt):
    return 1e-10 if dt == F64 else 2e-5


# ------------------------------------------------------------------------------------------------ problems
def shared_problem(seed, T, B, n, m, F_T, with_f=True, pivot=False, dt=F64):
    """Non-symmetric C_t and F_t that vary with t, shared over the batch; per-element x0, c, f, gx, gu.  The spectral radius
    of A_t stays near 0.9 + 0.1 at every n, so x does not grow over the horizon when F_u is small.  pivot: the control
    block of C is made of 2 x 2 blocks [[0.2, 1], [1.5, 0.3]] and F_u is small, so Quu stays close to C_uu and the
    pivoted elimination swaps rows in every step."""
    rs = np.random.RandomState(seed)
    s = n + m
    L = 0.85 / np.sqrt(s) * rs.randn(T, s, s)
    C = L @ np.swapaxes(L, 1, 2) + np.eye(s) + 0.05 * rs.randn(T, s, s)
    F = np.concatenate((0.9 * np.eye(n) + 0.1 / np.sqrt(n) * rs.randn(F_T, n, n), 0.3 * rs.randn(F_T, n, m)), axis=2)
    if pivot:
        base = np.eye(m)
        for i in range(0, m - 1, 2):
            base[i:i + 2, i:i + 2] = [[0.2, 1.0], [1.5, 0.3]]
        C[:, n:, n:] = base + 0.1 * (C[:, n:, n:] - np.eye(m))
        F[:, :, n:] *= 0.01
    pr = dict(T=T, B=B, n=n, m=m, F_T=F_T, C=C, F=F, c=rs.randn(T, B, s), x0=rs.randn(B, n),
              f=0.1 * rs.randn(T - 1, B, n) if with_f else None, gx=rs.randn(T, B, n), gu=rs.randn(T, B, m))
    if dt == F32:
        pr = {k: (v.astype(np.float32).astype(np.float64) if isinstance(v, np.ndarray) else v) for k, v in pr.items()}
    return pr


def oracle(pr, strict, gx_null=False, gu_null=False):
    T, B, n, m = pr["T"], pr["B"], pr["n"], pr["m"]
    s = n + m
    Cb = np.ascontiguousarray(np.broadcast_to(pr["C"], (B,) + pr["C"].shape).swapaxes(0, 1))
    Fb = np.ascontiguousarray(np.broadcast_to(pr["F"][:T - 1], (B,) + pr["F"][:T - 1].shape).swapaxes(0, 1))
    x, u, _, _ = olqr.lqr_solve(pr["x0"], Cb, pr["c"], Fb, pr["f"], n, m)
    gx = np.zeros((T, B, n)) if gx_null else pr["gx"]
    gu = np.zeros((T, B, m)) if gu_null else pr["gu"]
    dx0, dC, dc, dF, df = olqr.difflqr_backward(pr["x0"], Cb, pr["c"], Fb, x, u, gx, gu, n, m, strict, strict)
    # sum_b |term| bounds, from lambda / d-lambda of the reference recursions (differentiable_lqr.py:87-125)
    tau, dtau = np.concatenate((x, u), 2), dc
    lam, dlam = np.zeros((T, B, n)), np.zeros((T, B, n))
    for t in range(T - 1, -1, -1):
        lam[t] = np.einsum("ij,bj->bi", pr["C"][t][:n], tau[t]) + pr["c"][t][:, :n]
        dlam[t] = np.einsum("ij,bj->bi", pr["C"][t][:n], dtau[t]) + gx[t]
        if t < T - 1:
            lam[t] += np.einsum("ji,bj->bi", pr["F"][t][:, :n], lam[t + 1])
            dlam[t] += np.einsum("ji,bj->bi", pr["F"][t][:, :n], dlam[t + 1])
    a = np.einsum("tbi,tbj->tij", np.abs(dtau), np.abs(tau))
    bC = 0.5 * a + np.swapaxes(a, 1, 2) if strict else 0.5 * (a + np.swapaxes(a, 1, 2))
    sF = np.zeros((pr["F_T"], n, s))
    bF = np.zeros((pr["F_T"], n, s))
    if T > 1:
        sF[:T - 1] = dF.sum(1)
        bF[:T - 1] = (np.einsum("tbi,tbj->tij", np.abs(dlam[1:]), np.abs(tau[:-1])) +
                      np.einsum("tbi,tbj->tij", np.abs(lam[1:]), np.abs(dtau[:-1])))
    return dict(x=x, u=u, dx0=dx0, dc=dc, df=df, dC=dC.sum(1), dF=sF, bC=bC, bF=bF, dC_full=dC, dF_full=dF)


def assert_sum(got, want, bound, eps, what):
    err = np.abs(np.asarray(got, np.float64) - want)
    lim = eps * bound + 1e-300
    worst = float(np.max(err / lim)) if err.size else 0.0
    assert worst <= 1.0, (what, worst)


def assert_bounds_are_sharp(o, eps):
    """Leaving out element B-1, or the last step, moves a sum by more than its bound somewhere."""
    T, B = o["dC_full"].shape[:2]
    lim = lambda b: eps * b + 1e-300
    assert np.max(np.abs(o["dC_full"][:, B - 1]) / lim(o["bC"])) > 1.0
    assert np.max(np.abs(o["dC"][T - 1]) / lim(o["bC"][T - 1])) > 1.0
    if T > 1:
        assert np.max(np.abs(o["dF_full"][:, B - 1]) / lim(o["bF"][:T - 1])) > 1.0
        assert np.max(np.abs(o["dF"][T - 2]) / lim(o["bF"][T - 2])) > 1.0


# ------------------------------------------------------------------------------------------------ device calls
class Bufs:
    """Device tensors `off` elements past the start of a torch allocation (off = 1: aligned to the element type, not to
    16 bytes).  Outputs start as NaN, so an entry the kernels do not write fails the comparison."""

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


def run(ctx, pr, dt, strict, off=0, gx_null=False, gu_null=False, repeat=False):
    """Forward + adjoint through the C ABI; returns a dict of host arrays."""
    import torch
    T, B, n, m, F_T = pr["T"], pr["B"], pr["n"], pr["m"], pr["F_T"]
    s, R = n + m, NP[dt]
    bf = Bufs(off)
    x0, C, c, F = bf.put(pr["x0"], R), bf.put(pr["C"], R), bf.put(pr["c"], R), bf.put(pr["F"], R) if F_T else None
    f = bf.put(pr["f"], R) if pr["f"] is not None else None
    gx = None if gx_null else bf.put(pr["gx"], R)
    gu = None if gu_null else bf.put(pr["gu"], R)
    nb = ctx.lqr_shared_workspace_bytes(R, T, B, n, m)
    ws = bf.empty((nb,), np.uint8)
    o = {k: bf.empty(v, R) for k, v in dict(x=(T, B, n), u=(T, B, m), dx0=(B, n), dC=(T, s, s), dc=(T, B, s),
                                             dF=(F_T, n, s), df=(max(T - 1, 0), B, n)).items()}
    P = {k: bf.ptr(v) for k, v in o.items()}
    torch.cuda.synchronize()
    flags = 1 if strict else 0
    have_df = pr["f"] is not None and T > 1

    def call():
        ctx.lqr_solve_shared(R, T, B, n, m, x0, C, c, F, F_T, f, P["x"], P["u"], bf.ptr(ws), nb)
        ctx.lqr_adjoint_shared(R, T, B, n, m, C, c, F, F_T, P["x"], P["u"], gx, gu, bf.ptr(ws), P["dx0"], P["dC"],
                               P["dc"], P["dF"] if F_T else None, P["df"] if have_df else None, flags, ws_bytes=nb)
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
    for k in ("dx0", "dc"):
        assert rel_err(out[k], o[k]) < tol(dt, True), k
    if pr["f"] is not None and T > 1:
        assert rel_err(out["df"], o["df"]) < tol(dt, True), "df"
    assert_sum(out["dC"], o["dC"], o["bC"], sum_tol(dt), "dC")
    assert_sum(out["dF"], o["dF"], o["bF"], sum_tol(dt), "dF")
    if pr["F_T"] == T:
        assert np.all(out["dF"][T - 1] == 0)
    assert_bounds_are_sharp(o, sum_tol(dt))
    return o


# ------------------------------------------------------------------------------------------------ cases
# (n, m) -> kernel of the B = 1 matrix sweep
SWEEP = {(2, 1): "lqr_tpe_kernel<{R}, 2, 1,", (3, 1): "lqr_tpe_kernel<{R}, 3, 1,", (4, 2): "lqr_tpe_kernel<{R}, 4, 2,",
         (8, 4): "lqr_solve_kernel<{R}, 8, 4, 16>", (32, 8): "lqr_factor_dmma_warp_kernel<4, {R}>",
         (5, 1): "lqr_solve_kernel<{R}, 0, 0, 8>", (3, 9): "lqr_solve_kernel<{R}, 0, 0, 16>",
         (12, 10): "lqr_solve_kernel<{R}, 0, 0, 32>", (40, 24): "lqr_solve_kernel<{R}, 0, 0, 256>"}


def case(n, m, T=17, B=37, dt=F64, F_T=None, with_f=True, strict=True, pivot=None, off=0, gx_null=False, gu_null=False):
    return dict(n=n, m=m, T=T, B=B, dt=dt, F_T=T - 1 if F_T is None else F_T, with_f=with_f, strict=strict,
                pivot=(m >= 2) if pivot is None else pivot, off=off, gx_null=gx_null, gu_null=gu_null)


CASES = ([case(n, m) for (n, m) in SWEEP] +
         [case(n, m, dt=F32) for (n, m) in SWEEP] +
         [case(32, 8, T=100, B=300, F_T=100),                       # config-5 horizon, F with T rows
          case(32, 8, T=100, B=300, with_f=False, strict=False, dt=F32),
          case(32, 8, T=1, B=5, F_T=1), case(32, 8, T=2, B=64, with_f=False, strict=False),
          case(32, 8, T=17, B=1), case(3, 1, T=1, B=3, F_T=0, with_f=False), case(3, 1, T=2, B=2, F_T=2),
          case(4, 2, T=5, B=9473, with_f=False),                     # NB = 64, one-element last chunk
          case(8, 4, T=5, B=4737, strict=False),                     # NB = 32
          case(12, 10, T=9, B=2369),                                 # NB = 16
          case(3, 9, T=9, B=200, strict=False, gx_null=True), case(5, 1, T=9, B=50, gu_null=True),
          case(32, 8, off=1), case(3, 9, off=1, dt=F32), case(40, 24, T=6, B=9, off=1)])


def case_id(c):
    return "{dt}-n{n}m{m}-T{T}-B{B}-FT{F_T}{f}{s}{p}{o}{gx}{gu}".format(
        f="-f" if c["with_f"] else "", s="-strict" if c["strict"] else "", p="-piv" if c["pivot"] else "",
        o="-off1" if c["off"] else "", gx="-gxnull" if c["gx_null"] else "", gu="-gunull" if c["gu_null"] else "", **c)


def problem_of(c):
    seed = (c["n"] * 131 + c["m"] * 17 + c["T"] * 7 + c["B"]) % 100000
    return shared_problem(seed, c["T"], c["B"], c["n"], c["m"], c["F_T"], c["with_f"], c["pivot"], c["dt"])


def expected_kernels(c):
    R = CNAME[c["dt"]]
    sweep = SWEEP[(c["n"], c["m"])]
    if c["off"] and (c["n"], c["m"]) == (32, 8):     # C, F not 16-byte aligned: the DMMA sweep hands over to the group kernel
        sweep = "lqr_solve_kernel<{R}, 32, 8, 256>"
    return [sweep.format(R=R)] + ["lqr_shared_%s_kernel<%s>" % (k, R) for k in ("fwd", "adj", "reduce")]


@pytest.fixture(scope="module")
def ctx():
    import _native
    return _native.default_context(0)


@pytest.mark.parametrize("c", CASES, ids=case_id)
def test_oracle_parity(ctx, c):
    pr = problem_of(c)
    out = run(ctx, pr, c["dt"], c["strict"], c["off"], c["gx_null"], c["gu_null"], repeat=c["B"] == 300)
    check(pr, c["dt"], c["strict"], out, c["gx_null"], c["gu_null"])
    if "again" in out:                                              # a repeated call returns the same bits
        for k, v in out["again"].items():
            assert np.array_equal(v, out[k], equal_nan=True), k


def test_kernels_reached():
    """Every case in a child process under torch.profiler: the sweep kernel its shape selects and the dtype's new kernels
    ran; together the cases reach every sweep family and every instantiation of the new kernels."""
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
        for e in expected_kernels(c):
            assert any(e in k for k in got), (case_id(c), e, got)
        seen |= set(got)
    for R in CNAME.values():
        for k in ("fwd", "adj", "reduce"):
            assert any("lqr_shared_%s_kernel<%s>" % (k, R) in s for s in seen)


def test_cases_cover_every_sweep_family():
    """CPU-side bookkeeping of CASES: every sweep family in both dtypes, m > n, F with T rows, T = 1 and 2, B = 1."""
    for R in (F64, F32):
        assert {(c["n"], c["m"]) for c in CASES if c["dt"] == R} == set(SWEEP)
    assert any(c["m"] > c["n"] for c in CASES) and any(c["F_T"] == c["T"] for c in CASES)
    assert {1, 2, 17, 100} <= {c["T"] for c in CASES} and 1 in {c["B"] for c in CASES}
    assert any(not c["strict"] for c in CASES) and any(not c["with_f"] for c in CASES)


def test_agrees_with_per_element_path(ctx):
    """DiffLqrShared vs DiffLqr.apply_numpy / backward_numpy on the expanded tensors (config-5 shape, T = 20)."""
    from differentiable_lqr import DiffLqr, DiffLqrShared
    T, B, n, m = 20, 96, 32, 8
    pr = shared_problem(7, T, B, n, m, T - 1, pivot=True)
    bc = lambda a: np.ascontiguousarray(np.broadcast_to(a, (B,) + a.shape).swapaxes(0, 1))
    full = DiffLqr(T, B, n, m)
    x1, u1 = full.apply_numpy(pr["x0"], bc(pr["C"]), pr["c"], bc(pr["F"]), pr["f"])
    g1 = full.backward_numpy(pr["gx"], pr["gu"])
    sh = DiffLqrShared(T, B, n, m)
    x2, u2 = sh.apply_numpy(pr["x0"], pr["C"], pr["c"], pr["F"], pr["f"])
    g2 = sh.backward_numpy(pr["gx"], pr["gu"])
    errs = dict(x=rel_err(x2, x1), u=rel_err(u2, u1), dx0=rel_err(g2[0], g1[0]), dc=rel_err(g2[2], g1[2]),
                df=rel_err(g2[4], g1[4]), dC=rel_err(g2[1], g1[1].sum(1)), dF=rel_err(g2[3], g1[3].sum(1)))
    print("shared vs per-element rel_err:", errs)
    assert max(errs.values()) < 1e-11, errs


def test_capacity_full_config5_batch(ctx):
    """T = 100, n = 32, m = 8, B = 65536, fp64 in one call (the broadcast inputs of today's path would need > 150 GB).
    64 sampled elements match the oracle; dC and dF equal the sum of the two half-batch calls within the sum bound."""
    import torch
    T, B, n, m = 100, 65536, 32, 8
    s = n + m
    R = np.float64
    rs = np.random.RandomState(5)
    small = shared_problem(11, T, 1, n, m, T - 1)
    C, F = small["C"], small["F"]
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    g = torch.Generator(device="cuda").manual_seed(3)
    rn = lambda *shape: torch.randn(*shape, generator=g, device="cuda", dtype=torch.float64)
    x0, c, gx, gu = rn(B, n), rn(T, B, s), rn(T, B, n), rn(T, B, m)
    Cd, Fd = dev(C), dev(F)

    def call(lo, hi):
        b = hi - lo
        nb = ctx.lqr_shared_workspace_bytes(R, T, b, n, m)
        ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
        xs, us = [x0[lo:hi].contiguous(), c[:, lo:hi].contiguous(), gx[:, lo:hi].contiguous(), gu[:, lo:hi].contiguous()], None
        x = torch.empty(T, b, n, dtype=torch.float64, device="cuda"); u = torch.empty(T, b, m, dtype=torch.float64, device="cuda")
        dx0 = torch.empty(b, n, dtype=torch.float64, device="cuda"); dc = torch.empty(T, b, s, dtype=torch.float64, device="cuda")
        dC = torch.empty(T, s, s, dtype=torch.float64, device="cuda"); dF = torch.empty(T - 1, n, s, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        ctx.lqr_solve_shared(R, T, b, n, m, xs[0].data_ptr(), Cd.data_ptr(), xs[1].data_ptr(), Fd.data_ptr(), T - 1, None,
                             x.data_ptr(), u.data_ptr(), ws.data_ptr(), nb)
        ctx.lqr_adjoint_shared(R, T, b, n, m, Cd.data_ptr(), xs[1].data_ptr(), Fd.data_ptr(), T - 1, x.data_ptr(),
                               u.data_ptr(), xs[2].data_ptr(), xs[3].data_ptr(), ws.data_ptr(), dx0.data_ptr(),
                               dC.data_ptr(), dc.data_ptr(), dF.data_ptr(), None, 1, ws_bytes=nb)
        ctx.sync()
        del ws
        return x, u, dx0, dc, dC, dF

    x, u, dx0, dc, dC, dF = call(0, B)
    idx = np.sort(rs.choice(B, 64, replace=False))
    idx[-1] = B - 1
    ti = torch.from_numpy(idx).cuda()
    pr = dict(T=T, B=64, n=n, m=m, F_T=T - 1, C=C, F=F, f=None, x0=x0[ti].cpu().numpy(), c=c[:, ti].cpu().numpy(),
              gx=gx[:, ti].cpu().numpy(), gu=gu[:, ti].cpu().numpy())
    o = oracle(pr, True)
    assert rel_err(x[:, ti].cpu().numpy(), o["x"]) < 1e-10 and rel_err(u[:, ti].cpu().numpy(), o["u"]) < 1e-10
    assert rel_err(dx0[ti].cpu().numpy(), o["dx0"]) < 1e-10 and rel_err(dc[:, ti].cpu().numpy(), o["dc"]) < 1e-10
    # sum bounds over the whole batch: |dtau| |tau|^T and |d-lambda| |tau|^T + |lambda| |dtau|^T, lambda from the
    # reference recursion on the device
    tau, dtau = torch.cat((x, u), 2), dc
    a = torch.einsum("tbi,tbj->tij", dtau.abs(), tau.abs())
    bC = (0.5 * a + a.transpose(1, 2)).cpu().numpy()
    lam = torch.zeros(T, B, n, dtype=torch.float64, device="cuda"); dlam = torch.zeros_like(lam)
    for t in range(T - 1, -1, -1):
        lam[t] = tau[t] @ Cd[t][:n].T + c[t][:, :n]
        dlam[t] = dtau[t] @ Cd[t][:n].T + gx[t]
        if t < T - 1:
            lam[t] += lam[t + 1] @ Fd[t][:, :n]
            dlam[t] += dlam[t + 1] @ Fd[t][:, :n]
    bF = (torch.einsum("tbi,tbj->tij", dlam[1:].abs(), tau[:-1].abs()) +
          torch.einsum("tbi,tbj->tij", lam[1:].abs(), dtau[:-1].abs())).cpu().numpy()
    dC, dF = dC.cpu().numpy(), dF.cpu().numpy()
    del x, u, dx0, dc, tau, dtau, lam, dlam
    h1, h2 = call(0, B // 2), call(B // 2, B)
    assert_sum(dC, h1[4].cpu().numpy() + h2[4].cpu().numpy(), bC, 1e-10, "dC")
    assert_sum(dF, h1[5].cpu().numpy() + h2[5].cpu().numpy(), bF, 1e-10, "dF")


def test_lqrnet_training_trace_with_shared_node():
    """The LQRnet notebook (tests/golden/lqrnet_trace.npz: 190 RMSprop updates) through DiffLqrShared: C = I and c = p
    shared, F = the learner's [A B]; the gradient is sum_t dF.  The printed losses are reproduced to 6 digits."""
    from differentiable_lqr import DiffLqrShared
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
    C = np.broadcast_to(np.eye(s), (T, s, s)).copy()
    np.random.seed(2)
    LA = np.eye(n) + 0.2 * np.random.randn(n, n)
    LB = np.random.randn(n, m)
    msA, msB = np.zeros_like(LA), np.zeros_like(LB)
    node = DiffLqrShared(T, B, n, m)
    for i in range(191):
        x0 = np.random.randn(B, n)
        xt, ut = [np.asarray(getattr(v, "array", v)) for v in LqrRecursion(x0, Cb, c, expF, None, T, n, m).solve_recursion()]
        F = np.broadcast_to(np.concatenate((LA, LB), 1), (T - 1, n, s)).copy()
        xp_, up_ = node.apply_numpy(x0, C, c, F, None)
        loss = np.mean((ut - up_) ** 2) + np.mean((xt - xp_) ** 2)
        gsum = node.backward_numpy(-2 * (xt - xp_) / xp_.size, -2 * (ut - up_) / up_.size)[3].sum(0)
        for P, G, ms in ((LA, gsum[:, :n], msA), (LB, gsum[:, n:], msB)):
            ms *= 0.99
            ms += 0.01 * G * G
            P -= 1e-2 * G / (np.sqrt(ms) + 1e-8)
        ml = np.mean((LA - A) ** 2) + np.mean((LB - Bm) ** 2)
        if i in want:
            assert abs(loss - want[i][0]) < 1e-6 and abs(ml - want[i][1]) < 1e-6, (i, loss, ml)


@pytest.mark.parametrize("F_T,with_f", [(4, True), (5, False)])
def test_facade_gradient_shapes(F_T, with_f):
    from differentiable_lqr import DiffLqrShared
    T, B, n, m = 5, 7, 4, 2
    pr = shared_problem(3, T, B, n, m, F_T, with_f)
    node = DiffLqrShared(T, B, n, m, strict_reference=False)
    x, u = node.apply((pr["x0"], pr["C"], pr["c"], pr["F"], pr["f"]))
    x, u = np.asarray(getattr(x, "array", x)), np.asarray(getattr(u, "array", u))
    g = node.backward((0, 1, 2, 3, 4), (pr["gx"], pr["gu"]))
    g = [None if v is None else np.asarray(getattr(v, "array", v)) for v in g]
    assert g[0].shape == (B, n) and g[1].shape == (T, s_ := n + m, s_) and g[2].shape == (T, B, s_)
    assert g[3].shape == (F_T, n, s_)
    assert (g[4] is None) == (not with_f) and (g[4] is None or g[4].shape == (T - 1, B, n))
    o = oracle(pr, False)
    assert rel_err(x, o["x"]) < 1e-10 and rel_err(g[2], o["dc"]) < 1e-10
    assert_sum(g[1], o["dC"], o["bC"], 1e-10, "dC")
    assert_sum(g[3], o["dF"], o["bF"], 1e-10, "dF")


def test_errors(ctx):
    import ctypes
    lib, h = ctx.lib, ctx.h
    T, B, n, m = 4, 3, 3, 2
    sz = ctypes.c_size_t(0)
    assert lib.dmpc_lqr_shared_workspace_bytes(0, 0, B, n, m, ctypes.byref(sz)) == 1
    assert lib.dmpc_lqr_shared_workspace_bytes(0, T, B, n, m, None) == 1
    assert lib.dmpc_lqr_shared_workspace_bytes(0, T, B, n, 33, ctypes.byref(sz)) == 5
    assert lib.dmpc_lqr_shared_workspace_bytes(0, T, B, 400, 8, ctypes.byref(sz)) == 5
    assert lib.dmpc_lqr_shared_workspace_bytes(7, T, B, n, m, ctypes.byref(sz)) == 5
    assert lib.dmpc_lqr_shared_workspace_bytes(0, T, B, n, m, ctypes.byref(sz)) == 0
    nb = sz.value
    ws = ctx.empty((nb,), np.uint8)
    bufs = [ctx.empty((4096,), np.float64) for _ in range(12)]
    p = [b.ptr for b in bufs]
    solve = lambda **k: lib.dmpc_lqr_solve_shared(h, k.get("dt", 0), k.get("T", T), B, n, k.get("m", m), p[0], p[1], p[2],
                                                  k.get("F", p[3]), k.get("F_T", T - 1), None, k.get("x", p[4]), p[5],
                                                  ws.ptr, k.get("nb", nb), None)
    assert solve() == 0
    assert solve(T=0) == 1 and solve(F_T=T + 1) == 1 and solve(nb=nb - 1) == 1
    assert solve(F=None) == 6 and solve(x=None) == 6
    assert solve(m=40) == 5 and solve(dt=3) == 5
    adj = lambda **k: lib.dmpc_lqr_adjoint_shared(h, 0, T, B, n, m, p[1], p[2], p[3], k.get("F_T", T - 1), p[4], p[5],
                                                  None, None, ws.ptr, k.get("nb", nb), p[6], k.get("dC", p[7]), p[8],
                                                  k.get("dF", p[9]), None, 1, None)
    assert adj() == 0
    assert adj(nb=16) == 1 and adj(F_T=T - 2) == 1 and adj(dC=None) == 6 and adj(dF=None) == 6
    ctx.sync()
    for b in bufs:
        b.free()
    ws.free()
    from differentiable_lqr import DiffLqrShared
    pr = shared_problem(1, T, B, n, m, T - 1)
    node = DiffLqrShared(T, B, n, m)
    for bad, msg in ((dict(C=pr["C"][:, None]), "C dim"), (dict(c=pr["c"][:, :1]), "c dim"), (dict(F=pr["F"][:, :2]), "F dim"),
                     (dict(f=pr["f"][:1]), "f dim")):
        args = dict(x0=pr["x0"], C=pr["C"], c=pr["c"], F=pr["F"], f=pr["f"])
        args.update(bad)
        with pytest.raises(AssertionError, match=msg):
            node.apply_numpy(args["x0"], args["C"], args["c"], args["F"], args["f"])


def _child_main(path):
    import torch  # noqa: F401
    from torch.profiler import profile, ProfilerActivity
    import _native
    ctx = _native.default_context(0)
    res = {}
    for c in CASES:
        pr = problem_of(c)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run(ctx, pr, c["dt"], c["strict"], c["off"], c["gx_null"], c["gu_null"])
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
