"""Shared C / F batch: device-resident fwd+bwd of today's path against the shared-parameter path.

  today : dmpc_expand_time_batch (C, F) -> dmpc_lqr_solve (FACTOR|ROLLOUT|SAVE_FAC) -> dmpc_lqr_adjoint_reduced
  shared: dmpc_lqr_solve_shared -> dmpc_lqr_adjoint_shared

Both on the same inputs (C_t, F_t shared, c, f, x0, gx, gu per element), at the config-5 shape (n=32, m=8, T=100,
B=8192) and the config-2 shape (n=4, m=2, T=50, B=4096), fp64.  CUDA events on one stream after warm-up; the two paths
alternate in one process (REPS rounds of ITERS calls each).  The matrix sweep (the B = 1 dmpc_lqr_solve inside the
shared forward) is timed on its own.  Outputs are checked against each other: x, u, dx0 and sum dF / sum dC.
Writes profiles/r3/lqr_shared_timing.json (or the path given as argv[1]) with the card name and power limit.
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "chainer-differentiable-mpc_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import _native  # noqa: E402

REPS, ITERS = 5, 10
ctx = _native.Context(0)
dev = torch.device("cuda", 0)
st = torch.cuda.Stream(device=dev)
S = st.cuda_stream
P = lambda t: t.data_ptr()
R = np.float64


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def run_shape(n, m, T, B):
    s = n + m
    g = torch.Generator(device=dev).manual_seed(1)
    rn = lambda *sh: torch.randn(*sh, generator=g, device=dev, dtype=torch.float64)
    L = 0.3 * rn(T, s, s)
    C = L @ L.transpose(1, 2) + torch.eye(s, device=dev, dtype=torch.float64) + 0.05 * rn(T, s, s)
    F = torch.cat((0.9 * torch.eye(n, device=dev, dtype=torch.float64) + 0.05 * rn(T - 1, n, n), 0.3 * rn(T - 1, n, m)), 2)
    x0, c, f, gx, gu = rn(B, n), rn(T, B, s), 0.1 * rn(T - 1, B, n), rn(T, B, n), rn(T, B, m)
    e = lambda *sh: torch.empty(*sh, device=dev, dtype=torch.float64)
    # today's path: broadcast C, F on the device, then the per-element solve and the fused-reduction adjoint
    Cb, Fb, xa, ua, Ks, ks = e(T, B, s, s), e(T - 1, B, n, s), e(T, B, n), e(T, B, m), e(T, B, m, n), e(T, B, m)
    fac = e(ctx.lqr_fac_elems(T, B, n, m))
    rsz = ctx.reduced_grad_elems(n, m)
    dtau, part, dx0a, sums = e(T, B, s), e(B, rsz), e(B, n), e(rsz)

    def today():
        expand(Cb, C, T, s * s)
        expand(Fb, F, T - 1, n * s)
        ctx.lqr_solve(R, T, B, n, m, P(x0), P(Cb), P(c), P(Fb), T - 1, P(f), P(xa), P(ua), P(Ks), P(ks), P(fac),
                      _native.LQR_FACTOR | _native.LQR_ROLLOUT | _native.LQR_SAVE_FAC, S)
        ctx.lqr_adjoint_reduced(R, T, B, n, m, P(Cb), P(c), P(Fb), P(xa), P(ua), P(gx), P(gu), P(Ks), P(fac), P(dtau),
                                P(part), P(dx0a), P(sums), _native.ADJ_STRICT_REFERENCE, S)

    def expand(dst, src, rows, count):
        # dst[t, b, :] = src[t, :]: C_t and F_t vary with t, so every time row is broadcast over B on its own
        for t in range(rows):
            ctx.expand_time_batch(R, 1, B, P(src) + 8 * t * count, P(dst) + 8 * t * B * count, count, S)

    nb = ctx.lqr_shared_workspace_bytes(R, T, B, n, m)
    ws = torch.empty(nb, dtype=torch.uint8, device=dev)
    xs, us, dx0s, dc, dC, dF, df = e(T, B, n), e(T, B, m), e(B, n), e(T, B, s), e(T, s, s), e(T - 1, n, s), e(T - 1, B, n)

    def shared():
        ctx.lqr_solve_shared(R, T, B, n, m, P(x0), P(C), P(c), P(F), T - 1, P(f), P(xs), P(us), P(ws), nb, S)
        ctx.lqr_adjoint_shared(R, T, B, n, m, P(C), P(c), P(F), T - 1, P(xs), P(us), P(gx), P(gu), P(ws), P(dx0s), P(dC),
                               P(dc), P(dF), P(df), _native.ADJ_STRICT_REFERENCE, ws_bytes=nb, stream=S)

    # the matrix sweep alone: the B = 1 dmpc_lqr_solve the shared forward starts with
    c1, K1, k1 = torch.zeros(T, 1, s, device=dev, dtype=torch.float64), e(T, 1, m, n), e(T, 1, m)
    fac1 = e(ctx.lqr_fac_elems(T, 1, n, m))

    def sweep():
        ctx.lqr_solve(R, T, 1, n, m, None, P(C), P(c1), P(F), T - 1, None, None, None, P(K1), P(k1), P(fac1),
                      _native.LQR_FACTOR | _native.LQR_SAVE_FAC, S)

    def timed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        for _ in range(ITERS):
            fn()
        b.record(st)
        b.synchronize()
        return a.elapsed_time(b) / ITERS

    launches = {}
    with torch.cuda.stream(st):
        for name, fn in (("today", today), ("shared", shared), ("matrix_sweep", sweep)):
            n0 = ctx.launches
            fn()
            launches[name] = ctx.launches - n0
        st.synchronize()
        t_today, t_shared, t_sweep = [], [], []
        for _ in range(REPS):
            t_today.append(timed(today))
            t_shared.append(timed(shared))
            t_sweep.append(timed(sweep))
        st.synchronize()
    sF = sums[s * s + s:s * s + s + n * s].view(n, s)
    sC = sums[:s * s].view(s, s)
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))
    agree = dict(x=rel(xs, xa), u=rel(us, ua), dx0=rel(dx0s, dx0a), sum_dF=rel(dF.sum(0), sF), sum_dC=rel(dC.sum(0), sC))
    med = lambda v: float(np.median(v))
    return dict(shape=dict(n=n, m=m, T=T, B=B, dtype="float64"),
                today_ms=dict(median=med(t_today), all=t_today),
                shared_ms=dict(median=med(t_shared), all=t_shared),
                matrix_sweep_ms=dict(median=med(t_sweep), all=t_sweep),
                speedup=med(t_today) / med(t_shared), max_rel_diff=agree,
                launches=launches, workspace_bytes=nb)


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3", "lqr_shared_timing.json")
    res = dict(card=card(), method="CUDA events on one stream, %d alternating rounds of %d calls after one warm-up call "
                                    "of each path; median per call" % (REPS, ITERS),
               config5=run_shape(32, 8, 100, 8192), config2=run_shape(4, 2, 50, 4096))
    os.makedirs(os.path.dirname(out), exist_ok=True)
    with open(out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
