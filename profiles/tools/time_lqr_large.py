"""Large-system LQR (DESIGN.md §4.8): device-resident forward, adjoint and reduced adjoint at (64, 16) T=100 B=2048 and
(128, 32) T=50 B=1024, fp64 and fp32, against the same Riccati recursion written with torch (batched matmul +
torch.linalg.solve per step, fp64).

CUDA events on one stream after a warm-up of every call; the library calls and the torch forward alternate, REPS rounds
of one call each, and the median is kept.  The inputs (C, F alone are 2.3-13 GB) are far larger than the 126 MB L2.
Model flops and bytes come from the shapes (the per element-step model of DESIGN §4.8); the achieved FP64 rate is
reported against the 37.2 TFLOP/s DMMA peak measured in profiles/r1/fp64_peak.json.  The torch forward's Ks / x are
compared with the library's.  Writes profiles/r3/lqr_large_timing.json (or argv[1]) with the card's name, power limit
and max SM clock read in the same run.  Options: --small runs a tiny shape end to end (no timing claims).
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

PEAK_FP64 = 37.2e12
REPS = 5


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def model(n, m, T, B, w):
    s = n + m
    fl = 2 * n * n * (s + 1) + 2 * s * n * (s + 1) + 2 * m * m * (n + 1 + m) + 2 * m * m * (n + 1) + 2 * m ** 3 / 3 + 4 * m * n * (n + 1)
    by = w * ((s * s + s + n * s + n) + (2 * m * n + m + m * m + n * n + n))
    return fl * T * B, by * T * B


def torch_forward(C, c, F, f, x0, n, m):
    """The Riccati recursion of lqr_solve_kernel with batched torch ops, fp64: Ks, ks, then the rollout."""
    T = C.shape[0]
    V = v = None
    Ks, ks = [None] * T, [None] * T
    for t in range(T - 1, -1, -1):
        Q, q = C[t], c[t]
        if t < T - 1:
            Ft = F[t]
            Q = Q + Ft.transpose(1, 2) @ (V @ Ft)
            q = q + (Ft.transpose(1, 2) @ ((V @ f[t].unsqueeze(2)).squeeze(2) + v).unsqueeze(2)).squeeze(2)
        Quu, Qux, qu = Q[:, n:, n:], Q[:, n:, :n], q[:, n:]
        sol = torch.linalg.solve(Quu, -torch.cat((Qux, qu.unsqueeze(2)), 2))
        K, k = sol[:, :, :n], sol[:, :, n]
        Ks[t], ks[t] = K, k
        if t > 0:
            Qxu = Q[:, :n, n:]
            P = torch.cat((Qux, qu.unsqueeze(2)), 2) + Quu @ sol
            Vv = torch.cat((Q[:, :n, :n], q[:, :n].unsqueeze(2)), 2) + Qxu @ sol + K.transpose(1, 2) @ P
            V, v = Vv[:, :, :n], Vv[:, :, n]
    x = x0
    xs = []
    for t in range(T):
        u = (Ks[t] @ x.unsqueeze(2)).squeeze(2) + ks[t]
        xs.append(x)
        if t < T - 1:
            x = (F[t] @ torch.cat((x, u), 1).unsqueeze(2)).squeeze(2) + f[t]
    return torch.stack(Ks), torch.stack(xs)


def run_shape(ctx, n, m, T, B, dt, st):
    s = n + m
    R = torch.float64 if dt == np.float64 else torch.float32
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(0)
    rn = lambda *sh: torch.randn(*sh, generator=g, device=dev, dtype=torch.float64)
    with torch.cuda.stream(st):
        L = rn(T, B, s, s) * (0.85 / s ** 0.5)
        C = L @ L.transpose(2, 3)
        del L
        C += torch.eye(s, device=dev, dtype=torch.float64)
        F = torch.cat((0.9 * torch.eye(n, device=dev, dtype=torch.float64).expand(T - 1, B, n, n) + rn(T - 1, B, n, n) * (0.1 / n ** 0.5),
                       0.3 * rn(T - 1, B, n, m)), 3)
        c, f, x0 = rn(T, B, s), 0.1 * rn(T - 1, B, n), rn(B, n)
        gx, gu = rn(T, B, n), rn(T, B, m)
        Cr, cr, Fr, fr, x0r, gxr, gur = (a.to(R).contiguous() for a in (C, c, F, f, x0, gx, gu))
        if dt != np.float64:
            del C, F
        e = lambda *sh: torch.empty(*sh, device=dev, dtype=R)
        x, u, Ks, ks = e(T, B, n), e(T, B, m), e(T, B, m, n), e(T, B, m)
        fac = e(ctx.lqr_fac_elems(T, B, n, m))
        dx0, dC, dc, dF, df = e(B, n), e(T, B, s, s), e(T, B, s), e(T - 1, B, n, s), e(T - 1, B, n)
        rsz = ctx.reduced_grad_elems(n, m)
        part, sums, wdt, rdx0 = e(B, rsz), e(rsz), e(T, B, s), e(B, n)
    P = lambda t: t.data_ptr()
    S = st.cuda_stream
    calls = {
        "forward": lambda: ctx.lqr_solve(dt, T, B, n, m, P(x0r), P(Cr), P(cr), P(Fr), T - 1, P(fr), P(x), P(u), P(Ks),
                                         P(ks), P(fac), _native.LQR_FACTOR | _native.LQR_ROLLOUT | _native.LQR_SAVE_FAC, stream=S),
        "adjoint": lambda: ctx.lqr_adjoint(dt, T, B, n, m, P(Cr), P(cr), P(Fr), P(x), P(u), P(gxr), P(gur), P(Ks), P(fac),
                                           P(dx0), P(dC), P(dc), P(dF), P(df), 0, stream=S),
        "adjoint_reduced": lambda: ctx.lqr_adjoint_reduced(dt, T, B, n, m, P(Cr), P(cr), P(Fr), P(x), P(u), P(gxr), P(gur),
                                                           P(Ks), P(fac), P(wdt), P(part), P(rdx0), P(sums), 0, stream=S),
    }
    arms = dict(calls)
    if dt == np.float64:
        arms["torch_forward"] = lambda: torch_forward(C, c, F, f, x0, n, m)
    times = {k: [] for k in arms}
    with torch.cuda.stream(st):
        for k, fn in arms.items():                                  # warm-up of every call
            fn()
        st.synchronize()
        for _ in range(REPS):
            for k, fn in arms.items():
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(st)
                out = fn()
                b.record(st)
                st.synchronize()
                times[k].append(a.elapsed_time(b))
                if k == "torch_forward":
                    tK, tx = out
    fl, by = model(n, m, T, B, 8 if dt == np.float64 else 4)
    res = dict(n=n, m=m, T=T, B=B, dtype=np.dtype(dt).name, model_flops_forward=fl, model_bytes_forward=by,
               forward_dmma_floor_ms=fl / PEAK_FP64 * 1e3, forward_hbm_floor_ms_at_7_7TBs=by / 7.7e12 * 1e3)
    for k, v in times.items():
        res[k + "_ms_median"] = float(np.median(v))
        res[k + "_ms_all"] = [float(t) for t in v]
    res["forward_fp64_rate_tflops"] = fl / (res["forward_ms_median"] * 1e-3) / 1e12
    res["forward_fraction_of_dmma_peak"] = res["forward_fp64_rate_tflops"] * 1e12 / PEAK_FP64
    if dt == np.float64:
        res["torch_forward_fp64_rate_tflops"] = fl / (res["torch_forward_ms_median"] * 1e-3) / 1e12
        scale = lambda a: float(torch.max(torch.abs(a)))
        res["torch_vs_library_Ks_maxabs_over_maxabs"] = float(torch.max(torch.abs(tK - Ks))) / scale(tK)
        res["torch_vs_library_x_maxabs_over_maxabs"] = float(torch.max(torch.abs(tx - x))) / scale(tx)
    return res


def main():
    small = "--small" in sys.argv
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    out = args[0] if args else os.path.join(ROOT, "profiles", "r3", "lqr_large_timing.json")
    ctx = _native.Context(0)
    st = torch.cuda.Stream(device=torch.device("cuda", 0))
    shapes = [(64, 16, 100, 2048), (128, 32, 50, 1024)] if not small else [(64, 16, 3, 4)]
    rec = dict(card=card(), note="CUDA events, median of %d alternating rounds; model per DESIGN.md 4.8" % REPS, results=[])
    for n, m, T, B in shapes:
        for dt in (np.float64, np.float32):
            r = run_shape(ctx, n, m, T, B, dt, st)
            print(json.dumps(r), flush=True)
            rec["results"].append(r)
            torch.cuda.empty_cache()
            ctx.trim()
    os.makedirs(os.path.dirname(out), exist_ok=True)
    with open(out, "w") as fh:
        json.dump(rec, fh, indent=1)


if __name__ == "__main__":
    main()
