"""Large-system MPC step (DESIGN.md §4.9): device-resident forward, backward and reduced backward of the box-constrained
MPC step, and one BoxDDP solve with LinDx, at (64, 16) T=50 B=1024 and (128, 32) T=20 B=256, fp64 and fp32, with bounds
that clamp about a quarter of the controls.

CUDA events on one stream after a warm-up of every call; the calls alternate, REPS rounds of one call each, and the
median is kept.  The inputs (C and F alone are 1.3-2.9 GB) are far larger than the 126 MB L2.  Model flops come from the
shapes and the measured PNQP iterations / line-search passes (the per element-step model of DESIGN §4.9); the achieved
FP64 rate is reported against the 37.2 TFLOP/s DMMA peak of profiles/r1/fp64_peak.json.  Beside each time: the CPU oracle
port's (oracle/mpc.py, numpy) time per element for the same step, run on a few elements.  Writes
profiles/r3/mpc_large_timing.json (or argv[1]) with the card's name, power limit and max SM clock read in the same run.
Options: --small runs a tiny shape end to end (no timing claims).
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "chainer-differentiable-mpc_b200"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import _native  # noqa: E402
from oracle import mpc as ompc  # noqa: E402

PEAK_FP64 = 37.2e12
REPS = 5
ORACLE_ELEMS = 2


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def model_forward(n, m, T, B, qp_iters, ls_passes):
    """Flops of one forward: the §4.8 Riccati step (no factor cache), PNQP at m^3/3 + 2 m^2 per iteration, and
    2 (s^2 + n s + m n) per line-search pass and step."""
    s = n + m
    ric = 2 * n * n * (s + 1) + 2 * s * n * (s + 1) + 2 * m * m * (n + 1) + 4 * m * n * (n + 1)
    return (ric * T + (m ** 3 / 3 + 2 * m * m) * qp_iters + 2 * (s * s + n * s + m * n) * T * ls_passes) * B


def run_shape(ctx, n, m, T, B, dt, st):
    s = n + m
    R = torch.float64 if dt == np.float64 else torch.float32
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(0)
    rn = lambda *sh: torch.randn(*sh, generator=g, device=dev, dtype=torch.float64)
    e = lambda *sh, d=R: torch.empty(*sh, device=dev, dtype=d)
    S = st.cuda_stream
    P = lambda t: None if t is None else t.data_ptr()
    with torch.cuda.stream(st):
        L = rn(T, B, s, s) * (0.85 / s ** 0.5)
        C = L @ L.transpose(2, 3)
        del L
        C += torch.eye(s, device=dev, dtype=torch.float64)
        F = torch.cat((0.9 * torch.eye(n, device=dev, dtype=torch.float64).expand(T - 1, B, n, n) + rn(T - 1, B, n, n) * (0.1 / n ** 0.5),
                       0.3 * rn(T - 1, B, n, m)), 3)
        c, f, x0 = rn(T, B, s), 0.1 * rn(T - 1, B, n), rn(B, n)
        un = 0.1 * rn(T, B, m)
        Cr, cr, Fr, fr, x0r, unr = (a.to(R).contiguous() for a in (C, c, F, f, x0, un))
        xn = e(T, B, n)
        ctx.get_traj(dt, T, B, n, m, _native.DYN_LINEAR, P(x0r), P(unr), P(Fr), P(fr), None, P(xn), stream=S)
        o = dict(x=e(T, B, n), u=e(T, B, m), Ks=e(T, B, m, n), ks=e(T, B, m), uf=e(T, B, m), objs=e(T, B), costs=e(B),
                 old=e(B), al=e(B), nqp=e(T, B, d=torch.int32), free=e(T, B, m, d=torch.uint8), nls=e(B, d=torch.int32),
                 fl=e(B, d=torch.int32))
        big = torch.full((T, B, m), 1e6, device=dev, dtype=R)
        lo, hi = -big, big

    def fwd():
        ctx.mpc_step_forward(dt, T, B, n, m, P(Cr), P(cr), P(Fr), T - 1, None, P(xn), P(unr), P(lo), P(hi), P(Cr), P(cr),
                             _native.DYN_LINEAR, P(Fr), P(fr), None, 0.2, 64, True, _native.COUPLING_ELEMENT, P(o["x"]),
                             P(o["u"]), P(o["Ks"]), P(o["ks"]), P(o["uf"]), P(o["objs"]), P(o["costs"]), P(o["old"]),
                             P(o["al"]), P(o["nqp"]), P(o["free"]), P(o["nls"]), P(o["fl"]), stream=S)

    with torch.cuda.stream(st):                       # bounds at the 75 % quantile of |u| of an unconstrained step
        fwd()
        st.synchronize()
        b = float(torch.quantile(o["u"].abs().double().flatten()[:1 << 24], 0.75))
        lo = torch.full((T, B, m), -b, device=dev, dtype=R)
        hi = torch.full((T, B, m), b, device=dev, dtype=R)
        fwd()
        st.synchronize()
        clamped = float(((o["u"] - lo).abs() <= 1e-8).logical_or((o["u"] - hi).abs() <= 1e-8).double().mean())
        gx, gu = rn(T, B, n).to(R), rn(T, B, m).to(R)
        rsz = ctx.reduced_grad_elems(n, m)
        w = dict(K=e(T, B, m, n), k=e(T, B, m), d=e(T, B, s), act=e(T, B, m, d=torch.uint8), dx0=e(B, n), dC=e(T, B, s, s),
                 dc=e(T, B, s), dF=e(T - 1, B, n, s), part=e(B, rsz), sums=e(rsz))
        bo = dict(x=e(T, B, n), u=e(T, B, m), c=e(B), du=e(B))
        u0 = torch.zeros(T, B, m, device=dev, dtype=R)
    calls = {
        "forward": fwd,
        "backward": lambda: ctx.mpc_step_backward(dt, T, B, n, m, P(Cr), P(cr), P(Fr), T - 1, P(o["x"]), P(o["u"]), P(lo),
                                                  P(hi), P(gx), P(gu), P(w["K"]), P(w["k"]), P(w["d"]), P(w["act"]),
                                                  P(w["dx0"]), P(w["dC"]), P(w["dc"]), P(w["dF"]), None, stream=S),
        "backward_reduced": lambda: ctx.mpc_step_backward_reduced(dt, T, B, n, m, P(Cr), P(cr), P(Fr), T - 1, P(o["x"]),
                                                                  P(o["u"]), P(lo), P(hi), P(gx), P(gu), P(w["K"]),
                                                                  P(w["k"]), P(w["d"]), P(w["act"]), P(w["part"]),
                                                                  P(w["dx0"]), P(w["sums"]), stream=S),
    }
    box_iters = []

    def box():
        r = ctx.boxddp_solve(dt, T, B, n, m, P(x0r), P(Cr), P(cr), P(lo), P(hi), _native.DYN_LINEAR, P(Fr), T - 1, P(fr),
                             None, P(u0), 1e-5, 1e-4, 0.2, 5, 5, 64, _native.COUPLING_ELEMENT, P(bo["x"]), P(bo["u"]),
                             P(bo["c"]), P(bo["du"]), None, stream=S)
        box_iters.append(r[0])
    calls["boxddp_solve_5_iter_max"] = box
    times = {k: [] for k in calls}
    with torch.cuda.stream(st):
        for fn in calls.values():
            fn()
        st.synchronize()
        for _ in range(REPS):
            for k, fn in calls.items():
                a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(st)
                fn()
                b_.record(st)
                st.synchronize()
                times[k].append(a.elapsed_time(b_))
    qp_iters = float(o["nqp"].double().sum()) / B
    ls_passes = float(o["nls"].double().mean())
    fl = model_forward(n, m, T, B, qp_iters, ls_passes)
    res = dict(n=n, m=m, T=T, B=B, dtype=np.dtype(dt).name, share_of_controls_on_a_bound=clamped,
               mean_pnqp_iterations_per_element_over_horizon=qp_iters, mean_line_search_passes=ls_passes,
               boxddp_iterations=box_iters[-1], model_flops_forward=fl, forward_dmma_floor_ms=fl / PEAK_FP64 * 1e3)
    for k, v in times.items():
        res[k + "_ms_median"] = float(np.median(v))
        res[k + "_ms_all"] = [float(t) for t in v]
    res["forward_fp64_rate_tflops"] = fl / (res["forward_ms_median"] * 1e-3) / 1e12
    res["forward_fraction_of_dmma_peak"] = res["forward_fp64_rate_tflops"] * 1e12 / PEAK_FP64
    # the CPU oracle port on the first ORACLE_ELEMS elements of the same step, per element
    h = lambda t: t[:, :ORACLE_ELEMS].double().cpu().numpy() if t.dim() > 2 else t[:ORACLE_ELEMS].double().cpu().numpy()
    Cn, cn, Fn, fn_, xnn, unn, lon, hin = (h(a) for a in (Cr, cr, Fr, fr, xn, unr, lo, hi))
    t0 = time.perf_counter()
    ox, ou, _, _ = ompc.step_forward(Cn, cn, Fn, None, xnn, unn, lon, hin, (Cn, cn), ("linear", Fn, fn_), 0.2, 64, n, m, True,
                                     coupling="element")
    t1 = time.perf_counter()
    ompc.step_backward(Cn, cn, Fn, None, ox, ou, lon, hin, h(gx), h(gu), n, m)
    t2 = time.perf_counter()
    res["cpu_oracle_forward_ms_per_element"] = (t1 - t0) * 1e3 / ORACLE_ELEMS
    res["cpu_oracle_backward_ms_per_element"] = (t2 - t1) * 1e3 / ORACLE_ELEMS
    res["gpu_forward_ms_per_element"] = res["forward_ms_median"] / B
    res["gpu_backward_ms_per_element"] = res["backward_ms_median"] / B
    return res


def main():
    small = "--small" in sys.argv
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    out = args[0] if args else os.path.join(ROOT, "profiles", "r3", "mpc_large_timing.json")
    ctx = _native.Context(0)
    st = torch.cuda.Stream(device=torch.device("cuda", 0))
    shapes = [(64, 16, 50, 1024), (128, 32, 20, 256)] if not small else [(64, 16, 3, 4)]
    rec = dict(card=card(), note="CUDA events, median of %d alternating rounds; model per DESIGN.md 4.9" % REPS, results=[])
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
