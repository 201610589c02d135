"""Batch-shared c (DMPC_SHARE_C) and the LqrNet_cost_dx link on it, timed against the routes they replace.

1. Device resident, fp64, fwd+bwd, f None, C_t / F_t / c_t shared by the batch:
     broadcast c: dmpc_lqr_solve_shared + dmpc_lqr_adjoint_shared with c expanded to [T,B,s] (dc per element)
     shared c   : dmpc_lqr_solve_shared_ex + dmpc_lqr_adjoint_shared_ex with share = DMPC_SHARE_C (c [T,s], dc summed)
   at the config-5 shape (n=32, m=8, T=100, B=8192) and the config-2 shape (n=4, m=2, T=50, B=4096).  CUDA events on
   one stream after one warm-up call of each; the two alternate in one process (REPS rounds of ITERS calls), median.
2. One LqrNet_cost_dx training step through the host-array API (forward + backward_numpy, host arrays in and out):
     old link: util.expand_time_batch of C, c and [A B] on the host, DiffLqr.apply_numpy on the [T,B,...] tensors,
               DiffLqr.backward_reduced_numpy (what LqrNet_cost_dx ran before it moved to DiffLqrShared; restated here)
     new link: LqrNet_cost_dx.forward + backward_numpy (DiffLqrShared, c [T,s], f None)
   at the config-5 shape with B = 1024, and with B = 8192 when the host has the memory the old route's broadcast needs
   (otherwise the entry records that it was skipped and why).  Wall clock around whole steps (each ends in a
   device-to-host copy), the two alternating, median of REPS rounds.
3. Outputs of each pair compared: x, u, dx0 and the summed gradients (max |a - b| / max |b|).
Writes profiles/r3/lqrnet_shared_timing.json (or argv[1]) with the card name and power limit from nvidia-smi.
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
PKG = os.path.join(ROOT, "chainer-differentiable-mpc_b200")
sys.path[:0] = [ROOT, PKG, os.path.join(PKG, "lqr")]
import numpy as np  # noqa: E402
import torch  # noqa: E402
import _native  # noqa: E402
import differentiable_lqr as dl  # noqa: E402
from util import expand_time_batch  # noqa: E402

REPS, ITERS = 7, 10
R = np.float64


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), 1e-300))


def device_pair(ctx, n, m, T, B):
    dev = torch.device("cuda", 0)
    st = torch.cuda.Stream(device=dev)
    S = st.cuda_stream
    P = lambda t: t.data_ptr()
    s = n + m
    g = torch.Generator(device=dev).manual_seed(1)
    rn = lambda *sh: torch.randn(*sh, generator=g, device=dev, dtype=torch.float64)
    L = 0.3 * rn(T, s, s)
    C = L @ L.transpose(1, 2) + torch.eye(s, device=dev, dtype=torch.float64) + 0.05 * rn(T, s, s)
    F = torch.cat((0.9 * torch.eye(n, device=dev, dtype=torch.float64) + 0.05 * rn(T - 1, n, n), 0.3 * rn(T - 1, n, m)), 2)
    x0, cs, gx, gu = rn(B, n), rn(T, s), rn(T, B, n), rn(T, B, m)
    cb = cs[:, None].expand(T, B, s).contiguous()
    e = lambda *sh: torch.empty(*sh, device=dev, dtype=torch.float64)
    out = {}
    for name, share, c, dc in (("broadcast_c", None, cb, e(T, B, s)), ("shared_c", _native.SHARE_C, cs, e(T, s))):
        nb = ctx.lqr_shared_workspace_bytes(R, T, B, n, m, share)
        out[name] = dict(share=share, c=c, dc=dc, ws=torch.empty(nb, dtype=torch.uint8, device=dev), nb=nb,
                         x=e(T, B, n), u=e(T, B, m), dx0=e(B, n), dC=e(T, s, s), dF=e(T - 1, n, s))

    def call(o):
        ctx.lqr_solve_shared(R, T, B, n, m, P(x0), P(C), P(o["c"]), P(F), T - 1, None, P(o["x"]), P(o["u"]), P(o["ws"]),
                             o["nb"], S, share=o["share"])
        ctx.lqr_adjoint_shared(R, T, B, n, m, P(C), P(o["c"]), P(F), T - 1, P(o["x"]), P(o["u"]), P(gx), P(gu), P(o["ws"]),
                               P(o["dx0"]), P(o["dC"]), P(o["dc"]), P(o["dF"]), None, _native.ADJ_STRICT_REFERENCE,
                               ws_bytes=o["nb"], stream=S, share=o["share"])

    def timed(o):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        for _ in range(ITERS):
            call(o)
        b.record(st)
        b.synchronize()
        return a.elapsed_time(b) / ITERS

    launches, times = {}, {k: [] for k in out}
    with torch.cuda.stream(st):
        for k, o in out.items():
            n0 = ctx.launches
            call(o)
            launches[k] = ctx.launches - n0
        st.synchronize()
        for _ in range(REPS):
            for k, o in out.items():
                times[k].append(timed(o))
        st.synchronize()
    a, b = out["shared_c"], out["broadcast_c"]
    h = lambda t: t.cpu().numpy()
    agree = dict(x=rel(h(a["x"]), h(b["x"])), u=rel(h(a["u"]), h(b["u"])), dx0=rel(h(a["dx0"]), h(b["dx0"])),
                 dC=rel(h(a["dC"]), h(b["dC"])), dF=rel(h(a["dF"]), h(b["dF"])), dc=rel(h(a["dc"]), h(b["dc"].sum(1))))
    med = lambda v: float(np.median(v))
    res = dict(shape=dict(n=n, m=m, T=T, B=B, dtype="float64", f=None), launches=launches, max_rel_diff=agree,
               speedup=med(times["broadcast_c"]) / med(times["shared_c"]))
    for k in out:
        res[k + "_ms"] = dict(median=med(times[k]), all=times[k])
        res[k + "_workspace_bytes"] = out[k]["nb"]
    return res


def make_net(T, B, n, m):
    net = dl.LqrNet_cost_dx(T, B, n, m, 6)
    # a stable A and a well-conditioned C: at n = 32 the seeded I + 0.2 randn lets x grow over 100 steps
    A = np.eye(n) + 0.1 / np.sqrt(n) * np.random.RandomState(1).randn(n, n)
    net.A.array[...] = A * (0.9 / np.max(np.abs(np.linalg.eigvals(A))))
    net.C.array[...] = np.eye(n + m) + 0.05 * np.random.RandomState(2).randn(n + m, n + m)
    return net


def old_link_step(node, net, x0, gx, gu):
    """LqrNet_cost_dx as it was: host broadcast over [T, B], DiffLqr, fused (T,B)-sum in the adjoint."""
    T, B, n = net.T, net.n_batch, net.n_state
    AB = np.concatenate((net.A.array, net.B.array), axis=1)
    large_f = expand_time_batch(AB, T - 1, B)
    C = expand_time_batch(net.C.array, T, B)
    c = expand_time_batch(net.c.array, T, B)
    x, u = node.apply_numpy(x0, C, c, large_f, None)
    g = node.backward_reduced_numpy(gx, gu)
    return x, u, g[0], (g[3][:, :n].copy(), g[3][:, n:].copy(), g[1].copy(), g[2].copy())


def new_link_step(net, x0, gx, gu):
    x, u = [np.asarray(getattr(v, "array", v)) for v in net.forward((x0, None))]
    return x, u, [a.copy() for a in net.backward_numpy(gx, gu)]


def mem_available():
    try:
        with open("/proc/meminfo") as fh:
            for line in fh:
                if line.startswith("MemAvailable:"):
                    return int(line.split()[1]) * 1024
    except OSError:
        pass
    return None


def link_pair(n, m, T, B, reps):
    s = n + m
    old_bytes = 8 * (T * B * s * s + T * B * s + (T - 1) * B * n * s)    # the host broadcast of C, c and [A B]
    avail = mem_available()
    need = 2 * old_bytes + 8 * 4 * T * B * s                              # broadcast + its contiguous copy, x/u/gx/gu
    shape = dict(n=n, m=m, T=T, B=B, dtype="float64", f=None)
    if avail is not None and avail < need:
        return dict(shape=shape, skipped="host has %.1f GB available, the old route needs about %.1f GB"
                    % (avail / 1e9, need / 1e9))
    rs = np.random.RandomState(3)
    x0, gx, gu = rs.randn(B, n), rs.randn(T, B, n) / (T * B), rs.randn(T, B, m) / (T * B)
    net = make_net(T, B, n, m)
    node = dl.DiffLqr(T, B, n, m)
    o = old_link_step(node, net, x0, gx, gu)                              # warm-up (allocations) and the comparison
    nw = new_link_step(net, x0, gx, gu)
    dx0_new = net.lqr_layer.backward_numpy(gx, gu)[0]
    names = ("dA", "dB", "dC", "dc")
    agree = dict(x=rel(nw[0], o[0]), u=rel(nw[1], o[1]), dx0=rel(dx0_new, o[2]),
                 **{k: rel(a, b) for k, a, b in zip(names, nw[2], o[3])})
    t_old, t_new = [], []
    for _ in range(reps):
        t0 = time.perf_counter(); old_link_step(node, net, x0, gx, gu); t_old.append(time.perf_counter() - t0)
        t0 = time.perf_counter(); new_link_step(net, x0, gx, gu); t_new.append(time.perf_counter() - t0)
    med = lambda v: float(np.median(v)) * 1e3
    return dict(shape=shape, old_link_ms=dict(median=med(t_old), all=[1e3 * v for v in t_old]),
                new_link_ms=dict(median=med(t_new), all=[1e3 * v for v in t_new]),
                speedup=med(t_old) / med(t_new), max_rel_diff=agree, old_route_host_broadcast_bytes=old_bytes)


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3", "lqrnet_shared_timing.json")
    ctx = _native.default_context(0)
    res = dict(card=card(),
               method_device="CUDA events on one stream, %d alternating rounds of %d calls after one warm-up call of "
                             "each; median per fwd+bwd" % (REPS, ITERS),
               method_link="host wall clock around whole training steps (forward + backward_numpy, host arrays), "
                           "one warm-up step of each, then alternating rounds; median per step",
               device_config5=device_pair(ctx, 32, 8, 100, 8192), device_config2=device_pair(ctx, 4, 2, 50, 4096),
               link_config5_B1024=link_pair(32, 8, 100, 1024, REPS),
               link_config5_B8192=link_pair(32, 8, 100, 8192, 3))
    os.makedirs(os.path.dirname(out), exist_ok=True)
    with open(out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
