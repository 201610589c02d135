#!/usr/bin/env python
"""bench.py - LQR fwd+bwd solves/s (DiffLqr.apply + .backward) on B200, one JSON line.

    python bench.py --gpus N --steps K --warmup W [--workload c5|c2|c3s] [--impl reference] [--dump-outputs DIR]

Metric (BASELINE.json): "LQR fwd+bwd solves/sec"; one solve = one batch element's full
horizon through forward (Riccati + rollout) and the KKT-adjoint backward.
Default workload = BASELINE config 5 shape (n=32, m=8, T=100, fp64), weak-scaled:
8192 elements per GPU, i.e. batch 65536 on 8 GPUs (the full batch is 154 GB of inputs
and does not fit one GPU).  The batch dimension is sharded with no inter-GPU traffic
inside a solve (SURVEY.md §8e) -> "scaling": "weak".

The oracle (oracle/) is imported only for the cpu_baseline leg / --impl reference.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

# the benchmark may run from a read-only tree and must not leave __pycache__ in it
sys.dont_write_bytecode = True

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "chainer-differentiable-mpc_b200")
for p in (ROOT, PKG, os.path.join(PKG, "lqr"), os.path.join(PKG, "mpc"), os.path.join(PKG, "env_dx")):
    if p not in sys.path:
        sys.path.insert(0, p)

WORKLOADS = {
    # name: (n, m, T, B per GPU, description)
    "c5": (32, 8, 100, 8192, "BASELINE config 5: LQR n=32 m=8 T=100 fp64, 8192 elements/GPU (65536 on 8 GPUs)"),
    "c2": (4, 2, 50, 4096, "BASELINE config 2: LQR n=4 m=2 T=50 B=4096 fp64"),
    "c3s": (8, 4, 50, 16384, "BASELINE config 3 shape, unconstrained LQR fwd+bwd n=8 m=4 T=50 B=16384 fp64"),
    "c4s": (3, 1, 20, 8192, "pendulum shape LQR fwd+bwd n=3 m=1 T=20 B=8192/GPU fp64"),
    # BASELINE's second metric (batch-64 MPC-step p50 latency) as its own line: see run_c1
    "c1": (3, 1, 20, 64, "BASELINE config 1: pendulum box-DDP MPC step n=3 m=1 T=20 B=64 (one MPCstep.apply as env_dx/il_exp.py wires it)"),
}


def algorithmic_bytes(n, m, T, w=8):
    """SURVEY.md §8(d): compulsory traffic of fwd+bwd at the operator boundary, per solve."""
    s = n + m
    fwd = w * (n + T * s * s + T * s + (T - 1) * n * s + (T - 1) * n) + w * T * s
    bwd = w * (T * s * s + T * s + (T - 1) * n * s + 2 * T * s) + w * (n + T * s * s + T * s + (T - 1) * n * s + (T - 1) * n)
    return fwd, fwd + bwd


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            v = float(json.load(fh)["hbm_gbs"])
        if v > 0:
            return v, "measured (MEASURED_PEAKS.json)"
    except (OSError, ValueError, KeyError, TypeError):
        pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def kernel_fingerprint():
    """sha256 of the config-5 kernel sources with comments and whitespace removed: traffic.json records the value at
    capture time, so a kernel change after the ncu capture shows up as roofline.traffic_stale instead of going unnoticed."""
    import hashlib
    import re
    h = hashlib.sha256()
    d = os.path.join(ROOT, "chainer-differentiable-mpc_b200", "csrc")
    for name in ("lqr_dmma_warp.cuh", "lqr_dmma_launch.cu", "lqr_adjoint_fused.cuh", "lqr_kernels.cuh"):
        try:
            src = open(os.path.join(d, name)).read()
        except OSError:
            return None
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        src = re.sub(r"//[^\n]*", "", src)
        h.update(re.sub(r"\s+", "", src).encode())
    return h.hexdigest()[:16]


def ncu_traffic_fingerprint():
    try:
        with open(os.path.join(ROOT, "profiles", "r2", "traffic.json")) as fh:
            return json.load(fh).get("_kernel_fingerprint")
    except Exception:
        return None


def ncu_traffic():
    """Measured DRAM bytes per solve of each kernel (one ncu --set full capture each, committed under profiles/)."""
    path = os.path.join(ROOT, "profiles", "r2", "traffic.json")
    try:
        with open(path) as fh:
            return {k: v for k, v in json.load(fh).items() if not k.startswith("_")}
    except Exception:
        return {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._th = None

    def _run_nvml(self):
        """NVML through pynvml (nvidia-ml-py): microseconds per query, so a 0.3 s timed region yields dozens of samples
        (an nvidia-smi subprocess takes ~0.3 s by itself).  Returns False when NVML is not usable."""
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        except Exception:
            return False
        bits = ((pynvml.nvmlClocksThrottleReasonHwSlowdown, 2), (pynvml.nvmlClocksThrottleReasonHwThermalSlowdown, 3),
                (pynvml.nvmlClocksThrottleReasonSwThermalSlowdown, 4), (pynvml.nvmlClocksThrottleReasonSwPowerCap, 5))
        while not self._stop.is_set():
            try:
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                row = [str(sm), str(mx), "Not Active", "Not Active", "Not Active", "Not Active"]
                for bit, col in bits:
                    if r & bit:
                        row[col] = "Active"
                self.rows.append(row)
            except Exception:
                pass
            self._stop.wait(0.005)
        return True

    def _run(self):
        if self._run_nvml():
            self.source = "nvml"
            return
        self.source = "nvidia-smi"
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 6:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop.wait(0.02)

    def start(self):
        self._th = threading.Thread(target=self._run, daemon=True)
        self._th.start()

    def stop(self):
        self._stop.set()
        if self._th:
            self._th.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows), "source": getattr(self, "source", None)}


def elem_rel_err(a, b, floor_frac=1e-3):
    """Element-relative error with an absolute floor (same definition as tests/_helpers.rel_err): max over entries of
    |a-b| / (|b| + floor), floor = floor_frac x the largest magnitude of the entry's own (timestep, element) block (its
    timestep when that block holds fewer than 8 numbers)."""
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    if b.size == 0:
        return 0.0
    ab = np.abs(b)
    gmax = float(np.max(ab))
    if b.ndim >= 3 and int(np.prod(b.shape[2:])) >= 8:
        sl = np.max(ab, axis=tuple(range(2, b.ndim)), keepdims=True)
    elif b.ndim >= 3:
        sl = np.max(ab, axis=tuple(range(1, b.ndim)), keepdims=True)
    elif b.ndim == 2 and b.shape[1] >= 8:
        sl = np.max(ab, axis=1, keepdims=True)
    else:
        sl = gmax
    floor = np.maximum(np.maximum(floor_frac * sl, 1e-6 * gmax), 1e-300)
    d = np.abs(a - b)
    if not np.all(np.isfinite(d)):
        return float("inf")
    return float(np.max(d / (ab + floor)))


def parity_vs_oracle(chunk, n, m, T, k=16):
    """Checker leg (oracle = test infrastructure): the first k batch elements of the TIMED chunk - inputs and the outputs
    the last timed step left in HBM - against the oracle restatement of DiffLqr.apply + .backward."""
    from oracle import lqr as olqr
    pr, out = chunk
    k = min(k, pr["x0"].shape[0])
    h = lambda t: np.ascontiguousarray(t[:, :k].cpu().numpy())
    x0 = pr["x0"][:k].cpu().numpy()
    C, c, F, f, gx, gu = h(pr["C"]), h(pr["c"]), h(pr["F"]), h(pr["f"]), h(pr["gx"]), h(pr["gu"])
    ox, ou, oK, ok = olqr.lqr_solve(x0, C, c, F, f, n, m)
    og = olqr.difflqr_backward(x0, C, c, F, ox, ou, gx, gu, n, m)
    errs = {"x": elem_rel_err(h(out["x"]), ox), "u": elem_rel_err(h(out["u"]), ou), "Ks": elem_rel_err(h(out["Ks"]), oK),
            "ks": elem_rel_err(h(out["ks"]), ok), "dx0": elem_rel_err(out["dx0"][:k].cpu().numpy(), og[0])}
    for name, w in zip(("dC", "dc", "dF", "df"), og[1:]):
        errs[name] = elem_rel_err(h(out[name]), w)
    return {"max_rel": max(errs.values()), "per_output": errs, "elements": k,
            "metric": "element-relative, floor 1e-3 x block max (tests/_helpers.rel_err)",
            "oracle": "oracle/lqr.py (numpy restatement pinned to the live reference by tests/golden/make_golden.py)"}


# --dump-outputs: what DiffLqr.apply (x, u) and .backward (dx0, dC, dc, dF, df) return to a caller -> batch axis
LQR_OUTPUTS = {"x": 1, "u": 1, "dx0": 0, "dC": 1, "dc": 1, "dF": 1, "df": 1}
DUMP_BYTES = 63 * 10 ** 6


def dump_outputs(path, chunks, B):
    """Writes the outputs the last timed step left in HBM to path/<name>.npy (float64), so that two builds can be
    compared output for output.  The full outputs exceed DUMP_BYTES at most workloads (10 GB of dC alone at c5), so a
    fixed seeded sample of batch elements is written, each with its whole horizon; the inputs are seeded too."""
    import torch
    os.makedirs(path, exist_ok=True)
    Bc = chunks[0][1]["x"].shape[1]
    per_elem = sum(chunks[0][1][k].numel() // Bc * 8 for k in LQR_OUTPUTS)
    idx = np.sort(np.random.RandomState(0).choice(B, min(B, DUMP_BYTES // per_elem), replace=False))
    for name, axis in LQR_OUTPUTS.items():
        parts = []
        for i, (_, out) in enumerate(chunks):
            sel = idx[(idx >= i * Bc) & (idx < (i + 1) * Bc)] - i * Bc
            if sel.size:
                t = out[name].index_select(axis, torch.as_tensor(sel, device=out[name].device))
                parts.append(t.cpu().numpy())
        np.save(os.path.join(path, name + ".npy"), np.concatenate(parts, axis=axis))


# ------------------------------------------------------------------------------------- CPU port timing
def cpu_lqr_fwd_bwd(n, m, T, Bc, seed=0):
    """One DiffLqr.apply + .backward with the oracle port (numpy, all BLAS threads)."""
    from oracle import lqr as olqr
    from tests_helpers_local import lqr_problem_np
    pr = lqr_problem_np(seed, T, Bc, n, m)
    rs = np.random.RandomState(1)
    gx, gu = rs.randn(T, Bc, n), rs.randn(T, Bc, m)
    t0, c0 = time.perf_counter(), time.process_time()
    x, u, _, _ = olqr.lqr_solve(pr["x0"], pr["C"], pr["c"], pr["F"], pr["f"], n, m)
    olqr.difflqr_backward(pr["x0"], pr["C"], pr["c"], pr["F"], x, u, gx, gu, n, m)
    dt = time.perf_counter() - t0
    _CPU_USE.append((time.process_time() - c0) / max(dt, 1e-9))       # average number of busy host threads
    return dt


_CPU_USE = []


def cpu_threads_used():
    """Threads the numpy/BLAS port actually kept busy (process CPU time / wall time), at least 1."""
    return max(1, int(round(float(np.mean(_CPU_USE[-3:]))))) if _CPU_USE else 1


def _cpu_worker(args):
    n, m, T, Bc, seed = args
    cpu_lqr_fwd_bwd(n, m, T, min(Bc, 16), seed)          # import + warm-up outside the timed part
    return cpu_lqr_fwd_bwd(n, m, T, Bc, seed)


def cpu_sharded_all_cores(n, m, T, Bc):
    """What process-level batch sharding of the (single-threaded) reference port reaches on this host: one process
    per CPU, each solving its own B_cpu elements concurrently.  Reported beside the faithful single-process number;
    the reference itself has no such sharding."""
    import multiprocessing as mp
    P = max(1, len(os.sched_getaffinity(0)))
    ctx = mp.get_context("spawn")
    with ctx.Pool(P) as pool:
        pool.map(_cpu_worker, [(n, m, T, 8, 100 + i) for i in range(P)])          # spawn + import cost, untimed
        t0 = time.perf_counter()
        pool.map(_cpu_worker, [(n, m, T, Bc, i) for i in range(P)], chunksize=1)
        dt = time.perf_counter() - t0
    # each worker's call includes a 16-element warm-up solve: count those elements too
    return {"value": P * (Bc + min(Bc, 16)) / dt, "unit": "solves/s", "cores": P,
            "how": "%d concurrent processes, each running the oracle port on %d elements" % (P, Bc)}


def reference_under_stub_record(n, m, T):
    """The unmodified reference under the Chainer stub cannot run on the GPU box (/root/reference is absent there); it was
    timed beside the oracle port in the build container (profiles/tools/time_reference_under_stub.py).  Returned as a
    RECORDED annotation of the live port number: port / reference on the same host and inputs."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2", "reference_under_stub.json")) as fh:
            rec = json.load(fh)
        for cse in rec["cases"]:
            if (cse["n"], cse["m"], cse["T"]) == (n, m, T):
                return {"kind": "reference-under-stub (recorded in the build container, not live)",
                        "solves_per_sec_there": cse["solves_per_sec"]["reference_under_stub"],
                        "oracle_port_solves_per_sec_there": cse["solves_per_sec"]["oracle_port"],
                        "port_over_reference": cse["port_over_reference"], "B_cpu": cse["B_cpu"], "host": rec["host"],
                        "tool": "profiles/tools/time_reference_under_stub.py"}
    except Exception:
        pass
    return None


def cpu_sample_batch(n, m, T):
    # sized so one fwd+bwd takes a few seconds on ~8 host cores (BASELINE.md §2)
    return {(32, 8): 128, (8, 4): 1024, (4, 2): 4096, (3, 1): 4096}.get((n, m), 256)


def c1_problem():
    """BASELINE config 1 inputs: pendulum as env_dx/il_env.py:48-70 / pendulum.py:122-145 wires it, u_init = 0."""
    from oracle import mpc as ompc, pendulum as opend
    T, B, n, m = 20, 64, 3, 1
    rs = np.random.RandomState(0)
    th = rs.rand(B) * np.pi - np.pi / 2
    x0 = np.stack((np.cos(th), np.sin(th), rs.rand(B) * 2 - 1), axis=1)
    q = np.array([1.0, 1.0, 0.1, 0.001]); pv = np.array([-1.0, 0.0, 0.0, 0.0])
    C = np.repeat(np.repeat(np.diag(q)[None, None], T, 0), B, 1); c = np.repeat(np.repeat(pv[None, None], T, 0), B, 1)
    lo = np.full((T, B, m), -2.0); hi = np.full((T, B, m), 2.0)
    u = np.zeros((T, B, m))
    x_nom = ompc.get_traj(x0, u, ("pendulum", (10.0, 1.0, 1.0)))
    F, f = opend.linearize(x0, u)
    return dict(C=C, c=c, F=F, f=f, x_nom=x_nom, u=u, lo=lo, hi=hi)


def run_reference_c1(args):
    """Reference arm of `--workload c1`: the oracle port of MPCstep.forward on the host, p50 over --steps calls."""
    import warnings
    from oracle import mpc as ompc
    n, m, T, B, desc = WORKLOADS["c1"]
    pr = c1_problem()
    ts = []
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for _ in range(max(args.warmup, 1) + args.steps):
            t0 = time.perf_counter()
            ompc.step_forward(pr["C"], pr["c"], pr["F"], pr["f"], pr["x_nom"], pr["u"], pr["lo"], pr["hi"], (pr["C"], pr["c"]),
                              ("pendulum", (10.0, 1.0, 1.0)), 0.2, 5, n, m, need_expand=True, coupling="batch")
            ts.append(time.perf_counter() - t0)
    p50 = float(np.median(ts[max(args.warmup, 1):])) * 1e3
    emit({"impl": "reference", "metric": "mpc_step_p50_latency_ms", "value": p50, "unit": "ms", "n_gpus": args.gpus,
          "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": p50, "higher_is_better": False,
          "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
          "config": {"workload": "c1", "desc": desc, "n_state": n, "n_ctrl": m, "T": T, "batch": B, "coupling": "batch"},
          "cpu_baseline": {"value": p50, "unit": "ms", "cores": 1, "kind": "port",
                           "sample": "oracle port of MPCstep.forward (numpy), the same B=64 pendulum step, p50"},
          "e2e": {"value": p50, "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


def run_reference(args):
    n, m, T, Bg, desc = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload == "c1":
        return run_reference_c1(args)
    Bc = cpu_sample_batch(n, m, T)
    for _ in range(max(args.warmup, 1)):
        cpu_lqr_fwd_bwd(n, m, T, Bc)
    times = [cpu_lqr_fwd_bwd(n, m, T, Bc) for _ in range(args.steps)]
    tot = sum(times)
    val = Bc * len(times) / tot
    cores = cpu_threads_used()
    try:
        sharded = cpu_sharded_all_cores(n, m, T, max(Bc // 2, 8))
    except Exception as ex:
        sharded = {"error": repr(ex)[:200]}
    sample = ("oracle port (numpy restatement of DiffLqr.apply+backward, BLAS threads at their default), B_cpu=%d per step, "
              "same n/m/T; %d host CPUs available, %d kept busy on average" % (Bc, os.cpu_count(), cores))
    line = {"impl": "reference", "metric": "lqr_fwd_bwd_solves_per_sec", "value": val, "unit": "solves/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot / len(times),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": args.workload, "desc": desc, "n_state": n, "n_ctrl": m, "T": T, "batch_per_step": Bc},
            "cpu_baseline": {"value": val, "unit": "solves/s", "cores": cores, "kind": "port", "sample": sample,
                             "all_cores_value": sharded.get("value"), "all_cores": sharded.get("cores"),
                             "sharded_all_cores": sharded, "reference_under_stub": reference_under_stub_record(n, m, T)},
            "e2e": {"value": val, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def bind_to_gpu_numa(torch, local):
    """Pin this rank's host threads (and therefore its pinned staging buffers, first-touch) to the CPUs NVML reports
    as local to its GPU, so that the e2e feed does not cross sockets.  Best effort: any failure leaves affinity alone."""
    try:
        import pynvml
        pynvml.nvmlInit()
        props = torch.cuda.get_device_properties(local)
        h = None
        try:
            h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(props.uuid)).encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [i * 64 + b for i, w in enumerate(mask) for b in range(64) if (int(w) >> b) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        if cpus:
            os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:
        return 0


# ------------------------------------------------------------------------------------- GPU arm
def make_problem_torch(torch, dev, n, m, T, B, seed):
    """Synthetic random-stable dynamics, distinct per batch element (SURVEY.md §8d)."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    s = n + m
    f64 = torch.float64
    A = torch.eye(n, dtype=f64, device=dev) + 0.2 * torch.randn(B, n, n, dtype=f64, device=dev, generator=g)
    rho = torch.linalg.eigvals(A).abs().amax(dim=1)
    A = A * torch.clamp(0.95 / rho, max=1.0)[:, None, None]
    Bm = torch.randn(B, n, m, dtype=f64, device=dev, generator=g)
    Fb = torch.cat((A, Bm), dim=2)
    F = Fb[None].expand(T - 1, B, n, s).contiguous()
    L = 0.3 * torch.randn(B, s, s, dtype=f64, device=dev, generator=g)
    Cb = L @ L.transpose(1, 2) + torch.eye(s, dtype=f64, device=dev)
    C = Cb[None].expand(T, B, s, s).contiguous()
    c = torch.randn(T, B, s, dtype=f64, device=dev, generator=g)
    f = 0.1 * torch.randn(T - 1, B, n, dtype=f64, device=dev, generator=g)
    x0 = torch.randn(B, n, dtype=f64, device=dev, generator=g)
    gx = torch.randn(T, B, n, dtype=f64, device=dev, generator=g) / (T * B)
    gu = torch.randn(T, B, m, dtype=f64, device=dev, generator=g) / (T * B)
    return dict(x0=x0, C=C, c=c, F=F, f=f, gx=gx, gu=gu)


def dmma_shape(n, m):
    return (n, m) == (32, 8)


def fp32_step(torch, ctx, chunk, n, m, T, B, stream):
    """fwd+bwd of one chunk through the fp32 API (dtype DMPC_F32): inputs cast to float on the device, outputs checked
    against the fp64 outputs of the same chunk (north_star tolerance 1e-4 relative)."""
    import _native
    pr64, o64 = chunk
    f32 = torch.float32
    pr = {k: v.to(f32) for k, v in pr64.items()}
    o = {k: torch.empty(v.shape, dtype=f32, device=v.device) for k, v in o64.items()}
    P = lambda t: t.data_ptr()
    FULL = _native.LQR_FACTOR | _native.LQR_ROLLOUT | _native.LQR_SAVE_FAC

    def step():
        ctx.lqr_solve(np.float32, T, B, n, m, P(pr["x0"]), P(pr["C"]), P(pr["c"]), P(pr["F"]), T - 1, P(pr["f"]),
                      P(o["x"]), P(o["u"]), P(o["Ks"]), P(o["ks"]), P(o["fac"]), FULL, stream.cuda_stream)
        ctx.lqr_adjoint(np.float32, T, B, n, m, P(pr["C"]), P(pr["c"]), P(pr["F"]), P(o["x"]), P(o["u"]), P(pr["gx"]),
                        P(pr["gu"]), P(o["Ks"]), P(o["fac"]), P(o["dx0"]), P(o["dC"]), P(o["dc"]), P(o["dF"]), P(o["df"]),
                        _native.ADJ_STRICT_REFERENCE, stream.cuda_stream)

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    reps = 6
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    rel = {k: float((o[k].double() - o64[k]).norm() / o64[k].norm()) for k in ("x", "u", "dF")}
    _, tot_b = algorithmic_bytes(n, m, T, w=4)
    return {"dtype": "f32 tensors in HBM, f64 arithmetic in the Riccati sweep (lqr_factor_dmma_warp_kernel<4,float>)",
            "batch": B, "ms_per_step": ms, "solves_per_sec": B / (ms * 1e-3),
            "whole_step_hbm_frac": B * tot_b / (ms * 1e-3) / 1e9 / measured_peaks()[0],
            "rel_err_vs_f64_step": rel, "within_1e-4": all(v < 1e-4 for v in rel.values())}


def run_b200(args):
    import torch
    import _native
    n, m, T, B, desc = WORKLOADS[args.workload]
    if args.batch:
        B = args.batch
    s = n + m
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    n_local_cpus = bind_to_gpu_numa(torch, local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=dev)
    ctx = _native.Context(local)
    f64 = torch.float64
    K = max(1, args.chunks)
    assert B % K == 0, "--chunks must divide the per-GPU batch"
    Bc = B // K
    # K independent sub-batches (contiguous [T,Bc,...] tensors each): fwd(i+1) overlaps bwd(i) on two streams
    chunks = []
    for i in range(K):
        pr = make_problem_torch(torch, dev, n, m, T, Bc, seed=1234 + 1000 * rank + i)
        out = dict(x=torch.empty(T, Bc, n, dtype=f64, device=dev), u=torch.empty(T, Bc, m, dtype=f64, device=dev),
                   Ks=torch.empty(T, Bc, m, n, dtype=f64, device=dev), ks=torch.empty(T, Bc, m, dtype=f64, device=dev),
                   fac=torch.empty(ctx.lqr_fac_elems(T, Bc, n, m), dtype=f64, device=dev),
                   dx0=torch.empty(Bc, n, dtype=f64, device=dev), dC=torch.empty(T, Bc, s, s, dtype=f64, device=dev),
                   dc=torch.empty(T, Bc, s, dtype=f64, device=dev), dF=torch.empty(T - 1, Bc, n, s, dtype=f64, device=dev),
                   df=torch.empty(T - 1, Bc, n, dtype=f64, device=dev))
        chunks.append((pr, out))
    # non-default torch streams: their handles are passed to the C ABI (NULL would mean the library's own
    # stream) and the CUDA events below are recorded on the same streams
    sA = torch.cuda.Stream(device=dev)
    sB = torch.cuda.Stream(device=dev, priority=-1) if K > 1 else sA
    torch.cuda.synchronize()
    P = lambda t: t.data_ptr()

    def fwd(i, stream, flags):
        pr, out = chunks[i]
        ctx.lqr_solve(np.float64, T, Bc, n, m, P(pr["x0"]), P(pr["C"]), P(pr["c"]), P(pr["F"]), T - 1, P(pr["f"]),
                      P(out["x"]), P(out["u"]), P(out["Ks"]), P(out["ks"]), P(out["fac"]), flags, stream.cuda_stream)

    def bwd(i, stream, stage=0):
        pr, out = chunks[i]
        ctx.lqr_adjoint(np.float64, T, Bc, n, m, P(pr["C"]), P(pr["c"]), P(pr["F"]), P(out["x"]), P(out["u"]),
                        P(pr["gx"]), P(pr["gu"]), P(out["Ks"]), P(out["fac"]), P(out["dx0"]), P(out["dC"]),
                        P(out["dc"]), P(out["dF"]), P(out["df"]), _native.ADJ_STRICT_REFERENCE | stage, stream.cuda_stream)

    FULL = _native.LQR_FACTOR | _native.LQR_ROLLOUT | _native.LQR_SAVE_FAC

    def step():
        """fwd+bwd of the whole per-GPU batch; backward of chunk i waits for forward of chunk i."""
        for i in range(K):
            fwd(i, sA, FULL)
            if K > 1:
                ev = torch.cuda.Event()
                ev.record(sA)
                sB.wait_event(ev)
            bwd(i, sB)
        if K > 1:
            ev = torch.cuda.Event()
            ev.record(sB)
            sA.wait_event(ev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # L2 policy (timing rules): the default workload streams 19.5 GB of inputs per step, far beyond the 126 MB L2.
    # The small parity-shaped workloads (c2, c3s, c4s) would fit, so for them a 512 MB buffer is rewritten on the
    # launching stream between timed steps and every step is timed by its own pair of events (flush excluded).
    fwd_b_, tot_b_ = algorithmic_bytes(n, m, T)
    flush_buf = torch.empty(512 << 20, dtype=torch.uint8, device=dev) if B * tot_b_ < (1 << 30) else None

    def flush_l2():
        if flush_buf is not None:
            with torch.cuda.stream(sA):
                flush_buf.fill_(1)

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    # ---- kernel-level durations (serial, chunk 0, events on the launching stream) for the roofline.
    #      "forward" is the launch the timed step really makes (Riccati sweep + rollout fused); the factor-only
    #      and rollout-only launches are timed beside it to split it; "adjoint" = lqr_dtau_kernel + adjoint_out_kernel.
    rsz = ctx.reduced_grad_elems(n, m)
    red = dict(part=torch.empty(Bc, rsz, dtype=f64, device=dev), sums=torch.empty(rsz, dtype=f64, device=dev))

    def bwd_reduced(i, stream):
        pr, out = chunks[i]
        ctx.lqr_adjoint_reduced(np.float64, T, Bc, n, m, P(pr["C"]), P(pr["c"]), P(pr["F"]), P(out["x"]), P(out["u"]),
                                P(pr["gx"]), P(pr["gu"]), P(out["Ks"]), P(out["fac"]), P(out["dc"]), P(red["part"]),
                                P(out["dx0"]), P(red["sums"]), _native.ADJ_STRICT_REFERENCE, stream.cuda_stream)

    kt = {"forward": [], "factor": [], "rollout": [], "adjoint": [], "adjoint_reduced": [], "dtau": [], "adjoint_out": []}
    for _ in range(3):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(8)]
        flush_l2()
        e[0].record(sA)
        fwd(0, sA, FULL); e[1].record(sA)
        bwd(0, sA); e[2].record(sA)
        fwd(0, sA, _native.LQR_FACTOR | _native.LQR_SAVE_FAC); e[3].record(sA)
        fwd(0, sA, _native.LQR_ROLLOUT); e[4].record(sA)
        bwd_reduced(0, sA); e[5].record(sA)
        bwd(0, sA, _native.ADJ_STAGE_DTAU_ONLY); e[6].record(sA)
        bwd(0, sA, _native.ADJ_STAGE_OUT_ONLY); e[7].record(sA)
        torch.cuda.synchronize()
        kt["adjoint_reduced"].append(e[4].elapsed_time(e[5]))
        kt["dtau"].append(e[5].elapsed_time(e[6])); kt["adjoint_out"].append(e[6].elapsed_time(e[7]))
        kt["forward"].append(e[0].elapsed_time(e[1])); kt["adjoint"].append(e[1].elapsed_time(e[2]))
        kt["factor"].append(e[2].elapsed_time(e[3])); kt["rollout"].append(e[3].elapsed_time(e[4]))
    kt = {k: float(np.mean(v)) for k, v in kt.items()}
    # ---- timed region
    sampler = ClockSampler(local)
    sampler.start()
    l0 = ctx.launches
    barrier()
    if flush_buf is None:
        t_start = torch.cuda.Event(enable_timing=True); t_end = torch.cuda.Event(enable_timing=True)
        t_start.record(sA)
        for _ in range(args.steps):
            step()
        t_end.record(sA)
        barrier()
        ms_total = t_start.elapsed_time(t_end)
    else:
        evs = []
        for _ in range(args.steps):
            flush_l2()
            a = torch.cuda.Event(enable_timing=True); b = torch.cuda.Event(enable_timing=True)
            a.record(sA)
            step()
            b.record(sA)
            evs.append((a, b))
        barrier()
        ms_total = sum(a.elapsed_time(b) for a, b in evs)
    launches = ctx.launches - l0
    clocks = sampler.stop()
    if dist is not None:
        tt = torch.tensor([ms_total], dtype=f64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_total = float(tt.item())
    ms_step = ms_total / args.steps
    value = world * B / (ms_step * 1e-3)
    ok = all(bool(torch.isfinite(o["x"]).all().item() and torch.isfinite(o["dF"]).all().item()) for _, o in chunks)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, chunks, B)
    parity = None
    if rank == 0:
        try:
            parity = parity_vs_oracle(chunks[0], n, m, T)
        except Exception as ex:   # report, do not hide
            parity = {"max_rel": None, "error": repr(ex)[:200]}

    line = None
    if rank == 0:
        fwd_b, tot_b = algorithmic_bytes(n, m, T)
        peak, peak_src = measured_peaks()
        traffic = ncu_traffic()
        dmma = dmma_shape(n, m)
        tpe = (n, m) in ((2, 1), (3, 1), (4, 2)) and os.environ.get("DMPC_LQR_GROUP", "0") != "1"   # csrc/lqr_launch.cu
        fwd_name = "lqr_factor_dmma_warp_kernel" if dmma else ("lqr_tpe_kernel" if tpe else "lqr_solve_kernel")
        s_ = n + m
        dtau_b = 8 * (2 * (T - 1) * n * s_ + T * (m * m + n * m) + T * m * n + 2 * T * s_)        # F twice, factors, K, grads, d-tau
        fused_adj = dmma          # n=32/m=8: two-sweep adjoint on the saved V_t, v_t (csrc/lqr_adjoint_fused.cuh)
        k1 = "lqr_dtau_kernel<FUSED>" if fused_adj else ("lqr_dtau_tpe_kernel" if tpe else "lqr_dtau_kernel")
        k2 = "adjoint_fused_kernel" if fused_adj else "adjoint_out_kernel"
        kernels = {
            fwd_name: {"ms": kt["forward"], "launches_per_step": 1, "algorithmic_bytes": Bc * fwd_b,
                       "role": "Riccati sweep + rollout, one launch (factor-only %.3f ms, rollout-only %.3f ms)" % (kt["factor"], kt["rollout"])},
            k1: {"ms": kt["dtau"], "launches_per_step": 1, "algorithmic_bytes": None,
                 "role": ("adjoint sweep 1 (t down): k'_t, v'_t from the saved Quu^-1, Qxu" if fused_adj else
                          "adjoint LQR solve with the saved factors (two sweeps)") + "; its bytes are internal to the adjoint, "
                         "so only measured traffic is reported"},
            k2: {"ms": kt["adjoint_out"], "launches_per_step": 1, "algorithmic_bytes": Bc * (tot_b - fwd_b),
                 "role": ("adjoint sweep 2 (t up): d-tau rollout fused with lambda = V x + v, d-lambda = V dx + v' and " if fused_adj
                          else "lambda / d-lambda recursions + ") + "dC, dc, dF, df, dx0 (carries the adjoint's algorithmic bytes; "
                         "the pair takes %.3f ms)" % kt["adjoint"] +
                         ("; SURVEY 8(d)'s algorithmic figure counts a read of C_t, which the two-sweep adjoint does not need "
                          "(lambda comes from the saved V_t, v_t), so hbm_frac on algorithmic bytes can exceed 1 while the measured "
                          "DRAM traffic stays below the peak" if fused_adj else "")}}
        red_name = ("lqr_dtau_kernel<FUSED>+adjoint_fused_kernel<REDUCE_TB>+reduce_partials_kernel" if fused_adj else
                    ("lqr_dtau_tpe_kernel" if tpe else "lqr_dtau_kernel") + "+adjoint_out_kernel<REDUCE_TB>+reduce_partials_kernel")
        extra_kernels = {red_name: {
            "ms": kt["adjoint_reduced"], "role": "KKT adjoint with the (T,B)-sum of dC,dc,dF,df fused in (shared-parameter "
            "models; not part of the timed step, which materialises the full gradients as the reference does)"}}
        for name, k in kernels.items():
            if k["algorithmic_bytes"]:
                k["achieved_gbs"] = k["algorithmic_bytes"] / (k["ms"] * 1e-3) / 1e9
                k["hbm_frac"] = k["achieved_gbs"] / peak
            tname = name.split("<")[0] + ("_fused1" if name.endswith("<FUSED>") else "")
            k["traffic"] = Bc * traffic[tname]["bytes_per_solve"] if (dmma and tname in traffic) else None
            if k["traffic"]:
                k["traffic_gbs"] = k["traffic"] / (k["ms"] * 1e-3) / 1e9
                k["traffic_hbm_frac"] = k["traffic_gbs"] / peak
        dom = max(kernels, key=lambda x: kernels[x]["ms"])
        whole = B * tot_b / (ms_step * 1e-3) / 1e9
        if dmma and dom == fwd_name:
            # the dominant launch is bound by the FP64 tensor (DMMA) pipe: 400 DMMA m8n8k4 (512 flop) per element-step
            # (DESIGN.md 4.2) = 20.5 Mflop per solve; HBM floor of its algorithmic bytes is lower (see kernels[...])
            flops = 400 * 512 * T
            tf = Bc * flops / (kt["forward"] * 1e-3) / 1e12
            roof = {"bound": "tensor", "kernel": dom, "achieved": tf, "peak": 37.15, "unit": "TFLOP/s", "frac": tf / 37.15,
                    "traffic": kernels[dom]["traffic"],
                    "peak_source": "FP64 DMMA m8n8k4 peak measured on this pool's B200 (profiles/tools/fp64_peak.cu -> "
                                   "profiles/r1/fp64_peak.json); MEASURED_PEAKS.json carries no FP64 figure",
                    "algorithmic_flops_per_launch": Bc * flops,
                    "factor_only_frac": Bc * flops / (kt["factor"] * 1e-3) / 1e12 / 37.15}
        else:
            k = kernels[dom]
            ach = k.get("achieved_gbs") or k.get("traffic_gbs")
            roof = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s",
                    "frac": ach / peak, "traffic": k["traffic"], "peak_source": peak_src}
        roof.update({"hbm_peak_gbs": peak, "hbm_peak_source": peak_src, "kernels": kernels, "other_kernels": extra_kernels,
                     "adjoint_pair": {"ms": kt["adjoint"], "algorithmic_gbs": Bc * (tot_b - fwd_b) / (kt["adjoint"] * 1e-3) / 1e9,
                                      "hbm_frac": Bc * (tot_b - fwd_b) / (kt["adjoint"] * 1e-3) / 1e9 / peak},
                     "chunk_batch": Bc,
                     "whole_step_achieved_gbs": whole, "whole_step_hbm_frac": whole / peak,
                     "algorithmic_bytes_per_solve": {"fwd": fwd_b, "fwd_bwd": tot_b},
                     "traffic_source": "ncu dram__bytes_read+write per solve x launch batch (profiles/r2/traffic.json)",
                     # true when the kernel sources differ from the ones the ncu capture was taken with
                     "traffic_stale": (ncu_traffic_fingerprint() is not None and ncu_traffic_fingerprint() != kernel_fingerprint())})
        line = {"metric": "lqr_fwd_bwd_solves_per_sec", "value": value, "unit": "solves/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": args.workload, "desc": desc, "n_state": n, "n_ctrl": m, "T": T,
                           "batch_per_gpu": B, "global_batch": B * world, "parallelism": "batch-sharded x%d" % world,
                           "chunks_per_gpu": K, "overlap": "fwd(chunk i+1) || bwd(chunk i) on two streams" if K > 1 else "none",
                           "l2": ("inputs (%.1f GB/GPU) larger than L2" % (B * fwd_b / 1e9)) if flush_buf is None else
                                 "512 MB flush buffer rewritten between timed steps (working set %.2f GB/GPU), each step "
                                 "timed by its own event pair" % (B * tot_b / 1e9),
                           "finite_outputs": ok},
                "roofline": roof, "clocks": clocks, "gpu_launches": launches,
                "parity_max_rel": parity["max_rel"], "parity": parity}

    # ---- the one exchange step of a training iteration (SURVEY 8e): (T,B_local)-reduce the learned-dynamics
    #      gradient dF and all-reduce(sum) it over the ranks (NCCL); reported, not part of the solve metric
    exch = None
    if dist is not None:
        ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True); ev2 = torch.cuda.Event(enable_timing=True)
        red_ms, ar_ms = [], []
        for _ in range(8):
            ev0.record(sA)
            bwd_reduced(0, sA)
            ev1.record(sA)
            torch.cuda.current_stream().wait_stream(sA)
            ev1b = torch.cuda.Event(enable_timing=True); ev1b.record()
            dist.all_reduce(red["sums"], op=dist.ReduceOp.SUM)
            ev2.record()
            torch.cuda.synchronize()
            red_ms.append(ev0.elapsed_time(ev1)); ar_ms.append(ev1b.elapsed_time(ev2))
        exch = {"what": "adjoint with fused (T,B)-sum -> %d doubles (dC|dc|dF|df), then NCCL all_reduce(sum)" % rsz,
                "adjoint_reduced_ms": float(np.median(red_ms)), "allreduce_ms": float(np.median(ar_ms)), "world": world}

    # ---- the same step through the fp32 API (SURVEY 8d lists config 5 as "fp64 and fp32"): float tensors, reported
    #      beside the fp64 metric, never instead of it
    fp32 = None
    if dmma_shape(n, m) and world == 1 and not args.no_latency:
        try:
            fp32 = fp32_step(torch, ctx, chunks[0], n, m, T, Bc, sA)
        except Exception as ex:
            fp32 = {"error": repr(ex)[:200]}
        torch.cuda.empty_cache()

    # ---- e2e through the public API with host buffers (rank-local chunk) -----------------
    e2e = None
    try:
        e2e = run_e2e(args, torch, ctx, n, m, T, world, dist, dev, rank)
    except Exception as ex:  # report, do not hide
        e2e = {"value": None, "unit": "solves/s", "error": repr(ex)[:200]}
    e2e_shared = None
    try:
        e2e_shared = run_e2e_shared(args, torch, ctx, n, m, T, world, dist, dev, rank)
    except Exception as ex:
        e2e_shared = {"value": None, "unit": "solves/s", "error": repr(ex)[:200]}
    if rank == 0:
        line["e2e"] = e2e
        line["e2e_shared_params"] = e2e_shared
        if exch is not None:
            line["param_grad_exchange"] = exch
        if fp32 is not None:
            line["fp32_step"] = fp32
        if world == 1 and not args.no_cpu:
            Bcpu = cpu_sample_batch(n, m, T)
            cpu_lqr_fwd_bwd(n, m, T, min(Bcpu, 32))
            tcpu = min(cpu_lqr_fwd_bwd(n, m, T, Bcpu) for _ in range(2))
            sharded = cpu_sharded_all_cores(n, m, T, max(Bcpu // 2, 8))
            line["cpu_baseline"] = {"value": Bcpu / tcpu, "unit": "solves/s", "cores": cpu_threads_used(), "kind": "port",
                                    "host_cpus": os.cpu_count(),
                                    "all_cores_value": sharded.get("value"), "all_cores": sharded.get("cores"),
                                    "sharded_all_cores": sharded,
                                    "reference_under_stub": reference_under_stub_record(n, m, T),
                                    "sample": "oracle port of DiffLqr.apply+backward (numpy, BLAS threads at their default), "
                                              "B_cpu=%d, same n/m/T, best of 2" % Bcpu}
        if world == 1 and not args.no_latency:
            try:
                line["mpc_step_latency"] = mpc_step_latency(ctx, with_cpu=not args.no_cpu)
            except Exception as ex:
                line["mpc_step_latency"] = {"error": repr(ex)[:200]}
            try:
                line["mpc_step_throughput"] = mpc_step_throughput(ctx, torch, dev)
            except Exception as ex:
                line["mpc_step_throughput"] = {"error": repr(ex)[:200]}
    # ---- BASELINE config 4 at this N: every rank runs one IL iteration on its shard, all-reduce inside the timed region
    il = None
    if not args.no_latency:
        try:
            il = il_iteration(dist=dist, dev=dev, rank=rank, world=world, local=local)
        except Exception as ex:
            il = {"error": repr(ex)[:200]}
    if rank == 0:
        if il is not None:
            line["il_iteration"] = il
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def run_e2e(args, torch, ctx, n, m, T, world, dist, dev, rank):
    """Same metric through the reference-facing API (DiffLqr.apply + .backward) with HOST (pinned) numpy
    buffers: H2D of the inputs and D2H of x,u and all gradients are inside the timed region.  The per-GPU
    batch is fed in sub-batches of --e2e-batch; --e2e-workers host threads (one DiffLqr node, context and
    stream each) keep the PCIe link busy in both directions (ctypes releases the GIL during the calls)."""
    import threading
    import _native
    import differentiable_lqr as dl
    Be = args.e2e_batch
    W = max(1, args.e2e_workers)
    s = n + m

    def pinned(shape):
        return torch.empty(shape, dtype=torch.float64).pin_memory().numpy()

    workers = []
    for w in range(W):
        rs = np.random.RandomState(99 + 10 * rank + w)
        C = pinned((T, Be, s, s)); c = pinned((T, Be, s)); F = pinned((T - 1, Be, n, s)); f = pinned((T - 1, Be, n))
        x0 = pinned((Be, n)); gx = pinned((T, Be, n)); gu = pinned((T, Be, m))
        A = np.eye(n) + 0.2 * rs.randn(n, n)
        A *= min(1.0, 0.95 / np.max(np.abs(np.linalg.eigvals(A))))
        F[...] = np.concatenate((A, rs.randn(n, m)), axis=1)[None, None] + 0.01 * rs.randn(1, Be, n, s)
        L = 0.3 * rs.randn(Be, s, s)
        C[...] = (L @ L.transpose(0, 2, 1) + np.eye(s))[None]
        c[...] = rs.randn(T, Be, s); f[...] = 0.1 * rs.randn(T - 1, Be, n); x0[...] = rs.randn(Be, n)
        gx[...] = rs.randn(T, Be, n); gu[...] = rs.randn(T, Be, m)
        wctx = ctx if w == 0 else _native.Context(ctx.device)
        node = dl.DiffLqr(T, Be, n, m, pinned_outputs=True, context=wctx)
        workers.append(dict(node=node, args=(x0, C, c, F, f), g=(gx, gu), ctx=wctx))
    h2d = sum(a.nbytes for a in workers[0]["args"]) + sum(a.nbytes for a in workers[0]["g"])
    d2h = 8 * (T * Be * s + Be * n + T * Be * s * s + T * Be * s + (T - 1) * Be * n * s + (T - 1) * Be * n)

    def one(wk):
        wk["node"].apply_numpy(*wk["args"])
        return wk["node"].backward_numpy(*wk["g"])

    for wk in workers:
        one(wk); one(wk)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    reps = max(2, min(args.steps, 6))
    errs = []

    def loop(wk):
        try:
            for _ in range(reps):
                one(wk)
        except Exception as ex:   # surface worker failures
            errs.append(repr(ex))

    t0 = time.perf_counter()
    ths = [threading.Thread(target=loop, args=(wk,)) for wk in workers]
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if errs:
        raise RuntimeError(errs[0])
    if dist is not None:
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
    return {"value": world * W * Be * reps / dt, "unit": "solves/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "batch_per_call": Be, "host_workers": W, "cpus_bound_to_gpu_numa_node": len(os.sched_getaffinity(0)),
            "api": "DiffLqr.apply_numpy + backward_numpy (pinned host buffers, %d host worker threads)" % W}


def run_e2e_shared(args, torch, ctx, n, m, T, world, dist, dev, rank):
    """The same metric end to end for a SHARED-PARAMETER model (what the reference's callers of DiffLqr actually are:
    LqrNet broadcasts one A|B block, LqrNet_cost_dx also one C, c, over [T, B] with util.expand_time_batch,
    differentiable_lqr.py:186-198, 237-248): the host sends x_init [B,n], ONE parameter block and the upstream gradients
    gx, gu [T,B,.]; the broadcast runs on the device (dmpc_expand_time_batch) and the backward returns the (T,B)-summed
    parameter gradients (dmpc_lqr_adjoint_reduced) plus dx0 - DiffLqr.apply_shared_numpy + backward_reduced_numpy with
    pinned host buffers, H2D and D2H inside the timed region."""
    import threading
    import _native
    import differentiable_lqr as dl
    Be, W = 2048, 2
    s = n + m

    def pinned(shape):
        return torch.empty(shape, dtype=torch.float64).pin_memory().numpy()

    workers = []
    for w in range(W):
        rs = np.random.RandomState(199 + 10 * rank + w)
        x0 = pinned((Be, n)); gx = pinned((T, Be, n)); gu = pinned((T, Be, m))
        A = np.eye(n) + 0.2 * rs.randn(n, n)
        A *= min(1.0, 0.95 / np.max(np.abs(np.linalg.eigvals(A))))
        Fm = np.concatenate((A, rs.randn(n, m)), axis=1)
        L = 0.3 * rs.randn(s, s)
        C = L @ L.T + np.eye(s); c = rs.randn(s); f = 0.1 * rs.randn(n)
        x0[...] = rs.randn(Be, n); gx[...] = rs.randn(T, Be, n) / (T * Be); gu[...] = rs.randn(T, Be, m) / (T * Be)
        wctx = ctx if w == 0 else _native.Context(ctx.device)
        node = dl.DiffLqr(T, Be, n, m, pinned_outputs=True, context=wctx)
        workers.append(dict(node=node, fwd=(x0, C, c, Fm, f), g=(gx, gu)))
    h2d = workers[0]["fwd"][0].nbytes + 8 * (s * s + s + n * s + n) + sum(a.nbytes for a in workers[0]["g"])
    d2h = 8 * (T * Be * s + Be * n + s * s + s + n * s + n)

    def one(wk):
        wk["node"].apply_shared_numpy(*wk["fwd"])
        return wk["node"].backward_reduced_numpy(*wk["g"])

    for wk in workers:
        one(wk); one(wk)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    reps = max(2, min(args.steps, 6))
    errs = []

    def loop(wk):
        try:
            for _ in range(reps):
                one(wk)
        except Exception as ex:
            errs.append(repr(ex))

    t0 = time.perf_counter()
    ths = [threading.Thread(target=loop, args=(wk,)) for wk in workers]
    for th in ths:
        th.start()
    for th in ths:
        th.join()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if errs:
        raise RuntimeError(errs[0])
    if dist is not None:
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
    return {"value": world * W * Be * reps / dt, "unit": "solves/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "batch_per_call": Be, "host_workers": W,
            "api": "DiffLqr.apply_shared_numpy + backward_reduced_numpy: one C, c, A|B, f block broadcast over [T,B] on the "
                   "device, (T,B)-summed parameter gradients back (pinned host buffers, %d host worker threads)" % W}


def mpc_step_latency(ctx, n_calls=200, cpu_calls=10, with_cpu=True, kernel_events=None, dump=None):
    """Second half of BASELINE's metric: batch-64 MPC-step p50 latency on the pendulum
    (config 1: n=3, m=1, T=20, B=64, bounds +-2, as env_dx/il_exp.py wires it).  With `dump`, the x, u the last
    device-resident call computed (what MPCstep.apply returns) are written to dump/<name>.npy."""
    import _native
    from mpc_step import MPCstep
    from util import QuadCost
    from pendulum_dx import PendulumDx
    T, B, n, m = 20, 64, 3, 1
    rs = np.random.RandomState(0)
    th = rs.rand(B) * np.pi - np.pi / 2
    x0 = np.stack((np.cos(th), np.sin(th), rs.rand(B) * 2 - 1), axis=1)
    dx = PendulumDx()
    qv, pv = dx.get_true_obj()
    C = np.repeat(np.repeat(np.diag(qv)[None, None], T, 0), B, 1)
    c = np.repeat(np.repeat(pv[None, None], T, 0), B, 1)
    lo = np.full((T, B, m), -2.0); hi = np.full((T, B, m), 2.0)
    u = np.zeros((T, B, m))
    # nominal trajectory + linearisation on the device (as BoxDDP does each iteration)
    xd = ctx.empty((T, B, n)); Fo = ctx.empty((T - 1, B, 3, 4)); fo = ctx.empty((T - 1, B, 3))
    ctx.get_traj(np.float64, T, B, n, m, _native.DYN_PENDULUM, ctx.to_device(x0), ctx.to_device(u), None, None,
                 (10.0, 1.0, 1.0), xd, Fo, fo)
    x_nom, F, f = xd.download(), Fo.download(), fo.download()

    def facade_call():
        st = MPCstep(controls=u, T=T, u_upper=hi, u_lower=lo, n_batch=B, n_state=n, n_ctrl=m, current_states=x_nom,
                     true_cost=QuadCost(C, c), true_dynamics=dx, ls_decay=0.2, max_ls_iter=5, need_expand=True)
        return st.apply((x0, C, c, F, f))
    for _ in range(10):
        facade_call()
    ts = []
    for _ in range(n_calls):
        t0 = time.perf_counter(); facade_call(); ts.append(time.perf_counter() - t0)
    p50_facade = float(np.median(ts)) * 1e3
    # device-resident: one C-ABI call + stream sync
    d = {k: ctx.to_device(v) for k, v in dict(C=C, c=c, F=F, f=f, x=x_nom, u=u, lo=lo, hi=hi).items()}
    o = dict(x=ctx.empty((T, B, n)), u=ctx.empty((T, B, m)), Ks=ctx.empty((T, B, m, n)), ks=ctx.empty((T, B, m)),
             uf=ctx.empty((T, B, m)), objs=ctx.empty((T, B)), costs=ctx.empty((B,)), old=ctx.empty((B,)),
             al=ctx.empty((B,)), nqp=ctx.empty((T, B), np.int32), fr=ctx.empty((T, B, m), np.uint8),
             nls=ctx.empty((B,), np.int32), fl=ctx.empty((B,), np.int32))

    def dev_call():
        ctx.mpc_step_forward(np.float64, T, B, n, m, d["C"], d["c"], d["F"], T - 1, d["f"], d["x"], d["u"], d["lo"],
                             d["hi"], d["C"], d["c"], _native.DYN_PENDULUM, None, None, (10.0, 1.0, 1.0), 0.2, 64, True,
                             _native.COUPLING_BATCH, o["x"], o["u"], o["Ks"], o["ks"], o["uf"], o["objs"], o["costs"],
                             o["old"], o["al"], o["nqp"], o["fr"], o["nls"], o["fl"])
        ctx.sync()
    for _ in range(10):
        dev_call()
    ts = []
    for _ in range(n_calls):
        t0 = time.perf_counter(); dev_call(); ts.append(time.perf_counter() - t0)
    if dump:
        os.makedirs(dump, exist_ok=True)
        for name in ("x", "u"):
            np.save(os.path.join(dump, name + ".npy"), o[name].download())
    out = {"config": "c1 pendulum n=3 m=1 T=20 B=64 (one MPCstep.apply, need_expand, batch coupling)",
           "p50_ms": p50_facade, "p50_ms_device_resident": float(np.median(ts)) * 1e3, "calls": n_calls,
           "kernel": "mpc_forward_tpe_kernel" if os.environ.get("DMPC_MPC_GROUP") != "1" else "mpc_forward_kernel",
           "h2d_bytes": int(sum(v.nbytes for v in (C, c, F, x_nom, u, lo, hi))), "d2h_bytes": int(8 * (T * B * (n + m + m * n + m + m + 1) + 3 * B)),
           "api": "MPCstep.apply with host numpy buffers (H2D+kernel+D2H) / dmpc_mpc_step_forward + sync"}
    l0 = ctx.launches
    dev_call()
    out["launches"] = ctx.launches - l0
    if kernel_events is not None:      # kernel duration by CUDA events on the launching stream
        torch = kernel_events
        st = torch.cuda.Stream()
        ks = []
        for _ in range(50):
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(st)
            ctx.mpc_step_forward(np.float64, T, B, n, m, d["C"], d["c"], d["F"], T - 1, d["f"], d["x"], d["u"], d["lo"],
                                 d["hi"], d["C"], d["c"], _native.DYN_PENDULUM, None, None, (10.0, 1.0, 1.0), 0.2, 64, True,
                                 _native.COUPLING_BATCH, o["x"], o["u"], o["Ks"], o["ks"], o["uf"], o["objs"], o["costs"],
                                 o["old"], o["al"], o["nqp"], o["fr"], o["nls"], o["fl"], st.cuda_stream)
            e1.record(st)
            torch.cuda.synchronize()
            ks.append(e0.elapsed_time(e1))
        out["kernel_ms"] = float(np.median(ks[5:]))
    if with_cpu:
        from oracle import mpc as ompc
        import warnings
        ts = []
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            for _ in range(cpu_calls + 2):
                t0 = time.perf_counter()
                ompc.step_forward(C, c, F, f, x_nom, u, lo, hi, (C, c), ("pendulum", (10.0, 1.0, 1.0)), 0.2, 5, n, m,
                                  need_expand=True, coupling="batch")
                ts.append(time.perf_counter() - t0)
        out["cpu_port_p50_ms"] = float(np.median(ts[2:])) * 1e3
    return out


def run_c1(args):
    """`--workload c1`: BASELINE's second metric, batch-64 MPC-step p50 latency (one MPCstep.apply on the pendulum).
    value = p50 of one dmpc_mpc_step_forward call + stream sync with every tensor resident in HBM; e2e = p50 of
    MPCstep.apply with host numpy buffers (H2D + kernel + D2H); roofline = the kernel's CUDA-event duration against its
    dependent-chain floor (latency bound: 64 threads cannot fill a GPU; the floor is the length of the longest dependent
    instruction chain x the measured DFMA dependent-issue latency, profiles/r1/fp64_latency.json)."""
    import torch
    import _native
    n, m, T, B, desc = WORKLOADS["c1"]
    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=dev)
    ctx = _native.Context(local)
    sampler = ClockSampler(local); sampler.start()
    lat = mpc_step_latency(ctx, n_calls=args.steps, cpu_calls=10, with_cpu=(rank == 0 and not args.no_cpu), kernel_events=torch,
                           dump=args.dump_outputs if rank == 0 else None)
    clocks = sampler.stop()
    vals = torch.tensor([lat["p50_ms_device_resident"], lat["p50_ms"], lat["kernel_ms"]], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
    p50_dev, p50_api, k_ms = (float(v) for v in vals.tolist())
    if rank == 0:
        try:
            with open(os.path.join(ROOT, "profiles", "r1", "fp64_latency.json")) as fh:
                dfma_clk = float(json.load(fh)["dfma_dep_clk"])
        except Exception:
            dfma_clk = 10.3
        sm_mhz = clocks.get("sm_mhz") or 1900.0
        # longest dependent chain (DFMA-equivalents), counted from csrc/mpc_tpe_kernel.cuh: Riccati step = Taylor shift (4)
        # + V F (3) + F^T Mx (3) + PNQP iteration (~14 incl. two divisions at ~4 each) + K, P, V (5) ~ 30; rollout step =
        # control (5) + pendulum atan2/sin/cos (~70) + quadratic cost (9) ~ 85; three horizon passes (old cost, alpha = 1, and
        # the Riccati sweep) at T = 20
        chain = T * 30 + 2 * T * 85
        floor_ms = chain * dfma_clk / (sm_mhz * 1e3)
        line = {"metric": "mpc_step_p50_latency_ms", "value": p50_dev, "unit": "ms", "n_gpus": world, "steps": lat["calls"],
                "warmup": 10, "ms_per_step": p50_dev, "higher_is_better": False, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": "c1", "desc": desc, "n_state": n, "n_ctrl": m, "T": T, "batch": B, "coupling": "batch",
                           "parallelism": "replicas x%d (a batch-64 step does not shard)" % world,
                           "l2": "latency metric: 0.4 MB working set, L2-resident by nature of the workload (stated, not flushed)"},
                "roofline": {"bound": "latency", "kernel": lat["kernel"], "achieved": k_ms, "peak": floor_ms, "unit": "ms",
                             "frac": floor_ms / k_ms if k_ms else None, "traffic": None,
                             "note": "latency-bound: frac = dependent-chain floor / measured kernel duration; floor = %d dependent "
                                     "DFMA-equivalents x %.1f clk at %.0f MHz" % (chain, dfma_clk, sm_mhz)},
                "e2e": {"value": p50_api, "unit": "ms", "h2d_bytes_per_step": lat["h2d_bytes"], "d2h_bytes_per_step": lat["d2h_bytes"],
                        "api": lat["api"]},
                "clocks": clocks, "gpu_launches": lat["launches"]}
        if "cpu_port_p50_ms" in lat:
            line["cpu_baseline"] = {"value": lat["cpu_port_p50_ms"], "unit": "ms", "cores": 1, "kind": "port",
                                    "sample": "oracle port of MPCstep.forward (numpy), same B=64 step, p50 of 10 calls"}
        emit(line)
    if dist is not None:
        dist.barrier(); dist.destroy_process_group()


def il_iteration(B=8192, reps=3, dist=None, dev=None, rank=0, world=1, local=0):
    """BASELINE config 4 (pendulum imitation learning, batch 65536 sharded over 8 GPUs = 8192 per GPU): ONE training
    iteration as env_dx/il_exp.py:249-302 wires it, on every rank's shard - BoxDDP forward (device-resident loop) through
    the facade with host arrays, backward of loss = mean((u - u_expert)^2) through the final MPCstep with the (T,B)-sum
    fused in -> gradients of the repeated q (diag of C) and p (c) of IL_Env.mpc (il_env.py:120-129), then the ONE
    exchange step of the path: NCCL all-reduce(sum) of those 8 doubles (parallel.allreduce_param_grads), inside the
    timed iteration.  Time = max over ranks; solves/s = world x B / time."""
    import io
    import contextlib
    import warnings
    import parallel
    from box_ddp import BoxDDP
    from util import QuadCost
    from pendulum_dx import PendulumDx
    rs = np.random.RandomState(1000 * rank)        # rank 0 draws exactly the round-1 instance (seed 0)
    th = rs.rand(B) * np.pi - np.pi / 2
    x0 = np.stack((np.cos(th), np.sin(th), rs.rand(B) * 2 - 1), axis=1)
    dx = PendulumDx()
    qv, pv = dx.get_true_obj()
    T = 20
    rp = np.random.RandomState(0); rp.rand(B); rp.rand(B)      # the learner's parameters are shared by all ranks:
    q_learn = qv * (1.0 + 0.1 * rp.randn(4)); p_learn = pv + 0.05 * rp.randn(4)     # rank 0's stream, replayed
    if rank == 0:
        rs.randn(4); rs.randn(4)
    Q = np.repeat(np.repeat(np.diag(q_learn)[None, None], T, 0), B, 1)
    p = np.repeat(np.repeat(p_learn[None, None], T, 0), B, 1)
    u_exp = np.clip(rs.randn(T, B, 1), -2, 2)
    best = None
    for _ in range(reps):
        solver = BoxDDP(T=T, u_lower=dx.lower, u_upper=dx.upper, n_batch=B, n_state=3, n_ctrl=1, u_init=None,
                        eps=dx.mpc_eps, max_iter=500, exit_unconverged=False, detach_unconverged=True,
                        line_search_decay=dx.linesearch_decay, max_line_search_iter=dx.max_linesearch_iter,
                        update_dynamics=False, device=local)
        if dist is not None:
            dist.barrier()
        with warnings.catch_warnings(), contextlib.redirect_stdout(io.StringIO()):
            warnings.simplefilter("ignore")
            t0 = time.perf_counter()
            x, u, costs = solver((x0, QuadCost(Q, p), dx))
            t1 = time.perf_counter()
            un = np.asarray(getattr(u, "array", u))
            gu = 2.0 * (un - u_exp) / (un.size * world)
            g = solver.last_step.backward_reduced_numpy(None, gu)
            t2 = time.perf_counter()
            grads = {"q": np.diag(g[1]).copy(), "p": np.asarray(g[2]).copy()}
            if dist is not None:
                grads = parallel.allreduce_param_grads(grads, device=dev)
            t3 = time.perf_counter()
        dq, dp = grads["q"], grads["p"]
        cur = dict(fwd_ms=1e3 * (t1 - t0), bwd_ms=1e3 * (t2 - t1), allreduce_ms=1e3 * (t3 - t2), total_ms=1e3 * (t3 - t0),
                   n_iter=solver.info["n_iter"], status=solver.info["status"])
        if best is None or cur["total_ms"] < best["total_ms"]:
            best = cur
    if dist is not None:
        import torch
        tt = torch.tensor([best["total_ms"], best["fwd_ms"], best["bwd_ms"], best["allreduce_ms"]], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        best["total_ms"], best["fwd_ms"], best["bwd_ms"], best["allreduce_ms"] = (float(v) for v in tt.tolist())
    best.update({"config": "c4: pendulum IL iteration n=3 m=1 T=20, %d elements/GPU x %d GPU(s): BoxDDP (device loop) + MPCstep "
                           "backward with fused (T,B)-sum + all-reduce of the q, p gradients (%s), host numpy in/out"
                           % (B, world, "NCCL" if dist is not None else "single rank: no exchange"),
                 "n_gpus": world, "global_batch": B * world,
                 "mpc_solves_per_sec": world * B / (best["total_ms"] * 1e-3), "grad_q_finite": bool(np.isfinite(dq).all()),
                 "grad_p_finite": bool(np.isfinite(dp).all()), "timing": "max over ranks of the best of %d iterations" % reps,
                 "allreduce_note": "allreduce_ms is the time spent inside the call = wait for the slowest rank's solve (the ranks "
                                   "hold different instances and share the host's cores) + the transfer; the transfer alone is "
                                   "param_grad_exchange.allreduce_ms"})
    return best


def mpc_step_throughput(ctx, torch, dev, B=16384, reps=5):
    """BASELINE config 3: box-constrained MPC step sweep n=8, m=4, T=50, B=16384, device-resident, element coupling.
    The control bound is calibrated on a 2048-element sub-batch so that about 30 % of the timesteps end with a
    clamped control (SURVEY.md section 8d); the achieved fraction of the full run is reported."""
    import _native
    T, n, m = 50, 8, 4
    f64 = torch.float64
    P = lambda t: t.data_ptr()
    st = torch.cuda.Stream(device=dev)
    sh = st.cuda_stream

    def setup(Bq, bound):
        pr = make_problem_torch(torch, dev, n, m, T, Bq, seed=77)
        g = torch.Generator(device=dev); g.manual_seed(5)
        u = torch.clamp(0.2 * torch.randn(T, Bq, m, dtype=f64, device=dev, generator=g), -bound, bound)
        lo = torch.full((T, Bq, m), -bound, dtype=f64, device=dev); hi = -lo
        x = torch.empty(T, Bq, n, dtype=f64, device=dev)
        torch.cuda.synchronize()
        ctx.get_traj(np.float64, T, Bq, n, m, _native.DYN_LINEAR, P(pr["x0"]), P(u), P(pr["F"]), P(pr["f"]), None, P(x), None, None, sh)
        o = dict(x=torch.empty_like(x), u=torch.empty_like(u), Ks=torch.empty(T, Bq, m, n, dtype=f64, device=dev),
                 ks=torch.empty(T, Bq, m, dtype=f64, device=dev), uf=torch.empty_like(u), objs=torch.empty(T, Bq, dtype=f64, device=dev),
                 costs=torch.empty(Bq, dtype=f64, device=dev), old=torch.empty(Bq, dtype=f64, device=dev),
                 al=torch.empty(Bq, dtype=f64, device=dev), nqp=torch.empty(T, Bq, dtype=torch.int32, device=dev),
                 fr=torch.empty(T, Bq, m, dtype=torch.uint8, device=dev), nls=torch.empty(Bq, dtype=torch.int32, device=dev),
                 fl=torch.empty(Bq, dtype=torch.int32, device=dev))

        def call():
            ctx.mpc_step_forward(np.float64, T, Bq, n, m, P(pr["C"]), P(pr["c"]), P(pr["F"]), T - 1, P(pr["f"]), P(x), P(u),
                                 P(lo), P(hi), P(pr["C"]), P(pr["c"]), _native.DYN_LINEAR, P(pr["F"]), P(pr["f"]), None, 0.2, 64,
                                 True, _native.COUPLING_ELEMENT, P(o["x"]), P(o["u"]), P(o["Ks"]), P(o["ks"]), P(o["uf"]),
                                 P(o["objs"]), P(o["costs"]), P(o["old"]), P(o["al"]), P(o["nqp"]), P(o["fr"]), P(o["nls"]),
                                 P(o["fl"]), sh)

        def clamped():
            torch.cuda.synchronize()
            return float(((o["u"] <= -bound + 1e-8) | (o["u"] >= bound - 1e-8)).any(dim=2).double().mean().item())
        return call, clamped, o, (pr, u, lo, hi, x)

    cal = {}
    for b in (0.6, 0.8, 1.0, 1.2, 1.5):
        call, clamped, _, keep = setup(2048, b)
        call()
        cal[b] = clamped()
    bound = min(cal, key=lambda b: abs(cal[b] - 0.30))
    call, clamped, o, keep = setup(B, bound)
    for _ in range(2):
        call()
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(reps):
        call()
    e1.record(st)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    return {"config": "c3 n=8 m=4 T=50 B=%d box-constrained MPC step (element coupling), bounds +-%.1f" % (B, bound),
            "ms_per_step": ms, "mpc_steps_per_sec": B / (ms * 1e-3), "clamped_timestep_frac": clamped(),
            "bound_calibration": {"%.1f" % b: round(v, 3) for b, v in cal.items()},
            "mean_qp_iters_per_timestep": float(o["nqp"].double().mean().item()),
            "mean_line_search_passes": float(o["nls"].double().mean().item()),
            "flagged_elements": int((o["fl"] != 0).sum().item())}


_REAL_STDOUT = None


def claim_stdout():
    """Rank 0 prints exactly ONE JSON line on stdout.  Libraries write there too (NCCL's version banner, BoxDDP's
    reference-faithful "Converged" prints), so file descriptor 1 is pointed at stderr for the whole run and the JSON
    line goes to a private duplicate of the original stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
        sys.stdout = sys.stderr


def emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c5", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="override per-GPU batch")
    ap.add_argument("--e2e-batch", type=int, default=512)
    ap.add_argument("--e2e-workers", type=int, default=3)
    ap.add_argument("--chunks", type=int, default=1, help="sub-batches per GPU; >1 overlaps fwd(i+1) with bwd(i)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (seeded inputs, a fixed sample of the "
                         "batch, under 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the CUDA path computed; the reference arm runs other inputs")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "c1":
        run_c1(args)
    else:
        run_b200(args)


# tiny local copy of the numpy generator so bench.py does not import from tests/
class _Local:
    @staticmethod
    def lqr_problem_np(seed, T, B, n, m):
        rs = np.random.RandomState(seed)
        s = n + m
        A = np.eye(n) + 0.2 * rs.randn(B, n, n)
        rho = np.max(np.abs(np.linalg.eigvals(A)), axis=1)
        A *= np.minimum(1.0, 0.95 / rho)[:, None, None]
        Fb = np.concatenate((A, rs.randn(B, n, m)), axis=2)
        F = np.repeat(Fb[None], T - 1, axis=0)
        L = 0.3 * rs.randn(B, s, s)
        C = np.repeat((L @ L.transpose(0, 2, 1) + np.eye(s))[None], T, axis=0)
        return dict(x0=rs.randn(B, n), C=C, c=rs.randn(T, B, s), F=F, f=0.1 * rs.randn(T - 1, B, n))


sys.modules["tests_helpers_local"] = _Local

if __name__ == "__main__":
    main()
