"""bench.py's output contract (host logic, no GPU): the reference arm really runs here (it is the oracle port on host cores),
and the recorded B200 lines under profiles/r1 carry every key the driver reads."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config"}


def _last_json_line(text):
    lines = [ln for ln in text.strip().splitlines() if ln.startswith("{")]
    assert len(lines) == 1, "stdout must carry exactly one JSON line"
    return json.loads(lines[0])


def test_reference_arm_runs_on_host_cores_and_prints_one_line():
    env = dict(os.environ, OMP_NUM_THREADS="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c2",
                          "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = _last_json_line(out.stdout)
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["metric"] == "lqr_fwd_bwd_solves_per_sec" and d["unit"] == "solves/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["vs_baseline"] is None and d["dtype"] == "f64"
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"] == "c2" and d["steps"] == 1


@pytest.mark.gpu
def test_dump_outputs_writes_what_the_timed_steps_computed(tmp_path):
    T, B, n, m = 50, 256, 4, 2
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c2", "--batch", str(B), "--steps", "2",
                          "--warmup", "1", "--no-cpu", "--no-latency", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = _last_json_line(out.stdout)
    assert d["steps"] == 2 and d["parity_max_rel"] < 1e-9
    s = n + m
    # 256 elements fit the size cap: the whole batch is written
    shapes = {"x": (T, B, n), "u": (T, B, m), "dx0": (B, n), "dC": (T, B, s, s), "dc": (T, B, s), "dF": (T - 1, B, n, s),
              "df": (T - 1, B, n)}
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted(k + ".npy" for k in shapes)
    for name, shape in shapes.items():
        a = np.load(tmp_path / (name + ".npy"))
        assert a.dtype == np.float64 and a.shape == shape and np.isfinite(a).all(), name


def test_b200_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)


def test_recorded_b200_lines_carry_the_contract_keys():
    for name, n in (("bench_n1.json", 1), ("bench_n8.json", 8)):
        with open(os.path.join(ROOT, "profiles", "r1", name)) as fh:
            d = _last_json_line(fh.read())
        assert BASE_KEYS <= set(d), name
        assert d["n_gpus"] == n and d["scaling"] == "weak" and d["config"]["workload"] == "c5"
        assert d["gpu_launches"] > 0 and d["warmup"] >= 3
        r = d["roofline"]
        assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r)
        assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
        assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
        assert not ({"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(d["clocks"]["reasons"]))
        e = d["e2e"]
        assert e["value"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] < d["value"]
        if n == 1:
            cb = d["cpu_baseline"]
            assert {"value", "unit", "cores", "kind", "sample"} <= set(cb) and cb["kind"] == "port"
