"""bench.py obeys the driver's contract: exactly one JSON line on stdout with the required keys (GPU arm and the
CPU reference arm), on the smoke-sized workload."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches")


def _run(*extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "small", "--steps", "3",
                          "--warmup", "3", *extra], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, out.stdout
    return json.loads(lines[0])


def test_gpu_arm_line():
    d = _run()
    for key in REQUIRED + ("clocks", "roofline", "cpu_baseline"):
        assert key in d, key
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["dtype"] == "f64" and d["higher_is_better"] is True
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and "workload" in d["config"]
    assert d["value"] > 0 and abs(d["value"] - 1024 / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]
    assert d["gpu_launches"] > 0
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 8 * 1024 * (2 * 64 + 50) and e["d2h_bytes_per_step"] == 8 * 1024 * 64
    r = d["roofline"]
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and r["peak"] > 10 and 0 < r["frac"] < 1.2
    c = d["cpu_baseline"]
    # "reference" when the unmodified reference files travelled in baseline/_ref/ (oracle/stage_reference.py), else the port
    assert c["kind"] in ("reference", "port") and c["cores"] >= 1 and c["value"] > 0 and c["sample"] and c["J_sample"] == 1024
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    # the correctness probe of the timed step: hk through the Gram identity, 128 particles of U_next from the definition
    p = d["parity"]
    assert p["ok"] is True and p["hk_rel"] <= 1e-10 and p["probe_rel"] <= 1e-10 and p["tol"] == 1e-10


def test_dump_outputs_are_the_timed_step_and_repeat(tmp_path):
    """--dump-outputs writes what the last timed step returned (U_next, hk, the four metrics) in float64; the seeded
    inputs make a second run with the same arguments write the same outputs."""
    import numpy as np

    runs = []
    for name in ("a", "b"):
        d = _run("--steps", "2", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / name))
        assert d["steps"] == 2
        runs.append({f[:-4]: np.load(str(tmp_path / name / f)) for f in os.listdir(str(tmp_path / name))})
    a, b = runs
    assert sorted(a) == ["U_next", "bias", "bias-data", "hk", "self-bias", "self-bias-data"]
    assert a["U_next"].shape == (64, 1024) and a["hk"].shape == (1,) and all(v.dtype == np.float64 for v in a.values())
    assert np.isfinite(a["U_next"]).all() and a["hk"][0] > 0
    for key in a:
        assert np.abs(a[key] - b[key]).max() <= 1e-12 * np.abs(a[key]).max(), key


def test_reference_arm_line():
    d = _run("--impl", "reference")
    for key in REQUIRED + ("impl", "cpu_baseline"):
        assert key in d, key
    assert d["impl"] == "reference" and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["e2e"]["value"] == d["value"] == d["cpu_baseline"]["value"]
    assert d["config"]["J_sample"] == d["cpu_baseline"]["J_sample"] == 1024 and d["cpu_baseline"]["cores"] >= 1


def test_cfg1_run_line():
    """--workload cfg1: BASELINE.json configs[0] through sampling.run(T=1000) (ces/calibrate.py:270-416)."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg1", "--no-cpu-baseline"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    for key in REQUIRED + ("roofline",):
        assert key in d, key
    # (the whole run is ONE launch of small_run_kernel: forward map + update + stopping rule per iteration on the device)
    assert d["steps"] == 1000 and d["config"]["J"] == 100 and d["value"] > 0 and d["e2e"]["value"] > 0 and d["gpu_launches"] >= 1
    # the run converges to the analytic posterior mean of the notebook problem (linear.ipynb:695-697)
    assert abs(d["posterior_mean"][0] + 1.0367) < 0.1 and abs(d["posterior_mean"][1] - 2.0870) < 0.1


def test_darcy_workload_line():
    """--workload cfg2 (one ensemble Kalman iteration including the batched Darcy forward solve) prints the same contract
    line; its roofline object describes the CG solver."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg2", "--steps", "2", "--warmup", "3",
                          "--no-cpu-baseline"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    for key in REQUIRED + ("clocks", "roofline"):
        assert key in d, key
    assert d["config"]["grid"] == 64 and d["config"]["J"] == 1024 and d["config"]["update"] == "eki"
    assert d["value"] > 0 and d["gpu_launches"] > 0 and d["e2e"]["value"] > 0
    r = d["roofline"]
    assert "darcy_pcg_tile_kernel" in r["kernel"] and 0 < r["frac"] < 1 and 0.3 < r["share_of_step"] < 1
    assert 20 < r["cg_iterations_mean"] < 400
