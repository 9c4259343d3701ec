"""Cost of noise='ensemble' against the reference's Cholesky noise (DESIGN.md section 4g).

Both modes are timed alternately in one process (>= 3 repeats each; mean, min and max are reported), after a warm-up of
each.  Per workload: ms per step, the noise pass alone (between the ``noise:begin`` / ``noise:end`` timeline marks of one
extra step), the noise GEMM's rate 2 p J_l J_g / (pass - fill) and the fill's share of the pass (the fills of the same
panels timed on their own).  Update workloads: the ALDI step on device tensors (Engine.step) with the synthetic
linear-Gaussian problem of bench.py; the Darcy rows: ms per sampling.run iteration of examples/darcy_flow.py's ensemble
sizes on the full 16 x 16 model (p = 256), the forward solve included.  The card, its power limit and SM clock are read
in the same process and written with the numbers.

    python tools/bench_ensemble_noise.py [--repeats 3] [--steps 3] [--out profiles/r06_bench_ensemble_noise.json]

``--small`` times the single-CTA regime instead: sampling.run(T) of the aldi rule with the lineal map at BASELINE config 1
(p = 2, k = 10, J = 100) and at p = 8, k = 16, J = 128 ... 512, four arms alternated per repeat -- the Cholesky noise
in one launch (config 1's path), the ensemble noise in one launch, the ensemble noise through the per-iteration loop
(``fused_run = False``) on the phases (``CES_NO_SMALL_PATH=1``) and on the one-kernel step.  ms per iteration (wall clock
around the call, which ends in a synchronisation), launches per run, and the deviation of the one-launch ensemble run from
the phase loop.  The arms set the J limits of the ensemble noise on the single-CTA path: the one-launch run against the
phase loop (calibrate.py _FUSED_ENSEMBLE_J_MAX, lifted here), the one-kernel step against the phases (csrc/api.cu
kSmallEnsembleJMax; above it the last arm takes the phases, as its launch count shows).

    python tools/bench_ensemble_noise.py --small [--repeats 3] [--out profiles/r08_bench_small_ensemble_noise.json]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

UPDATE_WORKLOADS = [("target", 1024, 4096, 65536), ("cfg3", 1024, 4096, 16384), ("sweep", 1024, 4096, 4096),
                    ("sweep", 1024, 4096, 1024)]
DARCY_JS = (17, 51, 128, 258, 512, 768)       # examples/darcy_flow.py: p/15, p/5, p/2, p+2, 2p, 3p at p = 256
V_GEMM_TFLOPS = 35.6                          # DESIGN.md section 4: the V = U~ D GEMM at the target shape


def card():
    import torch

    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit"], out["sm_clock"], out["sm_clock_max"] = [x.strip() for x in q.split(",")]
    except Exception as e:                  # the numbers stay meaningful with the name alone; say what is missing
        out["nvidia_smi"] = "unavailable: %s" % e
    return out


def stats(v):
    return {"mean": float(np.mean(v)), "min": float(np.min(v)), "max": float(np.max(v)), "n": len(v)}


def noise_pass_ms(eng, fn):
    """Sum of the noise:begin -> noise:end intervals of one call of fn (timeline on for that call only)."""
    eng.timeline(True)
    fn()
    marks = eng.timeline_read()
    eng.timeline(False)
    total, begin = 0.0, None
    for name, ms in marks:
        if name == "noise:begin":
            begin = ms
        elif name == "noise:end" and begin is not None:
            total, begin = total + ms - begin, None
    return total


def fill_ms(eng, J, repeats=3):
    """The fills of one step's noise pass on their own: J x panel blocks covering J columns, CUDA events."""
    import torch

    from ces_b200 import _lib

    panel = min(eng.Jl, max(128, (8 << 30) // (8 * (-(-eng.Jl // 16) * 16)) // 128 * 128))
    buf = torch.empty(J, panel, dtype=torch.float64, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def once():
        for q0 in range(0, J, panel):
            nq = min(panel, J - q0)
            _lib.check(eng.lib.ces_fill_ensemble_noise(st, 1, 0, ctypes.c_void_p(buf.data_ptr()), panel, J, nq, 0, q0))

    once()
    best = []
    for _ in range(repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        once()
        e1.record()
        torch.cuda.synchronize()
        best.append(e0.elapsed_time(e1))
    del buf
    torch.cuda.empty_cache()
    return float(np.median(best))


def update_workload(name, p, k, J, steps, repeats):
    import torch

    from ces_b200.engine import Engine
    from oracle import eks_oracle as eo

    rs = np.random.RandomState(0)
    A = torch.from_numpy(rs.normal(size=(k, p)) / np.sqrt(p)).cuda()
    ustar = rs.normal(size=p)
    y = (A.cpu().numpy() @ ustar) + 0.1 * rs.normal(size=k)
    U = 10.0 * torch.randn(p, J, dtype=torch.float64, device="cuda")
    G = A @ U
    xi = torch.randn(p, J, dtype=torch.float64, device="cuda")
    out = torch.empty_like(U)
    eng = Engine(p, k, J)
    eng.set_problem(y, 0.01 * np.eye(k), 100.0 * np.eye(p), np.zeros(p), ustar)
    modes = {"cholesky": lambda: eng.step("aldi", U, G, xi, out=out),
             "ensemble": lambda: eng.step("aldi", U, G, None, out=out, noise=("ensemble", 1, 0, None))}
    for fn in modes.values():
        fn()
        fn()
    torch.cuda.synchronize()
    times = {m: [] for m in modes}
    for _ in range(repeats):
        for m, fn in modes.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            times[m].append(e0.elapsed_time(e1) / steps)
    pass_ms = noise_pass_ms(eng, modes["ensemble"])
    f_ms = fill_ms(eng, J)
    gemm_ms = max(pass_ms - f_ms, 1e-9)
    eng.close()
    del U, G, xi, out, A
    torch.cuda.empty_cache()
    rec = {"workload": name, "p": p, "k": k, "J": J, "rule": "aldi", "steps_per_repeat": steps,
           "ms_per_step": {m: stats(v) for m, v in times.items()},
           "ensemble_over_cholesky": float(np.mean(times["ensemble"]) / np.mean(times["cholesky"])),
           "noise_pass_ms": pass_ms, "fill_ms": f_ms, "fill_share": f_ms / pass_ms if pass_ms > 0 else None,
           "noise_gemm_tflops": 2.0 * p * J * J / gemm_ms * 1e-9, "v_gemm_tflops_design": V_GEMM_TFLOPS,
           "algorithmic_step_flops": eo.algorithmic_flops(J, p, k)}
    print(json.dumps(rec), flush=True)
    return rec


def darcy_rows(repeats, T):
    import ces_b200.darcy as darcy
    from ces_b200.calibrate import sampling

    model = darcy.model(Nmesh=16)
    model.set_initial()
    model.n_obs = 50
    model.model_name = "darcy-flow"
    np.random.seed(1)
    Uf = model(model.ustar, full_solution=True)
    model.obs_index = np.random.choice(int(model.p), model.n_obs, replace=False, p=Uf / Uf.sum())
    y = model(model.ustar) + 0.005 * np.random.normal(0, 1, model.n_obs)
    Gamma = 0.005 ** 2 * np.identity(model.n_obs)
    rows = []
    for J in DARCY_JS:
        s = sampling(p=model.p, n_obs=model.n_obs, J=J)
        s.ustar, s.T = model.ustar.reshape(model.p, -1), T
        s.mu, s.sigma, s.directory = np.zeros((model.p, 1)), 100.0 * np.identity(model.p), "/tmp"
        U0 = 10 * np.random.RandomState(J).normal(0, 1, [model.p, J])
        kw = {"cholesky": dict(rng="device"), "ensemble": dict(noise="ensemble")}

        def run(m):
            s.metrics = dict((key, []) for key in ("self-bias", "self-bias-data", "bias-data", "bias", "t"))
            s.Uall, s.Gall = [], []
            t0 = time.perf_counter()
            s.run(y, U0, model, Gamma, None, t_tol=1e9, seed=3, trace=False, **kw[m])
            return 1e3 * (time.perf_counter() - t0) / T

        for m in kw:
            run(m)
        times = {m: [] for m in kw}
        for _ in range(repeats):
            for m in kw:
                times[m].append(run(m))
        eng = s._engine
        s.T = 1
        pass_ms = noise_pass_ms(eng, lambda: s.run(y, U0, model, Gamma, None, t_tol=1e9, seed=3, trace=False, noise="ensemble"))
        f_ms = fill_ms(eng, J)
        rec = {"workload": "darcy-16x16-full", "p": int(model.p), "k": int(model.n_obs), "J": J, "rule": "aldi",
               "iterations_per_run": T, "ms_per_iteration": {m: stats(v) for m, v in times.items()},
               "cholesky_noise": "rng='device' (both modes draw on the device)",
               "noise_pass_ms": pass_ms, "fill_ms": f_ms, "fill_share": f_ms / pass_ms if pass_ms > 0 else None,
               "noise_gemm_tflops": 2.0 * model.p * J * J / max(pass_ms - f_ms, 1e-9) * 1e-9}
        print(json.dumps(rec), flush=True)
        rows.append(rec)
    return rows


SMALL_SHAPES = [("cfg1", 2, 10, 100)] + [("p8k16", 8, 16, J) for J in (128, 192, 256, 384, 512)]
SMALL_ARMS = {"cholesky_fused": dict(fused=True, small=True, kw={}),
              "ensemble_fused": dict(fused=True, small=True, kw=dict(noise="ensemble", seed=3)),
              "ensemble_loop_phases": dict(fused=False, small=False, kw=dict(noise="ensemble", seed=3)),
              "ensemble_loop_small_step": dict(fused=False, small=True, kw=dict(noise="ensemble", seed=3))}


def small_problem(name, p, k, J):
    if name == "cfg1":
        sys.path.insert(0, ROOT)
        from bench import cfg1_problem

        pr = cfg1_problem()
        return pr["A"], pr["ustar"], pr["y"], pr["Gamma"], pr["U0"]
    rs = np.random.RandomState(1000 * p + J)
    A = rs.normal(size=(k, p)) / np.sqrt(p)
    ustar = rs.normal(size=(p, 1))
    return A, ustar, A @ ustar[:, 0] + 0.1 * rs.normal(size=k), 0.01 * np.eye(k), 3.0 * rs.normal(size=(p, J))


def small_rows(repeats, T):
    from ces_b200 import calibrate, utils

    calibrate._FUSED_ENSEMBLE_J_MAX = 512       # time the one-launch arm at every J, past the limit that it sets too
    rows = []
    for name, p, k, J in SMALL_SHAPES:
        A, ustar, y, Gamma, U0 = small_problem(name, p, k, J)
        model = utils.lineal(A)
        samplers = {}
        for arm, cfg in SMALL_ARMS.items():
            s = calibrate.sampling(p, k, J)
            s.ustar, s.mu, s.sigma, s.T, s.fused_run = ustar, np.zeros((p, 1)), 100.0 * np.eye(p), T, cfg["fused"]
            if not cfg["small"]:
                os.environ["CES_NO_SMALL_PATH"] = "1"          # read when the handle is created
            s._get_engine(J)
            os.environ.pop("CES_NO_SMALL_PATH", None)
            samplers[arm] = s

        def run(arm):
            s = samplers[arm]
            s.metrics = dict((key, []) for key in ("self-bias", "self-bias-data", "bias-data", "bias", "t"))
            s.Uall, s.Gall = [], []
            np.random.seed(3)
            n0 = s._engine.launch_count()
            t0 = time.perf_counter()
            s.run(y, U0.copy(), model, Gamma, None, t_tol=1e30, **SMALL_ARMS[arm]["kw"])
            ms = 1e3 * (time.perf_counter() - t0) / len(s.metrics["t"])
            return ms, s._engine.launch_count() - n0

        for arm in SMALL_ARMS:
            run(arm)
        times, launches = {a: [] for a in SMALL_ARMS}, {}
        for _ in range(repeats):
            for arm in SMALL_ARMS:
                ms, launches[arm] = run(arm)
                times[arm].append(ms)
        ref = samplers["ensemble_loop_phases"].Ustar
        dev = float(np.abs(samplers["ensemble_fused"].Ustar - ref).max() / np.abs(ref).max())
        mean = {a: float(np.mean(v)) for a, v in times.items()}
        rec = {"workload": name, "p": p, "k": k, "J": J, "rule": "aldi", "map": "lineal", "iterations_per_run": T,
               "ms_per_iteration": {a: stats(v) for a, v in times.items()}, "launches_per_run": launches,
               "ensemble_fused_over_cholesky_fused": mean["ensemble_fused"] / mean["cholesky_fused"],
               "ensemble_fused_over_loop_phases": mean["ensemble_fused"] / mean["ensemble_loop_phases"],
               "small_step_over_phases_per_iteration": mean["ensemble_loop_small_step"] / mean["ensemble_loop_phases"],
               "ensemble_fused_vs_loop_phases_max_rel_dev": dev}
        print(json.dumps(rec), flush=True)
        rows.append(rec)
        for s in samplers.values():
            s._engine.close()
            s._engine = None
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--darcy-iterations", type=int, default=20)
    ap.add_argument("--out", default=None, help="default: profiles/r06_bench_ensemble_noise.json, "
                                                "profiles/r08_bench_small_ensemble_noise.json with --small")
    ap.add_argument("--only", default="", help="comma-separated J values of the update workloads (default: all)")
    ap.add_argument("--no-darcy", action="store_true")
    ap.add_argument("--small", action="store_true", help="the single-CTA regime only (sampling.run of small problems)")
    ap.add_argument("--small-iterations", type=int, default=1000)
    args = ap.parse_args()
    if args.repeats < 3:
        ap.error("--repeats must be >= 3")
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_ensemble_noise needs a CUDA device (sm_100a)")
    if args.small:
        out = args.out or os.path.join(ROOT, "profiles", "r08_bench_small_ensemble_noise.json")
        result = {"card": card(), "repeats": args.repeats, "small": small_rows(args.repeats, args.small_iterations)}
        result["card_after"] = card()
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as fh:
            json.dump(result, fh, indent=1)
        print("wrote", out)
        return
    result = {"card": card(), "repeats": args.repeats, "update": [], "darcy": []}
    only = {int(x) for x in args.only.split(",") if x}
    for name, p, k, J in UPDATE_WORKLOADS:
        if not only or J in only:
            result["update"].append(update_workload(name, p, k, J, args.steps, args.repeats))
    if not args.no_darcy:
        result["darcy"] = darcy_rows(args.repeats, args.darcy_iterations)
    result["card_after"] = card()
    out = args.out or os.path.join(ROOT, "profiles", "r06_bench_ensemble_noise.json")
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as fh:
        json.dump(result, fh, indent=1)
    print("wrote", out)


if __name__ == "__main__":
    main()
