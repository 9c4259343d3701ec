#!/usr/bin/env python
"""bench.py -- particle-updates/s of one EKS (ALDI) step on B200, the headline metric of BASELINE.json.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload target|cfg3|cfg1|cfg2|cfg4|small]
                    [--impl reference] [--no-configs] [--no-parity] [--no-cpu-baseline] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  A "step" is one ensemble Kalman update (sampling.eks_update_aldi,
ces/calibrate.py:451-490) of the synthetic linear-Gaussian ensemble of SURVEY.md section 8(d).

  value      J * steps / s with U, G, xi already resident in HBM (Engine.step, device pointers);
             timed with CUDA events on the stream the library launches on, max over ranks.
  e2e        the same metric through the reference-facing call sampling.eks_update_aldi(numpy arrays) at every N:
             pinned host buffers, host->device copies of U, G, xi and the device->host copy of U_next are
             inside the timed region.  N > 1: the sampler carries the process group (sampling.group) and every rank
             passes its column shard (local_shard=True).
  roofline   the dominant kernel (D = (1/J) E^T W, FP64 DMMA): algorithmic flops / CUDA-event duration of
             its launches inside the timed region (ces_profile_*), against the FP64 tensor peak.  The
             MEASURED_PEAKS.json file holds no FP64 figure, so the denominator is the cuBLAS DGEMM rate
             measured in this run (torch.matmul fp64, yardstick only); nominal 148 SM x 128 flop/clk x
             1.965 GHz = 37.2 TF/s is reported beside it.
  parity     after the timed region, at every N: hk against the Gram identity ||D||_F^2 = sum(EE^T o WW^T)/J^2, a
             128-particle probe of U_next recomputed from the definition with torch fp64 (cuBLAS; not the oracle, not
             our kernels), and at N > 1 rank 0's shard against a single-GPU engine run on the gathered ensemble.
  configs    (default workload only) short runs of the other BASELINE.json configs in the same process: cfg1 through
             sampling.run(T=1000) (ces/calibrate.py:270-416), cfg2 / cfg4 (update + batched Darcy forward), cfg3.
  cpu_baseline  N = 1 only: the REAL reference step (baseline/_ref/ces/calibrate.py, staged unmodified by
             oracle/stage_reference.py; kind "reference") on the host cores at a bounded ensemble size J_sample;
             the numpy port (oracle/, kind "port") only if the staged files are absent.
  --impl reference  times only that CPU arm: K steps of the real sampling.eks_update_aldi at J_sample (named in
             config), all host threads (torchrun's OMP_NUM_THREADS=1 is overridden), rank 0 only.
  --dump-outputs DIR  after the timed steps of the selected workload, what its last step returned to the caller as
             DIR/<name>.npy (float64, at most 64 MB in all; see dump_outputs), rank 0's column shard when N > 1.  The
             inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import os
import sys

if "reference" in sys.argv[1:] or "--impl=reference" in sys.argv[1:]:
    # the CPU arm must use every host core: torch.distributed.run exports OMP_NUM_THREADS=1 to its workers and
    # OpenBLAS reads it when numpy is imported -- set the pool size before that happens (threadpoolctl again below)
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(os.cpu_count() or 1)

import argparse
import json
import subprocess
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (d, k, J)
    "target": (1024, 4096, 65536),     # BASELINE.json "Target": one EKS step at J=65536, d=1024, k=4096
    "cfg3": (1024, 4096, 16384),       # BASELINE.json configs[2]
    "small": (64, 50, 1024),           # configs[1] shape (smoke-sized)
}
# One EKS iteration INCLUDING the batched Darcy forward solve (ces/darcy.py model_trunc): (grid, d, n_obs, J, update rule)
DARCY_WORKLOADS = {
    "cfg2": (64, 64, 50, 1024, "eki"),       # BASELINE.json configs[1]: EKI, 64 x 64 grid, d = 64 KL modes, J = 1024
    "cfg4": (128, 256, 50, 65536, "aldi"),   # configs[3]: EKS, 128 x 128 grid, d = 256, J = 65536 (8192 per GPU at N = 8)
}
METRIC = "particle-updates/sec (J*steps/s) for one EKS step"
NOMINAL_FP64_TFLOPS = 148 * 128 * 1.965e9 / 1e12
REF_J_CANDIDATES = (4096, 2048, 1024, 512)      # bounded ensemble sizes of the CPU arm, largest that fits the budget
REF_BUDGET_S = float(os.environ.get("CES_BENCH_REF_BUDGET_S", "420"))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=os.environ.get("CES_BENCH_WORKLOAD", "target"),
                    choices=sorted(list(WORKLOADS) + list(DARCY_WORKLOADS) + ["cfg1"]))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the short runs of the other BASELINE configs")
    ap.add_argument("--no-parity", action="store_true", help="skip the correctness probe after the timed region")
    ap.add_argument("--formulation", default="interaction", choices=["interaction", "factored"],
                    help="'interaction' forms the J x J matrix D like the reference (the graded formulation, default); "
                         "'factored' is the opt-in algorithmically reduced path (same update to rounding, D never formed)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (GPU arm only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arm; --impl reference has none")
    return args


# ------------------------------------------------------------------------------------------------ flop models
def algorithmic_flops(J, d, k, gamma_dense=False):
    """W_step of SURVEY.md section 8(d): the flops the D-forming formulation needs (no credit for the reference's
    redundant metric products)."""
    w = 2.0 * k * J * J + 2.0 * d * J * J
    w += 2.0 * k * k * J if gamma_dense else 1.0 * k * J
    return w + 6.0 * d * d * J + d ** 3 / 3.0


def reference_flops(J, d, k):
    """The step as the reference writes it (BASELINE.md section 3): 3 J x J x k products, 3 Gamma solves."""
    return 6.0 * k * J * J + 2.0 * d * J * J + 6.0 * k * k * J + 2.0 * k ** 3


def config_of(name, formulation, d, k, J, nranks):
    return {"workload": "EKS/ALDI step, synthetic linear-Gaussian, d=%d k=%d J=%d, Gamma=0.1^2 I, Sigma0=100 I (%s)"
                        % (d, k, J, name),
            "d": d, "k": k, "J": J, "update": "aldi", "time_step": "default 1/(||D||_F+1e-8)",
            "parallelism": "particle columns sharded over %d GPU(s)" % nranks,
            "formulation": ("interaction: D = (1/J) E^T W formed in panels (reference formulation)"
                            if formulation == "interaction" else
                            "factored: ALGORITHMICALLY REDUCED, (U~ E^T) W and Gram-matrix ||D||_F, D never formed"),
            "l2": "inputs per step (U, G, xi = %.2f GB) exceed the 126 MB L2; no explicit flush" % (8.0 * J * (2 * d + k) / 1e9)}


# ------------------------------------------------------------------------------------------------ CPU arm
def host_threads():
    try:
        from threadpoolctl import threadpool_info

        n = [p.get("num_threads", 1) for p in threadpool_info() if p.get("user_api") == "blas"]
        if n:
            return int(max(n))
    except Exception:
        pass
    return os.cpu_count() or 1


class all_host_threads(object):
    """BLAS pool = every host core for the duration of the CPU arm (torchrun exports OMP_NUM_THREADS=1)."""

    def __enter__(self):
        self.ctl = None
        try:
            from threadpoolctl import threadpool_limits

            self.ctl = threadpool_limits(limits=os.cpu_count() or 1)
        except Exception:
            pass
        return self

    def __exit__(self, *exc):
        if self.ctl is not None:
            self.ctl.restore_original_limits()


def linear_gaussian_problem(d, k, J, seed=0):
    """The synthetic problem of SURVEY.md section 8(d) / BASELINE.md section 3 (host arrays, for the CPU arm)."""
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((k, d)) / np.sqrt(d)
    ustar = rng.standard_normal(d)
    y = A @ ustar + 0.1 * rng.standard_normal(k)
    U0 = 10.0 * rng.standard_normal((d, J))
    return dict(ustar=ustar.reshape(d, 1), Gamma=0.01 * np.identity(k), y=y, mu=np.zeros((d, 1)),
                Sigma0=100.0 * np.identity(d), U0=U0, G=A @ U0, xi=np.random.RandomState(1).normal(0, 1, [d, J]))


def reference_stepper(d, k, Js):
    """(callable running ONE step of the CPU baseline at ensemble size Js, kind, description).  The real reference
    (sampling.eks_update_aldi of the staged, unmodified ces/calibrate.py) when available, else the numpy port."""
    from oracle import reference_loader as rl

    pr = linear_gaussian_problem(d, k, Js)
    if rl.available():
        def one():
            rl.reference_step("aldi", pr["y"], pr["U0"], pr["G"], pr["Gamma"], pr["mu"], pr["Sigma0"], pr["ustar"], pr["xi"])
        return one, "reference", ("the reference's own sampling.eks_update_aldi (ces/calibrate.py:451-490, unmodified file "
                                  "from %s, tab-expanded in memory)" % os.path.relpath(rl.REFERENCE_ROOT, ROOT)
                                  if rl.REFERENCE_ROOT.startswith(ROOT) else
                                  "the reference's own sampling.eks_update_aldi (ces/calibrate.py:451-490, %s)" % rl.REFERENCE_ROOT)
    from oracle import eks_oracle as eo

    def one_port():
        eo.step("aldi", pr["y"], pr["U0"], pr["G"], pr["Gamma"], pr["mu"], pr["Sigma0"], pr["ustar"], pr["xi"], as_written=True)
    return one_port, "port", "numpy restatement of sampling.eks_update_aldi as written (oracle/eks_oracle.py; staged reference absent)"


def pick_reference_J(d, k, J, total_steps, budget_s):
    """Largest candidate ensemble size whose total_steps steps fit the time budget, from one calibration step at the
    smallest candidate and the reference-as-written flop model (x 1.3 safety)."""
    cands = [c for c in REF_J_CANDIDATES if c <= J] or [J]
    if d * k < 1 << 16:
        return cands[0], None                              # small problems: seconds at any candidate
    Jc = cands[-1]
    one, _, _ = reference_stepper(d, k, Jc)
    one()
    t0 = time.perf_counter()
    one()
    tc = time.perf_counter() - t0
    rate = reference_flops(Jc, d, k) / tc
    for c in cands:
        if 1.3 * reference_flops(c, d, k) / rate * total_steps <= budget_s:
            return c, rate
    return Jc, rate


def cpu_step_rate(d, k, Js, steps, warmup):
    one, kind, what = reference_stepper(d, k, Js)
    for _ in range(warmup):
        one()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        one()
        ts.append(time.perf_counter() - t0)
    t = float(np.mean(ts))
    return Js / t, t, kind, what


def cpu_baseline(d, k, J, budget_s=25.0):
    """Bounded sample for the GPU arm's line (N = 1): about 10-30 s of CPU work."""
    with all_host_threads():
        Js, _ = pick_reference_J(d, k, J, 2, budget_s)
        rate, t, kind, what = cpu_step_rate(d, k, Js, 1, 1)
    full = rate * (reference_flops(Js, d, k) / Js) / (reference_flops(J, d, k) / J)
    return {"value": rate, "unit": "particle-updates/s", "cores": host_threads(), "kind": kind, "J_sample": Js,
            "sample": "%s, d=%d k=%d at J_sample=%d instead of J=%d, %.2f s/step; per-particle cost grows ~J so this "
                      "over-states the CPU at full J (flop-model extrapolation: %.3g particle-updates/s)"
                      % (what, d, k, Js, J, t, full),
            "extrapolated_full_J": full}


def cfg1_problem():
    """BASELINE.json configs[0]: the linear.ipynb problem (cell 4: np.random.seed(1), A = [1, 2 N(0,1)] 10 x 2,
    u* = (-1, 2), noise 0.1), prior N(0, 100 I), J = 100, 1000 steps (t_tol off)."""
    rs = np.random.RandomState(1)
    A = np.ones((10, 2))
    A[:, 1] = 2 * rs.normal(0, 1, 10)
    ustar = np.array([[-1.0], [2.0]])
    y = A @ ustar[:, 0] + np.sqrt(0.1) * rs.normal(0, 1, 10)
    return dict(A=A, ustar=ustar, y=y, Gamma=0.1 * np.eye(10), mu=np.zeros((2, 1)), Sigma0=100.0 * np.eye(2),
                U0=3.0 * rs.normal(0, 1, [2, 100]), J=100, T=1000)


def cfg1_reference_run(repeats=2):
    """The reference's own sampling.run(T=1000) on cfg1 with its own lineal model (ces/utils.py:5-31)."""
    from oracle import reference_loader as rl

    if not rl.available():
        return None
    cal, utils = rl.load_calibrate(), rl.load_utils()
    pr = cfg1_problem()
    best = 1e30
    for _ in range(repeats):
        eks = cal.sampling(p=2, n_obs=10, J=pr["J"])
        eks.ustar, eks.mu, eks.sigma, eks.T = pr["ustar"], pr["mu"], pr["Sigma0"], pr["T"]
        np.random.seed(3)
        t0 = time.perf_counter()
        eks.run(pr["y"], pr["U0"].copy(), utils.lineal(pr["A"]), pr["Gamma"], np.linalg.cholesky(pr["Gamma"]), t_tol=1e30)
        best = min(best, time.perf_counter() - t0)
    steps = len(eks.metrics["t"])
    return {"name": "cfg1", "value": pr["J"] * steps / best, "unit": "particle-updates/s", "ms_per_step": best / steps * 1e3,
            "steps": steps, "api": "reference sampling.run(T=1000, lineal d=2 k=10 J=100), wall clock, best of %d" % repeats,
            "posterior_mean": eks.Ustar.mean(axis=1).tolist()}


def darcy_problem(N, d, n_obs):
    """The scenario of examples/scripts/darcy-flow.py:9-36 on model_trunc: truth drawn with set_initial(seed=1), n_obs
    observation cells, gamma = 0.005, prior N(0, 100 I).  Host-side constants only; no solve happens here."""
    rng = np.random.default_rng(0)
    obs_index = np.sort(rng.choice(N * N, size=n_obs, replace=False))
    return {"obs_index": obs_index, "Gamma": 0.005 ** 2 * np.eye(n_obs), "mu": np.zeros((d, 1)),
            "Sigma0": 100.0 * np.eye(d)}


def darcy_cpu_rate(N, d, n_obs, J, rule, members, steps=1):
    """particle-updates/s of one host core running the scipy restatement of the Darcy solve (oracle/darcy_oracle.py, one
    sparse direct solve per member like the reference's MATLAB call) plus the update at a bounded ensemble."""
    from oracle import darcy_oracle as do
    from oracle import eks_oracle as eo

    pr = darcy_problem(N, d, n_obs)
    model = do.ModelTrunc(Nmesh=N, p=d)
    model.obs_index = pr["obs_index"]
    model.set_initial(seed=1)
    rng = np.random.default_rng(1)
    U = 10.0 * rng.standard_normal((d, members))
    y = model(model.ustar) + 0.005 * rng.standard_normal(n_obs)
    ts = []
    for _ in range(max(1, steps)):
        t0 = time.perf_counter()
        G = np.stack([model(U[:, j]) for j in range(members)], axis=1)
        xi = rng.standard_normal((d, members))
        eo.step("aldi" if rule != "eki" else "eki", y, U, G, pr["Gamma"], pr["mu"], pr["Sigma0"],
                model.ustar.reshape(d, 1), xi, as_written=(rule != "eki"))
        ts.append(time.perf_counter() - t0)
    t = float(np.median(ts))
    return members / t, t


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    base = {"impl": "reference", "unit": "particle-updates/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "gpu_launches": 0}
    if args.workload in DARCY_WORKLOADS:
        N, d, n_obs, J, rule = DARCY_WORKLOADS[args.workload]
        members = 8 if N > 64 else 32
        rate, t = darcy_cpu_rate(N, d, n_obs, J, rule, members, steps=max(1, args.steps))
        sample = ("scipy restatement of the Darcy solve (the reference's needs a MATLAB engine, SURVEY.md F4) + numpy update, "
                  "%d members instead of %d, %.2f s/step" % (members, J, t))
        base.update({"metric": METRIC + " including the batched Darcy forward solve", "value": rate, "ms_per_step": t * 1e3,
                     "config": {"workload": "%s (%s)" % (args.workload, rule), "d": d, "k": n_obs, "J": J, "grid": N,
                                "J_sample": members},
                     "cpu_baseline": {"value": rate, "unit": "particle-updates/s", "cores": 1, "kind": "port", "sample": sample,
                                      "J_sample": members},
                     "e2e": {"value": rate, "unit": "particle-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        emit(base)
        return
    if args.workload == "cfg1":
        with all_host_threads():
            rec = cfg1_reference_run()
        if rec is None:
            emit({"impl": "reference", "unavailable": "baseline/_ref/ces/calibrate.py is not staged (run __graft_entry__.build() "
                                                      "in the build container)"})
            return
        pr = cfg1_problem()
        base.update({"metric": METRIC + " through sampling.run", "value": rec["value"], "ms_per_step": rec["ms_per_step"],
                     "steps": rec["steps"], "warmup": 1,
                     "config": {"workload": "cfg1: sampling.run(T=1000), lineal d=2 k=10 J=100", "d": 2, "k": 10, "J": pr["J"]},
                     "cpu_baseline": {"value": rec["value"], "unit": "particle-updates/s", "cores": host_threads(),
                                      "kind": "reference", "sample": rec["api"], "J_sample": pr["J"]},
                     "e2e": {"value": rec["value"], "unit": "particle-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        emit(base)
        return
    d, k, J = WORKLOADS[args.workload]
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    with all_host_threads():
        Js, _ = pick_reference_J(d, k, J, steps + warmup, REF_BUDGET_S)
        rate, t, kind, what = cpu_step_rate(d, k, Js, steps, warmup)
        threads = host_threads()
        extra = None
        if args.workload == "target" and not args.no_configs:
            extra = cfg1_reference_run()
    full = rate * (reference_flops(Js, d, k) / Js) / (reference_flops(J, d, k) / J)
    sample = ("%s, d=%d k=%d at J_sample=%d (the full J=%d needs >= 3 J x J temporaries = %.0f GiB and ~%.0f s/step); "
              "%.2f s/step on %d BLAS threads; flop-model extrapolation to full J: %.3g particle-updates/s"
              % (what, d, k, Js, J, 3 * 8.0 * J * J / 2 ** 30, reference_flops(J, d, k) / (reference_flops(Js, d, k) / t), t,
                 threads, full))
    cfg = config_of(args.workload, "interaction", d, k, J, args.gpus)
    cfg["J_sample"] = Js                # the ensemble size this arm actually ran: NOT the same configuration as J
    cfg["workload"] += " -- CPU arm timed at J_sample=%d" % Js
    base.update({"metric": METRIC, "value": rate, "ms_per_step": t * 1e3, "steps": steps, "warmup": warmup, "config": cfg,
                 "cpu_baseline": {"value": rate, "unit": "particle-updates/s", "cores": threads, "kind": kind, "sample": sample,
                                  "J_sample": Js, "extrapolated_full_J": full},
                 "e2e": {"value": rate, "unit": "particle-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    if extra is not None:
        base["configs"] = [extra]
    emit(base)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler(object):
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.2 and len(r) >= 9] or [r for (_, r) in self.rows if len(r) >= 9]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(r[1]) for r in rows)
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            for name, val in zip(names, r[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "reasons": sorted(reasons),
                "power_w_max": max(float(r[3]) for r in rows), "samples": len(rows)}


# ------------------------------------------------------------------------------------------------ GPU arm
_REAL_STDOUT = None
# Deadline guard: the driver gives every run a wall-clock limit.  The headline record is published here as soon as its
# device measurement exists and is completed step by step (e2e, configs); if the run is still going at the deadline (a
# stuck collective in one of the later, optional legs, a slow box) rank 0 prints what is complete -- marked "truncated"
# -- and every rank leaves, instead of losing the whole line to the driver's kill.
PARTIAL = {"line": None, "done": False}
DEADLINE_S = float(os.environ.get("CES_BENCH_DEADLINE_S", "780"))


def _deadline_guard():
    def fire():
        if PARTIAL["done"]:
            return
        if int(os.environ.get("RANK", "0")) == 0 and PARTIAL["line"] is not None:
            line = dict(PARTIAL["line"])
            line["truncated"] = "deadline of %.0f s reached; legs not finished are absent" % DEADLINE_S
            emit(line)
        os._exit(0)

    t = threading.Timer(DEADLINE_S, fire)
    t.daemon = True
    t.start()
    return t


def emit(line):
    """Print the one JSON line on the real stdout (see main: fd 1 is pointed at stderr while the run is in progress so
    that library chatter such as NCCL's version banner cannot get in front of it)."""
    text = json.dumps(line) + "\n"
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, text.encode())
    else:
        sys.stdout.write(text)
        sys.stdout.flush()


DUMP_BYTES = 64 * 10 ** 6       # --dump-outputs: array data written in all


def dump_outputs(path, arrays):
    """Write ``arrays`` (name -> CUDA tensor, numpy array or number) as ``path/<name>.npy`` in float64, numbers as
    one-element arrays.  When they would exceed DUMP_BYTES, every (rows, particles) array keeps the same sorted sample of
    particle columns, drawn with a fixed seed, so that two runs are compared column for column."""
    import torch

    def host(a):
        return np.atleast_1d(a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)).astype(np.float64)

    wide = [n for n, a in arrays.items() if getattr(a, "ndim", 0) == 2]
    rest = {n: host(a) for n, a in arrays.items() if n not in wide}
    cols = {arrays[n].shape[1] for n in wide}
    assert len(cols) <= 1, "the (rows, particles) outputs must share one particle axis"
    rows = sum(arrays[n].shape[0] for n in wide)
    room = DUMP_BYTES - sum(a.nbytes for a in rest.values()) - 128 * len(arrays)     # 128: .npy header
    idx = None
    if wide and 8 * rows * max(cols) > room:
        idx = np.sort(np.random.default_rng(0).choice(max(cols), size=room // (8 * rows), replace=False))
    os.makedirs(path, exist_ok=True)
    for n in wide:
        a = arrays[n]
        if idx is not None:
            a = a[:, torch.as_tensor(idx, device=a.device)] if torch.is_tensor(a) else np.asarray(a)[:, idx]
        np.save(os.path.join(path, n + ".npy"), host(a))
    for n, a in rest.items():
        np.save(os.path.join(path, n + ".npy"), a)


class Ctx(object):
    """Device, ranks and the timing protocol shared by every workload of the GPU arm."""

    def __init__(self):
        import torch
        import torch.distributed as dist

        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.group = None
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
            self.group = dist.group.WORLD
        self._dgemm = None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, fn, steps):
        """K steps bracketed by barrier + synchronize; CUDA-event time, max over ranks (ms)."""
        torch = self.torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(ms, op=self.dist.ReduceOp.MAX)
        return float(ms.item())

    def dgemm_tflops(self):
        """FP64 yardstick (cuBLAS DGEMM through torch.matmul), measured once per process on every rank's own GPU."""
        if self._dgemm is None:
            torch = self.torch
            n = 8192
            a = torch.randn(n, 4096, dtype=torch.float64, device=self.dev)
            b = torch.randn(4096, n, dtype=torch.float64, device=self.dev)
            c = torch.empty(n, n, dtype=torch.float64, device=self.dev)
            best = 1e30
            for i in range(6):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                torch.matmul(a, b, out=c)
                e1.record()
                torch.cuda.synchronize()
                if i:
                    best = min(best, e0.elapsed_time(e1))
            self._dgemm = 2.0 * n * n * 4096 / best * 1e-9
            del a, b, c
            torch.cuda.empty_cache()
        return self._dgemm

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def parity_probe(ctx, d, k, J, y, ustar_h, U, G, xi, out, hk, ncols=128):
    """Correctness of the step just timed, from the definition, with torch fp64 (cuBLAS) -- independent of our kernels
    and of oracle/.  (i) hk against the Gram identity ||D||_F^2 = sum((E E^T) o (W W^T)) / J^2; (ii) ncols particles of
    rank 0's shard of U_next recomputed as U - h U~ D[:, c] - h C S^-1 (U - mu) + h alpha U~ + sqrt(2h) chol(C) xi
    (ces/calibrate.py:475-488) with D[:, c] = (1/J) E^T W[:, c] summed over the ranks' row blocks; (iii) N > 1: rank 0's
    shard against a single-GPU engine run on the gathered ensemble (the N = 1 formulation).  Collective on every rank."""
    torch, dist, world, rank = ctx.torch, ctx.dist, ctx.world, ctx.rank
    f64 = dict(dtype=torch.float64, device=ctx.dev)

    def allsum(t):
        if world > 1:
            dist.all_reduce(t)
        return t

    gbar = allsum(G.sum(dim=1)) / J
    ubar = allsum(U.sum(dim=1)) / J
    E = G - gbar[:, None]
    W = (G - y[:, None]) / 0.01
    Ut = U - ubar[:, None]
    frob2 = float((allsum(E @ E.t()) * allsum(W @ W.t())).sum()) / float(J) ** 2
    h_ref = 1.0 / (frob2 ** 0.5 + 1e-8)
    hk_rel = abs(hk - h_ref) / h_ref
    C = allsum(Ut @ Ut.t()) / (J - 1) + 1e-8 * torch.eye(d, **f64)
    L = torch.linalg.cholesky(C)
    n0 = min(ncols, U.shape[1]) if rank == 0 else 0
    ncount = torch.tensor([n0], device=ctx.dev)
    if world > 1:
        dist.broadcast(ncount, 0)
    nc = int(ncount.item())
    gen = torch.Generator(device=ctx.dev).manual_seed(7)
    cols = torch.randperm(U.shape[1], device=ctx.dev, generator=gen)[:nc] if rank == 0 else None
    Wc = W[:, cols].contiguous() if rank == 0 else torch.empty(k, nc, **f64)
    if world > 1:
        dist.broadcast(Wc, 0)
    V = allsum(Ut @ ((E.t() @ Wc) / J))
    probe_rel = None
    if rank == 0:
        ref = (U[:, cols] - h_ref * V - h_ref * (C @ (U[:, cols] / 100.0)) + h_ref * (d + 1.0) / J * Ut[:, cols]
               + (2 * h_ref) ** 0.5 * (L @ xi[:, cols]))
        probe_rel = float((out[:, cols] - ref).abs().max() / ref.abs().max())
    res = {"hk_rel": hk_rel, "probe_rel": probe_rel, "probe_columns": nc, "tol": 1e-10,
           "how": "torch fp64 (cuBLAS) from the definition; hk via the Gram identity"}
    del E, W, Ut, C, L, V
    if world > 1:
        from ces_b200.engine import Engine, shard_width

        Jl = shard_width(J, world)

        def gather(t):
            pad = torch.zeros(t.shape[0], Jl, **f64)
            pad[:, :t.shape[1]] = t
            parts = [torch.empty_like(pad) for _ in range(world)] if rank == 0 else None
            dist.gather(pad, parts, dst=0)
            return torch.cat(parts, dim=1)[:, :J].contiguous() if rank == 0 else None

        Uf, Gf, xf = gather(U), gather(G), gather(xi)
        if rank == 0:
            one = Engine(d, k, J)
            try:
                one.set_problem(y.cpu().numpy(), 0.01 * np.eye(k), 100.0 * np.eye(d), np.zeros((d, 1)), ustar_h)
                o1, h1, _ = one.step("aldi", Uf, Gf, xf)
                res["shard_vs_n1_rel"] = float((o1[:, :out.shape[1]] - out).abs().max() / o1.abs().max())
                res["hk_vs_n1_rel"] = abs(h1 - hk) / h1
            finally:
                one.close()
            del Uf, Gf, xf
        dist.barrier()
    if rank == 0:
        vals = [v for key, v in res.items() if key.endswith("_rel") and v is not None]
        res["ok"] = bool(max(vals) <= res["tol"])
    torch.cuda.empty_cache()
    return res


def update_workload(ctx, name, steps, warmup, formulation="interaction", with_cpu=True, with_parity=True, publish=False,
                    dump=None):
    """The headline measurement on one linear-Gaussian shape; returns the JSON record on rank 0 (None elsewhere).
    ``dump``: directory for dump_outputs of the last timed step."""
    torch, dist, world, rank, dev = ctx.torch, ctx.dist, ctx.world, ctx.rank, ctx.dev
    from ces_b200 import calibrate
    from ces_b200.engine import Engine, shard_range

    d, k, J = WORKLOADS[name]
    lo, hi = shard_range(J, rank, world)
    # synthetic problem (SURVEY.md 8d), generated on the device; every rank draws the same global data
    gen = torch.Generator(device=dev).manual_seed(0)
    rn = lambda *s: torch.randn(*s, dtype=torch.float64, device=dev, generator=gen)
    A = rn(k, d) / d ** 0.5
    ustar = rn(d)
    y = A @ ustar + 0.1 * rn(k)
    gen_c = torch.Generator(device=dev).manual_seed(100 + rank)
    U = 10.0 * torch.randn(d, hi - lo, dtype=torch.float64, device=dev, generator=gen_c)
    G = A @ U
    xi = torch.randn(d, hi - lo, dtype=torch.float64, device=dev, generator=gen_c)
    out = torch.empty_like(U)
    del A
    Gamma = 0.01 * np.eye(k)
    Sigma0 = 100.0 * np.eye(d)
    mu = np.zeros((d, 1))
    y_h, ustar_h = y.cpu().numpy(), ustar.cpu().numpy().reshape(d, 1)
    dgemm_tflops = ctx.dgemm_tflops()

    s = calibrate.sampling(d, k, J)
    s.mu, s.sigma, s.ustar = mu, Sigma0, ustar_h
    if ctx.group is not None:
        s.group = ctx.group
    eng = s._get_engine(J, ctx.group)
    s._sync_problem(eng, y_h, Gamma)
    last = [None]       # (U_next, hk, metrics) of the latest step

    def step_dev():
        last[0] = eng.step("aldi", U, G, xi, out=out, formulation=formulation)

    warmup = max(warmup, 3)
    for _ in range(warmup):
        step_dev()
    eng.profile(True)
    eng.profile_read()
    sampler = ClockSampler(ctx.local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    n0 = eng.launch_count()
    t0 = time.time()
    ms = ctx.timed(step_dev, steps)
    t1 = time.time()
    launches = eng.launch_count() - n0
    gemm_ms, gemm_n, gemm_flops = eng.profile_read()
    eng.profile(False)
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    ms_per_step = ms / steps
    value = J / (ms_per_step * 1e-3)
    hk = last[0][1]
    if dump is not None and rank == 0:
        dump_outputs(dump, dict(last[0][2], U_next=last[0][0], hk=hk))

    parity = None
    if with_parity and formulation == "interaction":
        parity = parity_probe(ctx, d, k, J, y, ustar_h, U, G, xi, out, hk)

    if publish and rank == 0:
        PARTIAL["line"] = {"metric": METRIC, "value": value, "unit": "particle-updates/s", "n_gpus": world, "steps": steps,
                           "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
                           "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                           "config": config_of(name, formulation, d, k, J, world), "e2e": None, "gpu_launches": int(launches),
                           "clocks": clocks, "parity": parity}
    # ---- end to end: the reference-facing call on pinned host arrays (every rank: its column shard)
    pin = lambda t: torch.empty(t.shape, dtype=torch.float64).pin_memory().copy_(t)
    Un, Gn, xn = pin(U).numpy(), pin(G).numpy(), pin(xi).numpy()
    kw = {"local_shard": True} if world > 1 else {}

    def step_e2e():
        s.eks_update_aldi(y_h, Un, Gn, Gamma, 0, xi=xn, formulation=formulation, **kw)

    step_e2e()
    e2e_steps = max(1, min(steps, 3))
    ms_e2e = ctx.timed(step_e2e, e2e_steps) / e2e_steps
    e2e = {"value": J / (ms_e2e * 1e-3), "unit": "particle-updates/s", "ms_per_step": ms_e2e,
           "h2d_bytes_per_step": 8 * J * (2 * d + k), "d2h_bytes_per_step": 8 * J * d,
           "api": "ces_b200.calibrate.sampling.eks_update_aldi(numpy arrays) -> ces_step_host" if world == 1 else
                  "ces_b200.calibrate.sampling.eks_update_aldi(numpy column shards, local_shard=True) with sampling.group"}
    eng.close()
    s._engine = None
    del U, G, xi, out
    torch.cuda.empty_cache()
    if rank != 0:
        return None

    flops_step = algorithmic_flops(J, d, k)
    if formulation == "factored":
        # flops of the reduced path: P1 and V (2dkJ each), two symmetric Gram matrices (k^2 J each), covariance,
        # prior and noise products, Cholesky
        flops_step = 4.0 * d * k * J + 2.0 * k * k * J + 6.0 * d * d * J + d ** 3 / 3.0 + k * J
    peak = dgemm_tflops
    achieved = gemm_flops / (gemm_ms * 1e-3) * 1e-12 if gemm_ms > 0 else None
    roofline = {"bound": "tensor", "kernel": "gemm_dmma_kernel<A_KM,B_KN> (D = (1/J) E^T W, FP64 DMMA.8x8x4 + TMA)",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": (achieved / peak) if achieved else None,
                "peak_source": "cuBLAS DGEMM 8192x8192x4096 measured in this run (MEASURED_PEAKS.json has no FP64 entry)",
                "peak_nominal": NOMINAL_FP64_TFLOPS,
                "launches": gemm_n, "ms_per_launch": gemm_ms / max(gemm_n, 1),
                "share_of_step": gemm_ms / ms if ms > 0 else None,
                "traffic": TRAFFIC_BYTES.get(name) if world == 1 else None,
                "step_achieved_tflops": flops_step / (ms_per_step * 1e-3) * 1e-12,
                "step_frac_of_peak": flops_step / (ms_per_step * 1e-3) * 1e-12 / (peak * world) if peak else None}
    if formulation == "factored":
        roofline.update({"kernel": "whole step, factored formulation (no single dominant kernel; D GEMM not launched)",
                         "achieved": roofline["step_achieved_tflops"], "frac": roofline["step_frac_of_peak"],
                         "launches": None, "ms_per_launch": None, "share_of_step": None, "traffic": None,
                         "algorithmically_reduced": True})
    line = {"metric": METRIC, "value": value, "unit": "particle-updates/s", "n_gpus": world, "steps": steps,
            "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_of(name, formulation, d, k, J, world),
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline}
    if parity is not None:
        line["parity"] = parity
    if publish:
        PARTIAL["line"] = dict(line)
    if world == 1 and with_cpu:
        line["cpu_baseline"] = cpu_baseline(d, k, J)
        if publish:
            PARTIAL["line"] = dict(line)
    return line


def darcy_workload(ctx, name, steps, warmup, with_cpu=True, dump=None):
    """cfg2 | cfg4: one ensemble Kalman iteration = batched Darcy forward solve of every member + update.
    ``dump``: directory for dump_outputs of the last timed step."""
    torch, dist, world, rank, dev = ctx.torch, ctx.dist, ctx.world, ctx.rank, ctx.dev
    from ces_b200 import calibrate
    from ces_b200 import darcy as cdarcy
    from ces_b200.engine import Engine, shard_range

    N, d, n_obs, J, rule = DARCY_WORKLOADS[name]
    pr = darcy_problem(N, d, n_obs)
    lo, hi = shard_range(J, rank, world)
    model = cdarcy.model_trunc(Nmesh=N, p=d)
    model.obs_index = pr["obs_index"]
    model.set_initial(seed=1)
    model.n_obs = n_obs
    ustar = np.asarray(model.ustar, dtype=np.float64).reshape(d, 1)
    eng = Engine(d, n_obs, J, group=ctx.group)
    rng = np.random.default_rng(1)
    y = model(model.ustar) + 0.005 * rng.standard_normal(n_obs)         # truth through the device solver
    eng.set_problem(y, pr["Gamma"], pr["Sigma0"], pr["mu"], ustar)
    gen = torch.Generator(device=dev).manual_seed(100 + rank)
    U = 10.0 * torch.randn(d, hi - lo, dtype=torch.float64, device=dev, generator=gen)      # darcy-flow.py:87
    xi = torch.randn(d, hi - lo, dtype=torch.float64, device=dev, generator=gen)
    G = torch.empty(n_obs, hi - lo, dtype=torch.float64, device=dev)
    out = torch.empty_like(U)
    stats = {"iters": 0, "members": 0, "ms": 0.0}
    last = [None]       # (U_next, hk, metrics) of the latest step

    def step_dev():
        model.evaluate_ensemble(eng, U, G)
        m_, it_, ms_ = model.last_stats()
        stats["iters"] += it_
        stats["members"] += m_
        stats["ms"] += ms_
        last[0] = eng.step(rule, U, G, None if rule == "eki" else xi, out=out)

    warmup = max(warmup, 3)
    for _ in range(warmup):
        step_dev()
    stats.update(iters=0, members=0, ms=0.0)
    sampler = ClockSampler(ctx.local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    n0 = eng.launch_count()
    t0 = time.time()
    ms = ctx.timed(step_dev, steps)
    t1 = time.time()
    launches = eng.launch_count() - n0
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    ms_per_step = ms / steps
    if dump is not None and rank == 0:
        dump_outputs(dump, dict(last[0][2], G=G, U_next=last[0][0], hk=last[0][1]))
    eng.close()

    # ---- end to end: sampling.run for ONE iteration from host arrays (H2D of U0, forward, update, the final forward
    # that run() always does, D2H of Ustar and Gstar); device Philox noise, no trace
    s = calibrate.sampling(d, n_obs, J)
    s.mu, s.sigma, s.ustar, s.T = pr["mu"], pr["Sigma0"], ustar, 1
    s.mute_bar = True
    if ctx.group is not None:
        s.group = ctx.group
    U0_h = 10.0 * np.random.default_rng(2).standard_normal((d, J))

    def step_e2e():
        if hasattr(s, "metrics"):
            del s.metrics
        s.run(y, U0_h, model, pr["Gamma"], None, trace=False, update=rule, rng="device", seed=1, t_tol=1e30)

    step_e2e()
    e2e_steps = max(1, min(steps, 3))
    ms_e2e = ctx.timed(step_e2e, e2e_steps) / e2e_steps
    if s._engine is not None:
        s._engine.close()
        s._engine = None
    model.stop()
    del U, G, xi, out
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    nodes = (N - 2) * (N - 2)
    flops = 18.0 * nodes * stats["iters"]                       # 9 FMA per node and CG iteration
    achieved = flops / (stats["ms"] * 1e-3) * 1e-12 if stats["ms"] > 0 else None
    peak = 148 * 64 * 2 * 1.965e9 / 1e12
    roofline = {"bound": "fp64-vector (the solver keeps a member in registers/shared memory of its cluster: neither an "
                         "HBM nor a tensor-core kernel; contract enum does not fit)",
                "kernel": "darcy_pcg_tile_kernel (preconditioned CG, one cluster per member)",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": (achieved / peak) if achieved else None,
                "peak_source": "nominal FP64 FMA rate 148 SM x 64 FMA/clk x 1.965 GHz (no measured FP64 entry in MEASURED_PEAKS.json)",
                "share_of_step": stats["ms"] / ms if ms > 0 else None,
                "cg_iterations_mean": stats["iters"] / max(stats["members"], 1),
                "node_iterations_per_s": nodes * stats["iters"] / (stats["ms"] * 1e-3) if stats["ms"] > 0 else None,
                "algorithmic_hbm_bytes": 16.0 * N * N * stats["members"],
                "hbm_gbs": 16.0 * N * N * stats["members"] / (stats["ms"] * 1e-3) * 1e-9 if stats["ms"] > 0 else None,
                "traffic": None}
    line = {"metric": METRIC + " including the batched Darcy forward solve", "value": J / (ms_per_step * 1e-3),
            "unit": "particle-updates/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": "%s iteration with batched Darcy forward (model_trunc Nmesh=%d, p=%d, n_obs=%d), J=%d (%s)"
                                   % (rule.upper(), N, d, n_obs, J, name),
                       "d": d, "k": n_obs, "J": J, "grid": N, "update": rule,
                       "parallelism": "particle columns sharded over %d GPU(s)" % world,
                       "l2": "per-step fields (3 x %.2f GB) exceed the 126 MB L2; no explicit flush" % (8.0 * N * N * min(J // world, 4096) / 1e9)},
            "e2e": {"value": J / (ms_e2e * 1e-3), "unit": "particle-updates/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": 8 * d * J, "d2h_bytes_per_step": 8 * (d + n_obs) * J,
                    "api": "ces_b200.calibrate.sampling.run(T=1, trace=False, rng='device'): forward + update + the final "
                           "forward run() always performs"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline}
    if world == 1 and with_cpu:
        members = 8 if N > 64 else 32
        rate, t = darcy_cpu_rate(N, d, n_obs, J, rule, members)
        line["cpu_baseline"] = {"value": rate, "unit": "particle-updates/s", "cores": 1, "kind": "port",
                                "sample": "scipy restatement of the Darcy solve (one sparse direct solve per member, like "
                                          "the reference's MATLAB call) + numpy update, %d members instead of %d, %.2f s"
                                          % (members, J, t)}
    return line


def cfg1_workload(ctx, repeats=3, with_cpu=True, dump=None):
    """BASELINE.json configs[0] through the reference-facing loop: sampling.run(T=1000) on the linear.ipynb problem
    (lineal, d=2, k=10, J=100), host arrays in, Uall / Gall / Ustar / metrics out -- exactly what ces/calibrate.py:270-416
    does in 1.1-1.3 s (BASELINE.md section 2).  Single GPU (J = 100 does not shard); value == e2e: the whole run is the
    public call, timed by CUDA events around it and by the wall clock.  ``dump``: directory for dump_outputs of the
    last run."""
    torch = ctx.torch
    from ces_b200 import calibrate, utils

    pr = cfg1_problem()
    model = utils.lineal(pr["A"])
    best_ms, best_wall, launches = 1e30, 1e30, 0
    for i in range(repeats + 1):
        s = calibrate.sampling(2, 10, pr["J"])
        s.ustar, s.mu, s.sigma, s.T = pr["ustar"], pr["mu"], pr["Sigma0"], pr["T"]
        np.random.seed(3)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        n0 = s._get_engine(pr["J"]).launch_count()
        t0 = time.perf_counter()
        e0.record()
        s.run(pr["y"], pr["U0"].copy(), model, pr["Gamma"], None, t_tol=1e30)
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        if i:                                       # first run = warm-up
            best_ms, best_wall = min(best_ms, e0.elapsed_time(e1)), min(best_wall, wall)
            launches = s._engine.launch_count() - n0
        steps = len(s.metrics["t"])
        post_mean = s.Ustar.mean(axis=1).tolist()
        if dump is not None and i == repeats:
            dump_outputs(dump, dict(s.metrics, Uall=s.Uall, Gall=s.Gall, Ustar=s.Ustar, Gstar=s.Gstar))
        s._engine.close()
        s._engine = None
    value = pr["J"] * steps / (best_ms * 1e-3)
    rec = {"name": "cfg1", "metric": METRIC + " through sampling.run", "value": value, "unit": "particle-updates/s",
           "ms_per_step": best_ms / steps, "steps": steps, "n_gpus": 1,
           "config": {"workload": "cfg1: sampling.run(T=1000, trace=True), lineal d=2 k=10 J=100 (linear.ipynb problem)",
                      "d": 2, "k": 10, "J": pr["J"]},
           "e2e": {"value": pr["J"] * steps / best_wall, "unit": "particle-updates/s", "ms_per_step": best_wall / steps * 1e3,
                   "h2d_bytes_per_step": 8 * 2 * pr["J"], "d2h_bytes_per_step": 8 * (2 + 10) * pr["J"],
                   "api": "ces_b200.calibrate.sampling.run(y, U0, lineal(A), Gamma, None) wall clock, best of %d" % repeats},
           "gpu_launches": int(launches),
           "roofline": {"bound": "latency", "kernel": "small_step_kernel (whole update in one CTA)", "achieved": None, "peak": None,
                        "unit": None, "frac": None, "traffic": None,
                        "note": "d=2, J=100: 3.3 kflop per step; the run is bounded by launch + host loop latency, not by a roofline"},
           "posterior_mean": post_mean}
    if with_cpu:
        with all_host_threads():
            ref = cfg1_reference_run()
        if ref is not None:
            rec["cpu_baseline"] = {"value": ref["value"], "unit": "particle-updates/s", "cores": host_threads(), "kind": "reference",
                                   "sample": ref["api"], "posterior_mean": ref["posterior_mean"]}
    return rec


def brief(line, name):
    """The fields of a workload line that go into the headline's ``configs`` array."""
    if line is None:
        return None
    keep = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "config", "e2e", "gpu_launches", "roofline",
            "parity", "cpu_baseline", "posterior_mean")
    rec = {"name": name}
    rec.update({key: line[key] for key in keep if key in line})
    return rec


def main():
    global _REAL_STDOUT
    args = parse()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        reference_arm(args)
        return
    _deadline_guard()
    ctx = Ctx()
    cpu = not args.no_cpu_baseline
    if args.workload in DARCY_WORKLOADS:
        line = darcy_workload(ctx, args.workload, args.steps, args.warmup, with_cpu=cpu, dump=args.dump_outputs)
    elif args.workload == "cfg1":
        line = None
        if ctx.rank == 0:
            rec = cfg1_workload(ctx, with_cpu=cpu, dump=args.dump_outputs)
            line = {"metric": rec["metric"], "value": rec["value"], "unit": rec["unit"], "n_gpus": ctx.world, "steps": rec["steps"],
                    "warmup": 1, "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "strong",
                    "vs_baseline": None, "dtype": "f64", "data": "synthetic"}
            line.update({key: rec[key] for key in ("config", "e2e", "gpu_launches", "roofline", "posterior_mean", "cpu_baseline")
                         if key in rec})
        ctx.barrier()
    else:
        line = update_workload(ctx, args.workload, args.steps, args.warmup, args.formulation, with_cpu=cpu,
                               with_parity=not args.no_parity, publish=True, dump=args.dump_outputs)
        if args.workload == "target" and args.formulation == "interaction" and not args.no_configs:
            # the other BASELINE.json configs, short runs in the same process (cfg1 / cfg2 are single-GPU shapes)
            configs = []
            short = max(2, min(args.steps, 5))

            def add(rec):
                if rec is not None:
                    configs.append(rec)
                if line is not None:
                    line["configs"] = list(configs)
                    PARTIAL["line"] = dict(line)

            def attempt(name, fn):
                # a failing side configuration must not take the headline line with it (an exception raised on every
                # rank alike; a rank-local one ends in the deadline guard)
                try:
                    add(fn())
                except Exception as exc:                        # noqa: BLE001
                    add({"name": name, "error": "%s: %s" % (type(exc).__name__, exc)} if ctx.rank == 0 else None)

            if ctx.world == 1:
                attempt("cfg1", lambda: cfg1_workload(ctx, with_cpu=cpu))
                attempt("cfg2", lambda: brief(darcy_workload(ctx, "cfg2", short, 3, with_cpu=False), "cfg2"))
            attempt("cfg3", lambda: brief(update_workload(ctx, "cfg3", short, 3, "interaction", with_cpu=False,
                                                          with_parity=not args.no_parity), "cfg3"))
            attempt("cfg4", lambda: brief(darcy_workload(ctx, "cfg4", 2, 3, with_cpu=False), "cfg4"))
    PARTIAL["done"] = True
    if ctx.rank == 0 and line is not None:
        emit(line)
    ctx.close()


# dram__bytes_read.sum + dram__bytes_write.sum per launch of the D GEMM, from the committed `ncu --set full` captures of
# round 2 (tools/gemm_traffic.py: the same kernel, operands and rasterisation as the step's launch).
TRAFFIC_BYTES = {
    # profiles/r02_ncu_full_gemm_d_cfg3.csv: 9.59 GB read + 2.14 GB written for the 16384 x 16384 x 4096 launch (60.41 ms)
    # (algorithmic: E 0.54 + W 0.54 + D 2.15 GB; the excess is E/W panels streamed once per wave of 148 tiles: a wave's
    # unique footprint, ~100 MB, fills the L2, so there is no cross-wave reuse; L2 hit rate 83.8 %, 3 % of HBM bandwidth)
    "cfg3": 11.73e9,
    # profiles/r02_ncu_full_gemm_d_target.csv: 42.69 GB read + 8.59 GB written per 65536 x 16384 x 4096 panel launch
    # (241.03 ms; algorithmic: E 2.15 + W panel 0.54 + D panel 8.59 GB), same mechanism; the serpentine traversal of the
    # contraction axis took the reads from 56.98 GB (round 1) to 42.69 GB
    "target": 51.28e9,
}

if __name__ == "__main__":
    main()
