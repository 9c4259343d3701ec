"""Benchmark of the Emulate stage on the device: GP fit, prediction and MH through the emulator (JSON lines).

    python tools/bench_emulate.py [--out FILE] [--quick] [--kernel SquaredExponential|Matern12|Matern32|Matern52 ...]

Workloads: the notebook scale of linear.ipynb (p = 2, k = 10, n = 100; 1 and 1024 chains) and a large emulator (p = 32,
k = 64, n = 4096; 4096 chains), for each covariance family named by --kernel (default: the squared exponential), the
families alternating within each workload.  Every line carries the GPU name and power limit read in the same run.  Times are CUDA
events around work that ends in a device synchronise, every shape warmed up first.  FLOP model of one prediction of m
points: k n^2 m (the lower-triangular GEMM V = L^-1 K*) + k n m (3 p + 2) (assembly of K*: p scaled differences, squares
and sums plus the scale and exp per entry, counted as 3 p + 2) + 4 k n m (mean and sum of squares).  The notebook quotes
47-255 it/s for "RW-MH on GP emulator" (GPflow on the author's laptop, BASELINE.md section 1).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

NOTEBOOK_EMULATOR_ITS = "47-255 it/s (GPflow, author's laptop)"


def gpu_info():
    import torch

    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(out[0]), float(out[1])
    except Exception as e:                                                 # noqa: BLE001
        info["power_limit_w"] = "unavailable: %s" % e
    return info


def problem(p, k, n, seed=0):
    rs = np.random.RandomState(seed)
    X = rs.normal(size=(p, n))
    W = rs.normal(size=(k, p)) / np.sqrt(p)
    G = np.sin(W @ X) + 0.3 * (W @ X) ** 2 + 0.05 * rs.normal(size=(k, n))
    return X, G


def flops_predict(p, k, n, m):
    return k * n * n * m + k * n * m * (3 * p + 2) + 4 * k * n * m


def timed(fn, reps):
    import torch

    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3 / reps


def run(p, k, n, chains, n_mcmc, predict_m, reps, do_fit, info, kernel="SquaredExponential"):
    import torch
    from scipy.stats import multivariate_normal

    from ces_b200 import calibrate
    from ces_b200.emulate import GPEmulator
    from ces_b200.sample import MCMC

    X, G = problem(p, k, n)
    emu = GPEmulator(U=X, G=G, Gamma=0.01 * np.eye(k), kernel=kernel)
    base = dict(info, kernel=kernel, p=p, k=k, n=n)
    lines = []
    if do_fit:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        emu.fit()
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        lines.append(dict(base, what="fit", seconds=sec, lml_evaluations=emu.fit_evaluations,
                          ms_per_evaluation=1e3 * sec / emu.fit_evaluations))
    else:
        emu.theta = emu.default_init()
        emu.theta[:, 1:-1] += 0.5
    t0 = time.perf_counter()
    emu.condition()
    torch.cuda.synchronize()
    cond_s = time.perf_counter() - t0
    U = torch.randn(p, predict_m, dtype=torch.float64, device="cuda")
    sec = timed(lambda: emu.predict_device(U), reps)
    fl = flops_predict(p, k, n, predict_m)
    lines.append(dict(base, what="predict", m=predict_m, seconds=sec, points_per_s=predict_m / sec, flop=fl,
                      tflops=fl / sec / 1e12, condition_seconds=cond_s,
                      flop_model="k n^2 m + k n m (3 p + 2) + 4 k n m"))
    enka = calibrate.sampling(p, k, n)
    enka.Ustar = X
    prior = multivariate_normal(np.zeros(p), 4.0 * np.eye(p))
    mc = MCMC()
    mc.y_obs = G[:, 0]
    mc.emulator_mh(emu, 5, prior, enka, delta=0.3, n_chains=chains)           # warm-up of the shapes
    del mc.samples
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    mc.emulator_mh(emu, n_mcmc, prior, enka, delta=0.3, n_chains=chains)
    sec = time.perf_counter() - t0
    lines.append(dict(base, what="emulator_mh", chains=chains, n_mcmc=n_mcmc, seconds=sec, steps_per_s=n_mcmc / sec,
                      proposals_per_s=n_mcmc * chains / sec, accept=float(mc.accept), notebook=NOTEBOOK_EMULATOR_ITS))
    return lines


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="small sizes only (a functional run)")
    ap.add_argument("--kernel", nargs="+", default=["SquaredExponential"],
                    choices=["SquaredExponential", "Matern12", "Matern32", "Matern52"], help="covariance families to run")
    args = ap.parse_args(argv)
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_emulate needs a CUDA device")
    info = gpu_info()
    lines = []
    workloads = [(2, 10, 100, 1, 2000, 1024, 200, True), (2, 10, 100, 1024, 2000, 1024, 200, False)]
    if not args.quick:
        workloads.append((32, 64, 4096, 4096, 20, 4096, 5, False))
    for w in workloads:
        for kernel in args.kernel:
            lines += run(*w, info, kernel=kernel)
    out = open(args.out, "w") if args.out else None
    for ln in lines:
        s = json.dumps(ln)
        print(s, flush=True)
        if out:
            out.write(s + "\n")
    if out:
        out.close()


if __name__ == "__main__":
    main()
