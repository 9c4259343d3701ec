"""Benchmark of MCMC.model_mh on the Darcy models (ces_darcy_mh, csrc/darcy_mh.cu) as JSON lines.

    python tools/bench_darcy_mh.py [--out FILE] [--quick]

Workloads: 16^2 model_trunc p = 10, n_obs = 50 with 1 and with 1024 chains; 64^2 model_trunc p = 64 (the cfg2 shape) with
1024 chains; the 16^2 full model (p = 256) with pCN and 1024 chains.  Every line carries the GPU name and power limit read
in the same run.  Every shape is warmed up by a short call first; a timed call is one model_mh call (host clock; the call
ends in a device synchronise and includes the copy of the samples back to the host).  `forward_share` is the time of one
ces_darcy_forward of the same batch (the chains' current states, timed alone over repeated calls, each ending in a
synchronise) over the time of one step.  The comparator is the host restatement: oracle/mcmc_oracle.model_mh stepping one
chain through the scipy Darcy oracle (oracle/darcy_oracle.py, sparse direct solve) on this machine's CPU -- the reference's
own path drives a MATLAB engine that is not available, so it cannot be run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


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


def problem(N, p, n_obs=50, sd=0.005, seed=0):
    """Truth from the N(0, I) prior, observed cells drawn proportionally to the pressure (examples/darcy_flow.py), an
    ensemble of p + 20 members around the truth.  p = None: the full model."""
    from scipy.stats import multivariate_normal

    from oracle import darcy_oracle as do

    ref = do.ModelTrunc(Nmesh=N, p=p)
    P = ref.p
    rs = np.random.RandomState(seed)
    truth = rs.normal(size=P)
    U = ref(truth, full_solution=True)
    ref.obs_index = np.sort(rs.choice(N * N, n_obs, replace=False, p=U / U.sum()))
    y = ref(truth) + sd * rs.normal(size=n_obs)
    Ustar = truth[:, None] + 0.05 * rs.normal(size=(P, P + 20))
    return ref, y, sd ** 2 * np.eye(n_obs), Ustar, multivariate_normal(np.zeros(P), np.eye(P))


def run(N, p, chains, n_mcmc, kw, info, oracle_steps):
    import torch

    from ces_b200 import calibrate, darcy
    from ces_b200.sample import MCMC
    from oracle import mcmc_oracle as mo

    ref, y, Gamma, Ustar, prior = problem(N, p)
    P, n_obs = ref.p, len(ref.obs_index)
    model = darcy.model(Nmesh=N) if p is None else darcy.model_trunc(Nmesh=N, p=p)
    model.obs_index = ref.obs_index
    enka = calibrate.sampling(P, n_obs, Ustar.shape[1])
    enka.Ustar = Ustar
    np.random.seed(1)
    warm = MCMC()
    warm.y_obs = y
    warm.model_mh(model, 3, prior, enka, Gamma, n_chains=chains, seed=1, **kw)           # warm-up of every shape
    mc = MCMC()
    mc.y_obs = y
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    mc.model_mh(model, n_mcmc, prior, enka, Gamma, n_chains=chains, seed=2, **kw)
    sec = time.perf_counter() - t0
    step = sec / n_mcmc
    # the same batch through the forward model alone
    last = mc.samples_chains[:, :, -1].T if chains > 1 else mc.samples[:, -1:]
    U_dev = torch.from_numpy(np.ascontiguousarray(last)).cuda()
    G_dev = torch.empty(n_obs, chains, dtype=torch.float64, device="cuda")
    h = model._handle(True)
    model._forward(h, U_dev, G_dev, False)
    reps = max(3, int(0.5 / max(step, 1e-5)))
    t0 = time.perf_counter()
    for _ in range(reps):
        model._forward(h, U_dev, G_dev, False)
    fwd = (time.perf_counter() - t0) / reps
    acc = mc.accept_chains.mean() if chains > 1 else mc.accept
    line = dict(info, what="darcy_model_mh", nmesh=N, p=P, n_obs=n_obs, chains=chains, update=kw.get("update") or "rw",
                n_mcmc=n_mcmc, seconds=sec, steps_per_s=n_mcmc / sec, proposals_per_s=n_mcmc * chains / sec,
                step_ms=1e3 * step, forward_ms=1e3 * fwd, forward_share=fwd / step, accept=float(acc),
                cg_iterations_last_forward=int(model.last_iterations), tol=model.tol)
    lines = [line]
    if oracle_steps:
        np.random.seed(1)
        t0 = time.perf_counter()
        mo.model_mh(ref, oracle_steps, prior, Ustar, y, Gamma, **kw)
        osec = time.perf_counter() - t0
        lines.append(dict(info, what="oracle_host_restatement", nmesh=N, p=P, n_obs=n_obs, chains=1,
                          update=kw.get("update") or "rw", n_mcmc=oracle_steps, seconds=osec, steps_per_s=oracle_steps / osec,
                          proposals_per_s=oracle_steps / osec,
                          note="oracle/mcmc_oracle.model_mh + oracle/darcy_oracle (scipy sparse direct solve) on the host CPU, "
                               "one chain; the reference's MATLAB-engine path cannot run here"))
    return lines


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true", help="few steps only (a functional run)")
    args = ap.parse_args(argv)
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_darcy_mh needs a CUDA device")
    info = gpu_info()
    q = args.quick
    rw, pcn = dict(delta=4.0, enka_scaling=True), dict(update="pCN", beta=0.02, enka_scaling=False)
    work = [(16, 10, 1, 50 if q else 5000, rw, 20 if q else 200),
            (16, 10, 1024, 20 if q else 2000, rw, 0),
            (64, 64, 1024, 5 if q else 200, rw, 5 if q else 20),
            (16, None, 1024, 20 if q else 400, pcn, 20 if q else 100)]
    out = open(args.out, "w") if args.out else None
    for N, p, chains, n_mcmc, kw, oracle_steps in work:
        for ln in run(N, p, chains, n_mcmc, kw, info, oracle_steps):
            s = json.dumps(ln)
            print(s, flush=True)
            if out:
                out.write(s + "\n")
    if out:
        out.close()


if __name__ == "__main__":
    main()
