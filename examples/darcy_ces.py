"""Calibrate -> Emulate -> Sample on the Darcy flow model, checked against Metropolis-Hastings on the true model.

The problem is examples/darcy_flow.py's on the truncated model: a 16 x 16 grid, the 10 leading KL modes as parameters, 50
observed cells drawn proportionally to the true pressure, noise sd 0.005, and one N(0, I) prior shared by every stage.
All four stages run on the B200:

  Calibrate   sampling.run (the ensemble Kalman sampler) from prior draws
  Emulate     GPEmulator(eks, Gamma, kernel=...).fit(): one exact GP per whitened observation, trained on
              (eks.Ustar, eks.Gstar), with the squared-exponential kernel or a Matern one (--kernel)
  Sample      MCMC.emulator_mh through the emulator, 64 chains, proposals scaled by eks.Ustar
  Gold        MCMC.model_mh on the Darcy model itself, 64 chains stepped in lockstep through the batched solver

It prints the mean and standard deviation of every mode for the EKS ensemble, the emulator chains and the true-model chains,
the gap between the emulator's and the true model's posterior means in true-posterior standard deviations, the ratio of
their standard deviations, and the wall time of each stage; main() returns them.

    python examples/darcy_ces.py [--nmesh 16] [--p 10] [--J 100] [--T 200] [--n-mcmc 20000] [--chains 64]
                                 [--kernel SquaredExponential|Matern12|Matern32|Matern52]
"""
import argparse
import os
import sys
import time

import numpy as np
from scipy.stats import multivariate_normal

sys.path.append(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from ces_b200.calibrate import *      # noqa: F401,F403   (reference: from ces.calibrate import *)
import ces_b200.darcy as darcy         # noqa: E402        (reference: import ces.darcy as darcy)
from ces_b200.sample import MCMC      # noqa: E402
from ces_b200.emulate import GPEmulator  # noqa: E402


def _pooled(mcmc, burn):
    x = mcmc.samples_chains[:, :, burn:] if hasattr(mcmc, "samples_chains") else mcmc.samples[None, :, burn:]
    return x.transpose(1, 0, 2).reshape(x.shape[1], -1)


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--nmesh", type=int, default=16)
    ap.add_argument("--p", type=int, default=10)
    ap.add_argument("--n-obs", type=int, default=50)
    ap.add_argument("--J", type=int, default=100)
    ap.add_argument("--T", type=int, default=200)
    ap.add_argument("--n-mcmc", type=int, default=20000)
    ap.add_argument("--chains", type=int, default=64)
    ap.add_argument("--delta", type=float, default=0.7)
    ap.add_argument("--kernel", default="SquaredExponential", choices=["SquaredExponential", "Matern12", "Matern32", "Matern52"],
                    help="the emulator's covariance family (GPflow's class names)")
    args = ap.parse_args(argv)

    # ---- the problem (examples/darcy_flow.py on model_trunc)
    model = darcy.model_trunc(Nmesh=args.nmesh, p=args.p)
    model.set_initial(seed=1)
    p, n_obs = int(model.p), args.n_obs
    U = model(model.ustar, full_solution=True)
    np.random.seed(1)
    model.obs_index = np.random.choice(args.nmesh ** 2, n_obs, replace=False, p=U / U.sum())
    gamma = 0.005
    Gamma = gamma ** 2 * np.identity(n_obs)
    y_obs = model(model.ustar) + gamma * np.random.normal(0, 1, n_obs)
    Jnoise = np.linalg.cholesky(Gamma)
    prior = multivariate_normal(np.zeros(p), np.identity(p))
    times = {}

    # ---- Calibrate
    t0 = time.perf_counter()
    eks = sampling(p=p, n_obs=n_obs, J=args.J)                   # noqa: F405
    eks.ustar, eks.mu, eks.sigma, eks.T = model.ustar.reshape(p, -1), np.zeros((p, 1)), np.identity(p), args.T
    eks.mute_bar = True
    U0 = np.random.normal(0, 1, [p, args.J])
    eks.run(y_obs, U0, model, Gamma, Jnoise, t_tol=1e30)
    times["calibrate"] = time.perf_counter() - t0

    # ---- Emulate
    t0 = time.perf_counter()
    emulator = GPEmulator(eks, Gamma, kernel=args.kernel).fit()
    times["emulate"] = time.perf_counter() - t0

    # ---- Sample through the emulator, and the gold standard on the true model
    burn = args.n_mcmc // 5
    emu_mcmc = MCMC()
    emu_mcmc.y_obs = y_obs
    t0 = time.perf_counter()
    emu_mcmc.emulator_mh(emulator, args.n_mcmc, prior, eks, delta=args.delta, enka_scaling=True, n_chains=args.chains, seed=1)
    times["sample_emulator"] = time.perf_counter() - t0
    model_mcmc = MCMC()
    model_mcmc.y_obs = y_obs
    t0 = time.perf_counter()
    model_mcmc.model_mh(model, args.n_mcmc, prior, eks, Gamma, delta=args.delta, enka_scaling=True, n_chains=args.chains, seed=2)
    times["sample_model"] = time.perf_counter() - t0

    emu_x, model_x = _pooled(emu_mcmc, burn), _pooled(model_mcmc, burn)
    out = {"truth": model.ustar, "eks_mean": eks.Ustar.mean(axis=1), "eks_sd": eks.Ustar.std(axis=1, ddof=1),
           "emulator_mean": emu_x.mean(axis=1), "emulator_sd": emu_x.std(axis=1, ddof=1),
           "model_mean": model_x.mean(axis=1), "model_sd": model_x.std(axis=1, ddof=1),
           "emulator_accept": float(np.mean(getattr(emu_mcmc, "accept_chains", emu_mcmc.accept))),
           "model_accept": float(np.mean(getattr(model_mcmc, "accept_chains", model_mcmc.accept))),
           "kernel": args.kernel, "times": times, "burn": burn, "eks": eks, "emulator": emulator, "emulator_mcmc": emu_mcmc, "model_mcmc": model_mcmc}
    print("Darcy %d^2, %d KL modes, %d observations; EKS J = %d (%d iterations), %d chains x %d steps (burn-in %d); "
          "emulator kernel %s" % (args.nmesh, p, n_obs, args.J, len(eks.metrics["t"]), args.chains, args.n_mcmc, burn, args.kernel))
    print("mode   truth      EKS mean / sd         emulator mean / sd    true-model mean / sd   (emu - model) / sd   emu sd / model sd")
    for i in range(p):
        print("%4d  %8.4f   %8.4f / %-8.4f   %8.4f / %-8.4f   %8.4f / %-8.4f    %+.3f               %.3f"
              % (i, out["truth"][i], out["eks_mean"][i], out["eks_sd"][i], out["emulator_mean"][i], out["emulator_sd"][i],
                 out["model_mean"][i], out["model_sd"][i], (out["emulator_mean"][i] - out["model_mean"][i]) / out["model_sd"][i],
                 out["emulator_sd"][i] / out["model_sd"][i]))
    gap, ratio = np.abs(out["emulator_mean"] - out["model_mean"]) / out["model_sd"], out["emulator_sd"] / out["model_sd"]
    print("emulator vs true model: max |mean gap| %.3f sd, sd ratio %.3f .. %.3f" % (gap.max(), ratio.min(), ratio.max()))
    print("acceptance: emulator %.3f, true model %.3f" % (out["emulator_accept"], out["model_accept"]))
    print("wall time [s]: " + ", ".join("%s %.2f" % kv for kv in times.items()))
    return out


if __name__ == "__main__":
    main()
