"""Calibrate -> Emulate -> Sample on the linear-Gaussian problem of the reference's examples/notebooks/linear.ipynb, all
three stages on the B200: the ensemble Kalman sampler (`sampling.run`) finds the posterior region, `GPEmulator(eks, Gamma)`
trains one exact GP per whitened output on the calibrated ensemble (eks.Ustar, eks.Gstar), and `MCMC.emulator_mh` samples
the posterior through the emulator -- the notebook's "RW-MH on GP emulator" -- with proposals scaled by eks.Ustar.  Same
problem as examples/linear_ces.py (which samples the true model instead).

    python examples/linear_ces_gp.py [--J 100] [--T 1000] [--n-mcmc 20000] [--chains 64]
"""
import argparse
import os
import sys

import numpy as np
from scipy.stats import multivariate_normal

sys.path.append(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from ces_b200.utils import *          # noqa: F401,F403   (reference: from ces.utils import *)
from ces_b200.calibrate import *      # noqa: F401,F403   (reference: from ces.calibrate import *)
from ces_b200.sample import MCMC      # noqa: E402        (reference: from ces.sample import *)
from ces_b200.emulate import GPEmulator  # noqa: E402


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--J", type=int, default=100)
    ap.add_argument("--T", type=int, default=1000)
    ap.add_argument("--n-mcmc", type=int, default=20000)
    ap.add_argument("--chains", type=int, default=64)
    args = ap.parse_args(argv)

    # ---- the problem (linear.ipynb cell 4): y = A u + noise, u* = (-1, 2), 10 observations
    np.random.seed(1)
    p, n_obs, noise = 2, 10, 0.1
    A = np.ones((n_obs, p))
    A[:, 1] = 2 * np.random.normal(0, 1, n_obs)
    u_star = np.array([-1.0, 2.0]).reshape(p, -1)
    y_obs = A.dot(u_star).flatten() + np.sqrt(noise) * np.random.normal(0, 1, n_obs)
    Gamma = noise * np.identity(n_obs)
    Jnoise = np.linalg.cholesky(Gamma)
    sigma2 = 100.0
    linear = lineal(A)                                           # noqa: F405

    # ---- Calibrate: EKS / ALDI from a wide initial ensemble
    eks = sampling(p=p, n_obs=n_obs, J=args.J)                   # noqa: F405
    eks.ustar, eks.mu, eks.sigma, eks.T = u_star, np.zeros((p, 1)), sigma2 * np.identity(p), args.T
    U0 = 3.0 * np.random.normal(0, 1, [p, args.J])
    eks.run(y_obs, U0, linear, Gamma, Jnoise, t_tol=1e30)

    # ---- the analytic posterior (cell 11)
    Sigma_n = np.linalg.inv(A.T.dot(A) / noise + np.identity(p) / sigma2)
    mean_n = Sigma_n.dot(A.T.dot(y_obs) / noise)

    # ---- Emulate: one GP per whitened output, trained on the calibrated ensemble
    emulator = GPEmulator(eks, Gamma).fit()

    # ---- Sample: Metropolis-Hastings on the emulator, proposals from the calibrated ensemble
    prior = multivariate_normal(np.zeros(p), sigma2 * np.identity(p))
    mcmc = MCMC()
    mcmc.y_obs = y_obs
    mcmc.emulator_mh(emulator, args.n_mcmc, prior, eks, delta=1.5, enka_scaling=True, n_chains=args.chains, seed=1)
    burn = args.n_mcmc // 5
    pooled = (mcmc.samples_chains[:, :, burn:] if args.chains > 1 else mcmc.samples[None, :, burn:])
    pooled = pooled.transpose(1, 0, 2).reshape(p, -1)

    out = {"posterior_mean": mean_n, "posterior_cov": Sigma_n, "eks_mean": eks.Ustar.mean(axis=1), "eks_cov": np.cov(eks.Ustar),
           "mcmc_mean": pooled.mean(axis=1), "mcmc_cov": np.cov(pooled), "accept": float(mcmc.accept), "eks": eks, "mcmc": mcmc,
           "emulator": emulator}
    print("analytic posterior mean %s" % mean_n)
    print("EKS ensemble mean       %s   (after %d iterations, t = %.3g)" % (out["eks_mean"], len(eks.metrics["t"]), eks.metrics["t"][-1]))
    print("GP emulator: %d outputs, fitted LML %s" % (emulator.k, np.round(emulator.fit_lml, 2)))
    print("MCMC mean (%d chains)   %s   acceptance %.2f" % (args.chains, out["mcmc_mean"], out["accept"]))
    print("analytic posterior cov\n%s\nMCMC cov\n%s" % (Sigma_n, out["mcmc_cov"]))
    return out


if __name__ == "__main__":
    main()
