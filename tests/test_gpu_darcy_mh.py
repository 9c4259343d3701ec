"""MCMC.model_mh on the Darcy models (ces_b200/sample.py -> ces_darcy_mh, csrc/darcy_mh.cu): chain 0 against
oracle/mcmc_oracle.py driving the scipy Darcy restatement of oracle/darcy_oracle.py (samples, acceptance, numpy's generator
state, resume), the prior recovered by 512 Philox chains when the data carry no information, the refusal of unconverged
solves and of a model without observations, and the Calibrate -> Emulate -> Sample example against the true-model chains.

The problems were chosen with the oracles alone so that chain 0 both accepts and rejects proposals."""
import os

import numpy as np
import pytest
from scipy.stats import multivariate_normal

pytestmark = pytest.mark.gpu

from ces_b200 import _lib, calibrate, darcy as cdarcy, sample as csample  # noqa: E402
from oracle import darcy_oracle as do, mcmc_oracle as mo  # noqa: E402

# name: (Nmesh, p (None: the full model), n_obs, noise sd, dense Gamma, sampler kwargs, n_mcmc)
CASES = {
    "trunc16_rw": (16, 10, 50, 0.005, False, dict(delta=4.0, enka_scaling=True), 150),
    "trunc16_pcn": (16, 10, 50, 0.005, False, dict(update="pCN", beta=0.03), 150),
    "full8_pcn": (8, None, 20, 0.002, True, dict(update="pCN", beta=0.01, enka_scaling=False), 120),
    "trunc32_rw_fixed": (32, 40, 60, 0.005, False, dict(delta=0.1, enka_scaling=False), 100),
}


def problem(name):
    """Seeded problem of CASES[name]: truth from the N(0, I) prior, observation cells drawn proportionally to the pressure
    (examples/darcy_flow.py), y = G(truth) + noise, and an ensemble clustered around the truth (for the proposal scales,
    the start and phi_point)."""
    N, p, n_obs, sd, dense, kw, n_mcmc = CASES[name]
    ref = do.ModelTrunc(Nmesh=N, p=p)
    P = ref.p
    rs = np.random.RandomState(sum(map(ord, name)))
    truth = rs.normal(size=P)
    U = ref(truth, full_solution=True)
    obs = np.sort(rs.choice(N * N, n_obs, replace=False, p=U / U.sum()))
    ref.obs_index = obs
    Gamma = sd ** 2 * np.eye(n_obs)
    if dense:
        Q = rs.normal(size=(n_obs, n_obs))
        Gamma = sd ** 2 * (np.eye(n_obs) + 0.3 * Q @ Q.T / n_obs)
    y = ref(truth) + np.linalg.cholesky(Gamma) @ rs.normal(size=n_obs)
    J = P + 20
    Ustar = truth[:, None] + 0.05 * rs.normal(size=(P, J))
    prior = multivariate_normal(np.zeros(P), np.eye(P))
    return ref, obs, y, Gamma, Ustar, prior, kw, n_mcmc


def device_model(name, obs):
    N, p = CASES[name][:2]
    m = cdarcy.model(Nmesh=N) if p is None else cdarcy.model_trunc(Nmesh=N, p=p)
    m.obs_index = obs
    m.tol = 1e-13
    return m


def _sampler(Ustar, y, n_obs):
    enka = calibrate.sampling(Ustar.shape[0], n_obs, Ustar.shape[1])
    enka.Ustar = Ustar
    mc = csample.MCMC()
    mc.y_obs = y
    return enka, mc


def _same_state(a, b):
    return np.array_equal(a[1], b[1]) and a[2] == b[2] and a[3] == b[3] and (a[3] == 0 or a[4] == b[4])


@pytest.mark.parametrize("name", sorted(CASES))
def test_chain_zero_is_the_oracle_chain(name):
    ref, obs, y, Gamma, Ustar, prior, kw, n_mcmc = problem(name)
    np.random.seed(21)
    want, want_acc = mo.model_mh(ref, n_mcmc, prior, Ustar, y, Gamma, **kw)
    state = np.random.get_state()
    enka, mc = _sampler(Ustar, y, len(obs))
    m = device_model(name, obs)
    np.random.seed(21)
    mc.model_mh(m, n_mcmc, prior, enka, Gamma, **kw)
    assert mc.samples.shape == want.shape == (ref.p, n_mcmc + 1)
    assert np.abs(mc.samples - want).max() <= 1e-9 * np.abs(want).max(), name
    assert mc.accept == want_acc and 0.0 < want_acc < 1.0, (mc.accept, want_acc)
    assert _same_state(np.random.get_state(), state)
    if name == "trunc16_rw":
        # resume: a second call continues from the last sample (Phi_current still the ensemble mean's)
        want2, want_acc2 = mo.model_mh(ref, 60, prior, Ustar, y, Gamma, samples=want, **kw)
        state2 = np.random.get_state()
        np.random.set_state(state)
        mc.model_mh(m, 60, prior, enka, Gamma, **kw)
        assert mc.samples.shape == want2.shape == (ref.p, n_mcmc + 61)
        assert np.abs(mc.samples - want2).max() <= 1e-9 * np.abs(want2).max()
        assert mc.accept == want_acc2 and _same_state(np.random.get_state(), state2)


def test_many_chains_run_beside_chain_zero():
    ref, obs, y, Gamma, Ustar, prior, kw, n_mcmc = problem("trunc16_rw")
    enka, mc = _sampler(Ustar, y, len(obs))
    m = device_model("trunc16_rw", obs)
    np.random.seed(21)
    mc.model_mh(m, 40, prior, enka, Gamma, n_chains=200, seed=4, **kw)
    one = csample.MCMC()
    one.y_obs = y
    np.random.seed(21)
    one.model_mh(m, 40, prior, enka, Gamma, **kw)
    assert mc.samples_chains.shape == (200, ref.p, 41)
    # chain 0 is the single chain (the batch width only changes which GEMM tile shapes run: last-bit differences)
    assert np.abs(mc.samples - one.samples).max() <= 1e-12 * np.abs(one.samples).max() and mc.accept == one.accept
    assert np.array_equal(mc.samples_chains[0], mc.samples)
    assert np.all(mc.accept_chains > 0.0) and np.all(mc.accept_chains < 1.0)
    assert np.array_equal(mc.samples_chains[1:, :, 0], Ustar.T[np.arange(1, 200) % Ustar.shape[1]])
    assert not np.array_equal(mc.samples_chains[1, :, 1:], mc.samples_chains[1 + Ustar.shape[1], :, 1:])


def test_prior_is_recovered_without_information():
    """Gamma = 1e8 I: the misfit is below 1e-9 for every proposal, so the random walk samples the prior itself.  512 Philox
    chains start from exact prior draws (stationary from the first state) and run 400 steps.  The chains are independent,
    so the Monte Carlo error of a pooled statistic is the spread of its per-chain values over sqrt(512); each pooled mean
    and covariance entry must lie within 5 of those standard errors of the prior's value (plus 1e-12)."""
    N, p, n_obs, C, n_mcmc = 16, 10, 30, 512, 400
    rs = np.random.RandomState(3)
    mu = 0.3 * rs.normal(size=p)
    S = rs.normal(size=(p, p))
    cov = 0.5 * np.eye(p) + 0.5 * S @ S.T / p
    prior = multivariate_normal(mu, cov)
    Ustar = rs.multivariate_normal(mu, cov, size=C).T
    m = cdarcy.model_trunc(Nmesh=N, p=p)
    m.obs_index = rs.choice(N * N, n_obs, replace=False)
    enka, mc = _sampler(Ustar, np.zeros(n_obs), n_obs)
    np.random.seed(0)
    mc.model_mh(m, n_mcmc, prior, enka, 1e8 * np.eye(n_obs), delta=2.38 / np.sqrt(p), enka_scaling=True, n_chains=C, seed=11)
    X = mc.samples_chains[1:, :, 1:]                                   # chain 0 starts at the ensemble mean: left out
    means = X.mean(axis=2)                                             # (chains, p)
    d = X - mu[None, :, None]
    covs = np.einsum("cin,cjn->cij", d, d) / X.shape[2]                # per-chain covariance about the prior mean
    se_mean = means.std(axis=0, ddof=1) / np.sqrt(X.shape[0])
    se_cov = covs.std(axis=0, ddof=1) / np.sqrt(X.shape[0])
    assert np.all(np.abs(means.mean(axis=0) - mu) <= 5 * se_mean + 1e-12), (means.mean(axis=0) - mu) / se_mean
    assert np.all(np.abs(covs.mean(axis=0) - cov) <= 5 * se_cov + 1e-12), np.abs(covs.mean(axis=0) - cov) / se_cov
    assert 0.1 < mc.accept_chains.mean() < 0.6


def test_unconverged_solve_raises_and_changes_nothing():
    ref, obs, y, Gamma, Ustar, prior, kw, n_mcmc = problem("trunc16_rw")
    enka, mc = _sampler(Ustar, y, len(obs))
    m = device_model("trunc16_rw", obs)
    np.random.seed(5)
    mc.model_mh(m, 10, prior, enka, Gamma, **kw)
    before, state = mc.samples.copy(), np.random.get_state()
    m.max_iter = 2
    with pytest.raises(_lib.CesError, match="max_iter = 2"):
        mc.model_mh(m, 10, prior, enka, Gamma, n_chains=3, **kw)
    assert np.array_equal(mc.samples, before) and _same_state(np.random.get_state(), state)
    assert not hasattr(mc, "samples_chains")
    m.max_iter = 0                                          # the default limit again: the same call now runs
    mc.model_mh(m, 10, prior, enka, Gamma, **kw)
    assert mc.samples.shape == (ref.p, 21)


def test_refusals():
    ref, obs, y, Gamma, Ustar, prior, kw, n_mcmc = problem("trunc16_rw")
    enka, mc = _sampler(Ustar, y, len(obs))
    m = cdarcy.model_trunc(Nmesh=16, p=10)
    state = np.random.get_state()
    with pytest.raises(ValueError, match="obs_index"):
        mc.model_mh(m, 10, prior, enka, Gamma, **kw)
    m.obs_index = obs[:-1]
    with pytest.raises(ValueError):                          # n_obs of the ensemble and of the model disagree
        mc.model_mh(m, 10, prior, enka, Gamma, **kw)
    assert _same_state(np.random.get_state(), state) and not hasattr(mc, "samples")
    # the C entry point itself: a handle without observations, n_mcmc / n_chains < 1, NULL arrays
    lib = _lib.load()
    v, mt, g = np.zeros(64 * 64), np.zeros(626, dtype=np.uint32), np.zeros(1)
    acc = np.zeros(4, dtype=np.int32)
    h = m._handle(False)
    args = lambda n_mcmc, n_chains, y_: (y_, v.ctypes.data, v.ctypes.data, v.ctypes.data, v.ctypes.data, 0, 0.5, n_mcmc,
                                         n_chains, v.ctypes.data, v.ctypes.data, mt.ctypes.data, g.ctypes.data, 0,
                                         v.ctypes.data, acc.ctypes.data)
    assert lib.ces_darcy_mh(h, 1e-10, 0, *args(1, 1, v.ctypes.data)) == _lib.CES_ERR_INVALID
    m.obs_index = obs
    h = m._handle(True)
    assert lib.ces_darcy_mh(h, 1e-10, 0, *args(0, 1, v.ctypes.data)) == _lib.CES_ERR_INVALID
    assert lib.ces_darcy_mh(h, 1e-10, 0, *args(1, 0, v.ctypes.data)) == _lib.CES_ERR_INVALID
    assert lib.ces_darcy_mh(h, 1e-10, 0, *args(1, 1, None)) == _lib.CES_ERR_INVALID


def _split_rhat(chains):
    """Split-R^ (Gelman et al., BDA3 11.4) per coordinate of chains (n_chains, p, n)."""
    n = chains.shape[2] // 2
    halves = np.concatenate([chains[:, :, :n], chains[:, :, n:2 * n]], axis=0)
    W = halves.var(axis=2, ddof=1).mean(axis=0)
    B = n * halves.mean(axis=2).var(axis=0, ddof=1)
    return np.sqrt(((n - 1) / n * W + B / n) / W)


def test_calibrate_emulate_sample_example_against_the_true_model():
    """examples/darcy_ces.py at reduced size: the true-model chains have mixed (split-R^ < 1.1 per mode) at a sensible
    acceptance, and the emulator's posterior mean lies within EMU_BOUND true posterior standard deviations of theirs.
    EMU_BOUND is set from the first measured gap (DESIGN.md section 4f): at most 0.043 sd over the 10 modes at this size,
    of the order of the Monte Carlo error of two pooled means of 64 x 2400 correlated samples; 0.2 sd leaves room for that
    noise and still flags an emulator that misplaces the posterior."""
    import importlib.util

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("darcy_ces_example", os.path.join(root, "examples", "darcy_ces.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = mod.main(["--n-mcmc", "3000", "--chains", "64"])
    burn = out["burn"]
    rhat = _split_rhat(out["model_mcmc"].samples_chains[:, :, burn:])
    gap = np.abs(out["emulator_mean"] - out["model_mean"]) / out["model_sd"]
    print("split-R^", np.round(rhat, 3), "emulator gap / sd", np.round(gap, 3), "accept", out["model_accept"])
    assert np.all(rhat < 1.1), rhat
    assert 0.05 < out["model_accept"] < 0.9
    assert np.all(gap < EMU_BOUND), gap


EMU_BOUND = 0.2
