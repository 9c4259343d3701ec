"""GPEmulator and MCMC.emulator_mh on the device (ces_b200/emulate.py, csrc/emulate.cu) against scikit-learn's values in
tests/golden/gp_cases.npz and against oracle/gp_oracle.py: LML and gradient, bit-identical repeats, latent predictions,
the ill-conditioned case, non-SPD K, the fit, chains sample for sample with numpy's generator, and the Calibrate ->
Emulate -> Sample example on the analytic posterior."""
import os

import numpy as np
import pytest
from scipy.stats import multivariate_normal

pytestmark = pytest.mark.gpu

from ces_b200 import calibrate, sample as csample  # noqa: E402
from ces_b200.emulate import GPEmulator  # noqa: E402

GP = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gp_cases.npz"))
NAMES = [str(n) for n in GP["names"]]
JITTER = float(GP["jitter"])


def _emulator(name):
    """Golden outputs are already whitened: Gamma = I, whose eigh is exactly the identity, feeds them through unchanged."""
    X, G = GP[name + "/X"], GP[name + "/G"]
    emu = GPEmulator(U=X, G=G, Gamma=np.eye(G.shape[0]), jitter=JITTER)
    assert np.array_equal(emu.transform, np.eye(G.shape[0]))
    return emu


@pytest.mark.parametrize("name", NAMES)
def test_lml_and_gradient_match_sklearn_and_repeat_bitwise(name):
    emu = _emulator(name)
    theta = GP[name + "/theta"]
    lml, grad = emu.log_marginal_likelihood(theta, eval_gradient=True)
    want, want_g = GP[name + "/lml"], GP[name + "/grad"]
    tol = 1e-6 if name.startswith("cond") else 1e-9          # cond(K) ~ 1e10 (see tests/test_gp_oracle.py)
    assert np.all(np.abs(lml - want) <= tol * np.abs(want)), name
    assert np.all(np.abs(grad - want_g) <= tol * np.maximum(np.abs(want_g).max(axis=1, keepdims=True), 1.0)), name
    lml2, grad2 = emu.log_marginal_likelihood(theta, eval_gradient=True)
    assert np.array_equal(lml, lml2) and np.array_equal(grad, grad2)
    assert np.array_equal(emu.log_marginal_likelihood(theta), lml)


@pytest.mark.parametrize("name,m", [("p2_n100_k10", 1), ("p2_n100_k10", 33), ("p2_n100_k10", 1000), ("p8_n1000_k64", 1),
                                    ("p8_n1000_k64", 33), ("p1_n37_k1", 40), ("p32_n200_k3", 50), ("cond_p2_n100_k1", 40)])
def test_predict_matches_sklearn(name, m):
    emu = _emulator(name)
    theta = GP[name + "/theta"]
    emu.set_hyperparameters(np.exp(theta[:, 0]), np.exp(theta[:, 1:-1]), np.exp(theta[:, -1]))
    assert np.allclose(emu.theta, theta, rtol=0, atol=1e-14)
    emu.theta = theta
    mean, var = emu.predict(GP[name + "/U"][:, :m])
    Y = GP[name + "/G"] - GP[name + "/G"].mean(axis=1, keepdims=True)
    scale = np.abs(Y).max(axis=1)[:, None]
    sf2 = np.exp(theta[:, :1])
    assert mean.shape == var.shape == (Y.shape[0], m)
    assert np.all(np.abs(mean - GP[name + "/mean"][:, :m]) <= 1e-10 * scale), name
    assert np.all(var >= 0.0)
    tol_v = 1e-8 if name.startswith("cond") else 1e-10
    assert np.all(np.abs(var - GP[name + "/var"][:, :m]) <= tol_v * sf2), name


def test_non_spd_covariance_raises():
    X = np.zeros((2, 10))                                     # identical points, no noise, no jitter: K = sf2 * ones
    emu = GPEmulator(U=X, G=np.arange(10.0)[None], Gamma=np.eye(1), jitter=0.0)
    th = np.array([[0.0, 0.0, 0.0, np.log(1e-300)]])
    with pytest.raises(np.linalg.LinAlgError):
        emu.log_marginal_likelihood(th)
    emu.theta = th
    with pytest.raises(np.linalg.LinAlgError):
        emu.predict(np.zeros((2, 1)))


@pytest.mark.parametrize("name", [n for n in NAMES if (n + "/fit_lml") in GP.files])
def test_fit_reaches_sklearn_optimum(name):
    emu = _emulator(name)
    emu.fit()
    want = GP[name + "/fit_lml"]
    assert np.all(emu.fit_lml >= want - 1e-8 * np.abs(want)), (emu.fit_lml - want)
    assert np.allclose(emu.log_marginal_likelihood(), emu.fit_lml, rtol=1e-12, atol=0)


def _chain_setup():
    name = "p2_n100_k10"
    emu = _emulator(name)
    emu.theta = GP[name + "/theta"]
    Ustar = GP["chain/Ustar"]
    enka = calibrate.sampling(2, emu.k, Ustar.shape[1])
    enka.Ustar = Ustar
    prior = multivariate_normal(GP["chain/prior_mean"], GP["chain/prior_cov"])
    mc = csample.MCMC()
    mc.y_obs = GP["chain/ytil"]
    return emu, enka, prior, mc


def _state_equal(tag, suffix=""):
    st = np.random.get_state()
    return (np.array_equal(st[1], GP["chain/%s/key%s" % (tag, suffix)]) and [st[2], st[3]] == list(GP["chain/%s/pos%s" % (tag, suffix)])
            and (st[3] == 0 or abs(st[4] - float(GP["chain/%s/gauss%s" % (tag, suffix)])) <= 1e-14 * max(1.0, abs(st[4]))))


@pytest.mark.parametrize("tag,kw,use_var", [("rw", dict(delta=0.8, enka_scaling=True), True),
                                            ("rw_fixed", dict(delta=0.1, enka_scaling=False), True),
                                            ("pcn", dict(update="pCN", beta=0.05), True),
                                            ("rw_novar", dict(delta=0.8, enka_scaling=True), False)])
def test_emulator_mh_chain_zero_is_the_oracle_chain(tag, kw, use_var):
    emu, enka, prior, mc = _chain_setup()
    np.random.seed(13)
    mc.emulator_mh(emu, 150, prior, enka, use_variance=use_var, **kw)
    want = GP["chain/%s/samples" % tag]
    assert mc.samples.shape == want.shape
    assert np.abs(mc.samples - want).max() <= 1e-10 * np.abs(want).max(), tag
    assert abs(mc.accept - float(GP["chain/%s/accept" % tag])) < 1e-12 and _state_equal(tag)
    if tag == "rw":
        mc.emulator_mh(emu, 40, prior, enka, **kw)
        want2 = GP["chain/rw/samples_resumed"]
        assert mc.samples.shape == want2.shape
        assert np.abs(mc.samples - want2).max() <= 1e-10 * np.abs(want2).max()
        assert abs(mc.accept - float(GP["chain/rw/accept_resumed"])) < 1e-12 and _state_equal("rw", "2")


def test_many_chains_run_beside_chain_zero():
    emu, enka, prior, mc = _chain_setup()
    np.random.seed(13)
    mc.emulator_mh(emu, 150, prior, enka, delta=0.8, n_chains=300, seed=3)
    assert mc.samples_chains.shape == (300, 2, 151) and np.all(mc.accept_chains > 0.0)
    assert np.abs(mc.samples - GP["chain/rw/samples"]).max() <= 1e-10 * np.abs(mc.samples).max()
    assert not np.array_equal(mc.samples_chains[1], mc.samples_chains[2])


def test_calibrate_emulate_sample_example():
    """examples/linear_ces_gp.py: sampling.run -> GPEmulator(eks, Gamma).fit() -> emulator_mh with 64 chains reproduces the
    analytic posterior of linear.ipynb to the bounds of the Calibrate -> Sample example."""
    import importlib.util

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("linear_ces_gp_example", os.path.join(root, "examples", "linear_ces_gp.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = mod.main(["--J", "100", "--T", "400", "--n-mcmc", "6000", "--chains", "64"])
    print("mean gap", out["mcmc_mean"] - out["posterior_mean"], "cov ratio", np.diag(out["mcmc_cov"]) / np.diag(out["posterior_cov"]))
    assert np.abs(out["mcmc_mean"] - out["posterior_mean"]).max() < 0.01
    ratio = np.diag(out["mcmc_cov"]) / np.diag(out["posterior_cov"])
    assert np.all(np.abs(ratio - 1.0) < 0.15) and 0.05 < out["accept"] < 0.9
