"""oracle/gp_oracle.py (the checker of the device emulator) against scikit-learn, live and through the golden vectors of
tests/golden/gp_cases.npz; the misfit identity that ties emulator_mh to model_mh; argument checks of the C ABI (CPU)."""
import ctypes
import os

import numpy as np
import pytest
from scipy.stats import multivariate_normal

from oracle import gp_oracle as go, mcmc_oracle as mo

GP = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gp_cases.npz"))
NAMES = [str(n) for n in GP["names"]]
JITTER = float(GP["jitter"])


def _case(name):
    X, G = GP[name + "/X"], GP[name + "/G"]
    ybar = G.mean(axis=1)
    return X, G - ybar[:, None], ybar


@pytest.mark.parametrize("name", NAMES)
def test_oracle_matches_the_golden_sklearn_values(name):
    X, Y, ybar = _case(name)
    theta = GP[name + "/theta"]
    # cond(K) ~ 1e10: two correct implementations may differ by ~cond * eps in W = alpha alpha^T - K^-1
    tol = 1e-6 if name.startswith("cond") else 1e-10
    for i in range(Y.shape[0]) if Y.shape[0] <= 10 else (0, 31, 63):
        v, g = go.lml(X, Y[i], theta[i], JITTER, eval_gradient=True)
        want_v, want_g = GP[name + "/lml"][i], GP[name + "/grad"][i]
        assert abs(v - want_v) <= tol * abs(want_v), (name, i)
        assert np.abs(g - want_g).max() <= tol * max(np.abs(want_g).max(), 1.0), (name, i)
    U = GP[name + "/U"]
    mean, var = go.predict(X, Y, ybar, theta, U, JITTER)
    scale = np.abs(Y).max(axis=1)[:, None]
    sf2 = np.exp(theta[:, :1])
    tol_v = 1e-8 if name.startswith("cond") else 1e-10
    assert np.all(np.abs(mean - GP[name + "/mean"]) <= 1e-10 * scale), name
    assert np.all(np.abs(var - GP[name + "/var"]) <= tol_v * sf2), name
    assert np.all(var >= 0.0)


def test_oracle_matches_live_sklearn():
    sk = pytest.importorskip("sklearn.gaussian_process")
    from sklearn.gaussian_process.kernels import RBF, ConstantKernel, WhiteKernel

    rs = np.random.RandomState(3)
    for p, n in ((1, 20), (3, 150), (32, 60)):
        X = rs.normal(size=(p, n))
        y = np.sin(X.sum(axis=0)) + 0.1 * rs.normal(size=n)
        y -= y.mean()
        theta = np.concatenate([[0.3], rs.uniform(-0.5, 1.0, p), [np.log(1e-2)]])
        ker = ConstantKernel(1.0) * RBF(np.ones(p)) + WhiteKernel(1.0)
        g = sk.GaussianProcessRegressor(ker, alpha=JITTER, optimizer=None).fit(X.T, y)
        want_v, want_g = g.log_marginal_likelihood(theta, eval_gradient=True)
        v, gr = go.lml(X, y, theta, JITTER, eval_gradient=True)
        assert abs(v - want_v) <= 1e-10 * abs(want_v)
        assert np.all(np.abs(gr - want_g) <= 1e-10 * np.abs(want_g).max())
        U = rs.normal(size=(p, 9))
        latent = ConstantKernel(np.exp(theta[0]), "fixed") * RBF(np.exp(theta[1:1 + p]), "fixed")
        gl = sk.GaussianProcessRegressor(latent, alpha=np.exp(theta[-1]) + JITTER, optimizer=None).fit(X.T, y)
        mu, sd = gl.predict(U.T, return_std=True)
        mean, var = go.predict(X, y[None], np.zeros(1), theta[None], U, JITTER)
        assert np.abs(mean[0] - mu).max() <= 1e-10 * np.abs(y).max()
        assert np.abs(var[0] - sd ** 2).max() <= 1e-10 * np.exp(theta[0])


def test_oracle_fit_reaches_the_sklearn_optimum():
    name = "p2_n100_k10"
    X, Y, _ = _case(name)
    theta, lml = go.fit(X, Y[:3], JITTER)
    want = GP[name + "/fit_lml"][:3]
    assert np.all(lml >= want - 1e-8 * np.abs(want))


def test_oracle_chains_match_the_golden_chains():
    name = "p2_n100_k10"
    X, Y, ybar = _case(name)
    theta = GP[name + "/theta"]

    def predict_one(u):
        mu, v = go.predict(X, Y, ybar, theta, np.asarray(u, dtype=float).reshape(-1, 1), JITTER)
        return mu[:, 0], v[:, 0]

    prior = multivariate_normal(GP["chain/prior_mean"], GP["chain/prior_cov"])
    np.random.seed(13)
    s, acc = go.emulator_mh(predict_one, 150, prior, GP["chain/Ustar"], GP["chain/ytil"], delta=0.8, enka_scaling=True)
    assert np.abs(s - GP["chain/rw/samples"]).max() <= 1e-12 * np.abs(s).max()
    assert acc == float(GP["chain/rw/accept"])
    st = np.random.get_state()
    assert np.array_equal(st[1], GP["chain/rw/key"]) and [st[2], st[3]] == list(GP["chain/rw/pos"])


def test_misfit_without_variance_is_model_mh_misfit():
    """use_variance=False: 1/2 |ytil - mean|^2 = (y - G)^T (2 Gamma)^-1 (y - G) with G = T^-1 mean, so emulator_mh on an
    exact emulator samples what model_mh samples."""
    rs = np.random.RandomState(11)
    for k in (1, 5, 64):
        Q = rs.normal(size=(k, k))
        Gamma = 0.1 * (np.eye(k) + Q @ Q.T / k)
        T = go.whitening(Gamma)
        assert np.allclose(T @ Gamma @ T.T, np.eye(k), atol=1e-12)
        y, Gu = rs.normal(size=k), rs.normal(size=k)
        model = (y - Gu).dot(np.linalg.solve(2.0 * Gamma, y - Gu))
        emulated = go.phi(T @ Gu, np.zeros(k), T @ y, use_variance=False)
        assert abs(model - emulated) <= 1e-12 * abs(model)
    # and the whole chain: emulator_mh with an exact linear emulator is model_mh's chain
    p, k = 2, 6
    A = rs.normal(size=(k, p))
    Q = rs.normal(size=(k, k))
    Gamma = 0.05 * (np.eye(k) + Q @ Q.T / k)
    T = go.whitening(Gamma)
    y = A @ np.array([0.3, -0.5]) + 0.1 * rs.normal(size=k)
    Ustar = np.array([[0.3], [-0.5]]) + 0.1 * rs.normal(size=(p, 30))
    prior = multivariate_normal(np.zeros(p), np.eye(p))
    np.random.seed(5)
    want, want_acc = mo.model_mh(lambda th: A @ th, 200, prior, Ustar, y, Gamma, delta=0.8)
    np.random.seed(5)
    got, acc = go.emulator_mh(lambda u: (T @ (A @ u), np.zeros(k)), 200, prior, Ustar, T @ y, delta=0.8, use_variance=False)
    assert np.abs(got - want).max() <= 1e-10 * np.abs(want).max() and acc == want_acc


def test_gp_abi_rejects_bad_arguments_without_a_gpu():
    from ces_b200 import _lib

    lib = _lib.load()
    X, Y, yb = np.zeros(33 * 8), np.zeros(65 * 8), np.zeros(65)
    h = ctypes.c_void_p()
    for p, k, n in ((33, 1, 8), (1, 65, 8), (1, 1, 1), (0, 1, 8)):
        assert lib.ces_gp_create(None, p, k, n, X.ctypes.data, Y.ctypes.data, yb.ctypes.data, ctypes.byref(h)) == _lib.CES_ERR_INVALID
    assert lib.ces_gp_create(None, 1, 1, 8, None, Y.ctypes.data, yb.ctypes.data, ctypes.byref(h)) == _lib.CES_ERR_INVALID
    assert lib.ces_gp_create(None, 1, 1, 8, X.ctypes.data, Y.ctypes.data, yb.ctypes.data, None) == _lib.CES_ERR_INVALID
    th = np.zeros(3)
    assert lib.ces_gp_lml(None, 0, 1, th.ctypes.data, 1e-10, th.ctypes.data, None) == _lib.CES_ERR_INVALID
    assert lib.ces_gp_condition(None, th.ctypes.data, 1e-10) == _lib.CES_ERR_INVALID
    assert lib.ces_gp_predict(None, None, 1, 1, None, 1, None, 1) == _lib.CES_ERR_INVALID
    assert lib.ces_gp_mh(None, None, 1, None, None, None, 0, 0.5, 10, 1, None, None, None, None, 0, None, None) == _lib.CES_ERR_INVALID
    assert lib.ces_gp_destroy(None) == _lib.CES_OK
