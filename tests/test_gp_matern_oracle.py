"""oracle/gp_matern_oracle.py (the checker of the device emulator's Matern kernels) against scikit-learn, live and through
the golden vectors of tests/golden/gp_matern_cases.npz; the kernel family's checks in the C ABI and in GPEmulator that
need no GPU."""
import ctypes
import os

import numpy as np
import pytest
from scipy.stats import multivariate_normal

from oracle import gp_matern_oracle as gm, gp_oracle as go

GM = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gp_matern_cases.npz"))
NAMES = [str(n) for n in GM["names"]]
FAMILIES = [str(f) for f in GM["families"]]
NU = {"Matern12": 0.5, "Matern32": 1.5, "Matern52": 2.5}
JITTER = float(GM["jitter"])


def _case(name):
    X, G = GM[name + "/X"], GM[name + "/G"]
    ybar = G.mean(axis=1)
    return X, G - ybar[:, None], ybar


@pytest.mark.parametrize("fam", FAMILIES)
@pytest.mark.parametrize("name", NAMES)
def test_oracle_matches_the_golden_sklearn_values(fam, name):
    X, Y, ybar = _case(name)
    pre = "%s/%s/" % (fam, name)
    theta = GM[pre + "theta"]
    # ill-conditioned K: two correct implementations may differ by ~cond * eps in W = alpha alpha^T - K^-1
    tol = 1e-6 if name.startswith("cond") else 1e-10
    for i in range(Y.shape[0]) if Y.shape[0] <= 10 else (0, 31, 63):
        v, g = gm.lml(X, Y[i], theta[i], fam, JITTER, eval_gradient=True)
        want_v, want_g = GM[pre + "lml"][i], GM[pre + "grad"][i]
        assert abs(v - want_v) <= tol * abs(want_v), (fam, name, i)
        assert np.abs(g - want_g).max() <= tol * max(np.abs(want_g).max(), 1.0), (fam, name, i)
    mean, var = gm.predict(X, Y, ybar, theta, GM[name + "/U"], fam, JITTER)
    scale = np.abs(Y).max(axis=1)[:, None]
    sf2 = np.exp(theta[:, :1])
    # cond(K) up to 7e9: the latent mean too is held to the ill-conditioned bound there
    tol_v = 1e-8 if name.startswith("cond") else 1e-10
    assert np.all(np.abs(mean - GM[pre + "mean"]) <= tol_v * scale), (fam, name)
    assert np.all(np.abs(var - GM[pre + "var"]) <= tol_v * sf2), (fam, name)
    assert np.all(var >= 0.0)


def _live_cases(rs):
    """(X, y): random inputs at three shapes, one with exact duplicate points (r = 0 off the diagonal), and one
    ill-conditioned (near-duplicate points, sn2 = 1e-10; the last entry of each tuple is its log sn2)."""
    out = []
    for p, n in ((1, 20), (3, 150), (32, 60)):
        out.append((rs.normal(size=(p, n)), np.log(1e-2)))
    X = rs.normal(size=(3, 30))
    out.append((np.hstack([X, X[:, :8], X[:, :1]]), np.log(1e-2)))
    X = rs.uniform(-1, 1, size=(2, 40))
    out.append((np.hstack([X, X[:, :30] + 3e-5 * rs.normal(size=(2, 30))]), np.log(1e-10)))
    return out


@pytest.mark.parametrize("fam", ["Matern12", "Matern32", "Matern52"])
def test_oracle_matches_live_sklearn(fam):
    sk = pytest.importorskip("sklearn.gaussian_process")
    from sklearn.gaussian_process.kernels import ConstantKernel, Matern, WhiteKernel

    rs = np.random.RandomState(4)
    for c, (X, log_sn2) in enumerate(_live_cases(rs)):
        p, n = X.shape
        ill = log_sn2 < np.log(1e-5)                                          # noise-free outputs, as sn2 says
        y = np.sin(X.sum(axis=0)) + (0.0 if ill else 0.1) * rs.normal(size=n)
        y -= y.mean()
        theta = np.concatenate([[0.3], rs.uniform(-0.5, 1.0, p), [log_sn2]])
        if ill:
            theta[1:-1] = np.log(0.7)                                         # as the golden cond case
        tol = 1e-6 if ill else 1e-10
        ker = ConstantKernel(1.0) * Matern(np.ones(p), nu=NU[fam]) + WhiteKernel(1.0)
        g = sk.GaussianProcessRegressor(ker, alpha=JITTER, optimizer=None).fit(X.T, y)
        want_v, want_g = g.log_marginal_likelihood(theta, eval_gradient=True)
        v, gr = gm.lml(X, y, theta, fam, JITTER, eval_gradient=True)
        assert abs(v - want_v) <= tol * abs(want_v), (fam, c)
        assert np.all(np.abs(gr - want_g) <= tol * np.abs(want_g).max()), (fam, c)
        assert np.all(np.isfinite(gr))
        U = np.hstack([rs.normal(size=(p, 8)), X[:, :1]])                   # a test point on a training point: r = 0
        latent = ConstantKernel(np.exp(theta[0]), "fixed") * Matern(np.exp(theta[1:1 + p]), "fixed", nu=NU[fam])
        gl = sk.GaussianProcessRegressor(latent, alpha=np.exp(theta[-1]) + JITTER, optimizer=None).fit(X.T, y)
        mu, sd = gl.predict(U.T, return_std=True)
        mean, var = gm.predict(X, y[None], np.zeros(1), theta[None], U, fam, JITTER)
        # ill-conditioned K: the predictions too differ by ~cond * eps (2.2e-8 relative measured for Matern52 here)
        assert np.abs(mean[0] - mu).max() <= tol * np.abs(y).max(), (fam, c)
        assert np.abs(var[0] - sd ** 2).max() <= tol * np.exp(theta[0]), (fam, c)


def test_oracle_rejects_an_unknown_kernel():
    X, _, _ = _case("p2_n100_k10")
    th = GM["Matern52/p2_n100_k10/theta"]
    for bad in ("Matern72", "SquaredExponential"):
        with pytest.raises(ValueError):
            gm.kernel_f(X, X, th[0], bad)


@pytest.mark.parametrize("fam", FAMILIES)
def test_oracle_fit_reaches_the_sklearn_optimum(fam):
    name = "p2_n100_k10"
    X, Y, _ = _case(name)
    _, lml = gm.fit(X, Y[:3], fam, JITTER)
    want = GM["%s/%s/fit_lml" % (fam, name)][:3]
    assert np.all(lml >= want - 1e-8 * np.abs(want)), (fam, lml - want)


@pytest.mark.parametrize("fam", FAMILIES)
def test_oracle_chains_match_the_golden_chains(fam):
    name = "p2_n100_k10"
    X, Y, ybar = _case(name)
    theta = GM["%s/%s/theta" % (fam, name)]

    def predict_one(u):
        mu, v = gm.predict(X, Y, ybar, theta, np.asarray(u, dtype=float).reshape(-1, 1), fam, JITTER)
        return mu[:, 0], v[:, 0]

    prior = multivariate_normal(GM["chain/prior_mean"], GM["chain/prior_cov"])
    pre = "%s/chain/pcn/" % fam
    np.random.seed(13)
    s, acc = go.emulator_mh(predict_one, 150, prior, GM["chain/Ustar"], GM["chain/ytil"], update="pCN", beta=0.05)
    assert np.abs(s - GM[pre + "samples"]).max() <= 1e-12 * np.abs(s).max()
    assert acc == float(GM[pre + "accept"])
    st = np.random.get_state()
    assert np.array_equal(st[1], GM[pre + "key"]) and [st[2], st[3]] == list(GM[pre + "pos"])


def test_set_kernel_abi_rejects_bad_arguments_without_a_gpu():
    from ces_b200 import _lib

    lib = _lib.load()
    for kind in range(4):
        assert lib.ces_gp_set_kernel(None, kind) == _lib.CES_ERR_INVALID
    assert b"ces_gp_set_kernel" in lib.ces_last_error()
    # an unknown kind is refused before the model is touched (a zeroed host block stands in for one: were it written,
    # the call would return CES_OK and the block would change)
    block = ctypes.create_string_buffer(4096)
    for kind in (-1, 4, 72):
        assert lib.ces_gp_set_kernel(ctypes.cast(block, ctypes.c_void_p), kind) == _lib.CES_ERR_INVALID
    assert block.raw == bytes(4096)
    assert sorted(_lib.GP_KERNELS.values()) == [0, 1, 2, 3]


def test_header_names_the_kernel_constants():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    from ces_b200 import _lib

    header = open(os.path.join(root, "include", "ces_b200.h")).read()
    for name, c in (("SquaredExponential", "CES_GP_SE"), ("Matern12", "CES_GP_MATERN12"), ("Matern32", "CES_GP_MATERN32"),
                    ("Matern52", "CES_GP_MATERN52")):
        assert "#define %s %d " % (c, _lib.GP_KERNELS[name]) in header, c


def test_emulator_rejects_an_unknown_kernel_before_any_device_work():
    from ces_b200.emulate import GPEmulator

    with pytest.raises(ValueError, match="Matern72"):
        GPEmulator(U=np.zeros((2, 5)), G=np.zeros((1, 5)), Gamma=np.eye(1), kernel="Matern72")
    with pytest.raises(ValueError):
        GPEmulator(U=np.zeros((2, 5)), G=np.zeros((1, 5)), Gamma=np.eye(1), kernel="matern52")
