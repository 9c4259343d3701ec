"""Golden vectors of the Emulate stage from scikit-learn (and of oracle/gp_oracle.py's chains).

    python tests/golden/make_golden_gp.py   -> tests/golden/gp_cases.npz

Every case stores whitened outputs G (k x n) directly (the device is fed them with Gamma = I, whose eigh is exactly the
identity) and the training inputs X (p x n).  sklearn pins, per output y_i = G_i - mean(G_i):
  * LML and gradient at a given theta: GaussianProcessRegressor(C * RBF(ARD) + WhiteKernel, alpha=1e-10);
  * latent predictions at test points U: GaussianProcessRegressor(C * RBF, alpha=sn2 + 1e-10), whose std^2 excludes sn2;
  * (fit cases) the fitted theta and LML from oracle.gp_oracle.default_init / default_bounds, n_restarts_optimizer=0.
The chain cases are oracle.gp_oracle.emulator_mh runs with numpy's global generator seeded, and its state afterwards.
"""
import os
import sys
import warnings

import numpy as np
import sklearn
from scipy.stats import multivariate_normal
from sklearn.gaussian_process import GaussianProcessRegressor as GPR
from sklearn.gaussian_process.kernels import RBF, ConstantKernel, WhiteKernel

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import gp_oracle as go  # noqa: E402

JITTER = 1e-10


def _outputs(rs, X, k, noise):
    """k smooth functions of the inputs (+ noise): the whitened forward map of a case."""
    p, n = X.shape
    W = rs.normal(size=(k, p)) / np.sqrt(p)
    b = rs.uniform(0, 2 * np.pi, size=k)
    amp = rs.uniform(0.5, 3.0, size=k)
    return amp[:, None] * np.sin(W @ X + b[:, None]) + 0.3 * (W @ X) ** 2 / p + 1.0 + noise * rs.normal(size=(k, n))


def cases():
    rs = np.random.RandomState(2024)
    out = []
    # name, X, G, theta (k x (p + 2)), test points, fit?
    X = rs.uniform(-2, 2, size=(1, 37))
    out.append(("p1_n37_k1", X, _outputs(rs, X, 1, 0.05), True, 40))
    X = np.vstack([rs.normal(-1, 0.3, 100), rs.normal(2, 1.5, 100)])            # anisotropic inputs, notebook scale
    out.append(("p2_n100_k10", X, _outputs(rs, X, 10, 0.05), True, 1000))
    X = rs.normal(size=(8, 1000)) * np.linspace(0.5, 2.0, 8)[:, None]
    out.append(("p8_n1000_k64", X, _outputs(rs, X, 64, 0.1), False, 33))
    X = rs.normal(size=(32, 200))
    out.append(("p32_n200_k3", X, _outputs(rs, X, 3, 0.1), True, 50))
    # near-duplicate points and sn2 = 1e-10: cond(K) ~ 1e10
    X = rs.uniform(-1, 1, size=(2, 60))
    X = np.hstack([X, X[:, :40] + 3e-5 * rs.normal(size=(2, 40))])
    out.append(("cond_p2_n100_k1", X, _outputs(rs, X, 1, 0.0), False, 40))
    return out


def given_theta(rs, X, Y, name):
    init = go.default_init(X, Y)
    th = init + rs.uniform(-0.5, 0.5, size=init.shape)
    th[:, -1] = np.log(np.maximum(np.exp(th[:, -1]), 1e-3 * np.exp(th[:, 0])))
    if name.startswith("cond"):
        th[:, 1:-1] = np.log(0.7)
        th[:, -1] = np.log(1e-10)
    return th


def sk_kernel(th, p, bounds=None):
    b = bounds if bounds is not None else [(1e-5, 1e5)] * 3 + [(1e-10, 1e1)]
    return (ConstantKernel(np.exp(th[0]), b[0]) * RBF(np.exp(th[1:1 + p]), b[1]) + WhiteKernel(np.exp(th[-1]), b[3]))


def main():
    rs = np.random.RandomState(7)
    data = {"sklearn_version": np.array(sklearn.__version__), "jitter": np.array(JITTER)}
    names = []
    for name, X, G, do_fit, m in cases():
        p, n = X.shape
        k = G.shape[0]
        ybar = G.mean(axis=1)
        Y = G - ybar[:, None]
        th = given_theta(rs, X, Y, name)
        U = X[:, rs.randint(0, n, m)] + 0.5 * rs.normal(size=(p, m)) * X.std(axis=1)[:, None]
        lml, grad, mean, var = np.empty(k), np.empty((k, p + 2)), np.empty((k, m)), np.empty((k, m))
        for i in range(k):
            g = GPR(sk_kernel(th[i], p), alpha=JITTER, optimizer=None).fit(X.T, Y[i])
            lml[i], grad[i] = g.log_marginal_likelihood(th[i], eval_gradient=True)
            latent = ConstantKernel(np.exp(th[i][0]), "fixed") * RBF(np.exp(th[i][1:1 + p]), "fixed")
            gl = GPR(latent, alpha=np.exp(th[i][-1]) + JITTER, optimizer=None).fit(X.T, Y[i])
            mu, sd = gl.predict(U.T, return_std=True)
            mean[i], var[i] = ybar[i] + mu, sd ** 2
        c = {"X": X, "G": G, "theta": th, "lml": lml, "grad": grad, "U": U, "mean": mean, "var": var}
        if do_fit:
            init, bounds = go.default_init(X, Y), go.default_bounds(p)
            fth, flml = np.empty((k, p + 2)), np.empty(k)
            for i in range(k):
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    g = GPR(sk_kernel(init[i], p, [tuple(np.exp(b)) for b in bounds[[0, 1, 1, p + 1]]]), alpha=JITTER,
                            n_restarts_optimizer=0).fit(X.T, Y[i])
                fth[i], flml[i] = g.kernel_.theta, g.log_marginal_likelihood_value_
            c.update(fit_theta=fth, fit_lml=flml)
        for key, v in c.items():
            data["%s/%s" % (name, key)] = v
        names.append(name)
        print(name, "lml", lml[:3], "fit" if do_fit else "")
    data["names"] = np.array(names)

    # chains through the oracle emulator of the notebook-scale case
    name = "p2_n100_k10"
    X, G, theta = data[name + "/X"], data[name + "/G"], data[name + "/theta"]
    ybar = G.mean(axis=1)
    Y = G - ybar[:, None]
    ytil = G[:, 7] + 0.05 * rs.normal(size=G.shape[0])

    def predict_one(u):
        mu, v = go.predict(X, Y, ybar, theta, np.asarray(u, dtype=float).reshape(-1, 1), JITTER)
        return mu[:, 0], v[:, 0]

    Ustar = X[:, :60]
    prior = dict(mean=np.array([-1.0, 2.0]), cov=np.array([[1.0, 0.2], [0.2, 4.0]]))
    data["chain/ytil"], data["chain/Ustar"] = ytil, Ustar
    data["chain/prior_mean"], data["chain/prior_cov"] = prior["mean"], prior["cov"]
    pr = multivariate_normal(prior["mean"], prior["cov"])
    chains = [("rw", dict(delta=0.8, enka_scaling=True), True), ("rw_fixed", dict(delta=0.1, enka_scaling=False), True),
              ("pcn", dict(update="pCN", beta=0.05), True), ("rw_novar", dict(delta=0.8, enka_scaling=True), False)]
    for tag, kw, use_var in chains:
        np.random.seed(13)
        s, acc = go.emulator_mh(predict_one, 150, pr, Ustar, ytil, use_variance=use_var, **kw)
        st = np.random.get_state()
        data["chain/%s/samples" % tag], data["chain/%s/accept" % tag] = s, np.array(acc)
        data["chain/%s/key" % tag], data["chain/%s/pos" % tag] = st[1], np.array([st[2], st[3]])
        data["chain/%s/gauss" % tag] = np.array(st[4])
        if tag == "rw":                                                      # resume: 40 more from the last sample
            s2, acc2 = go.emulator_mh(predict_one, 40, pr, Ustar, ytil, samples=s, **kw)
            st = np.random.get_state()
            data["chain/rw/samples_resumed"], data["chain/rw/accept_resumed"] = s2, np.array(acc2)
            data["chain/rw/key2"], data["chain/rw/pos2"], data["chain/rw/gauss2"] = st[1], np.array([st[2], st[3]]), np.array(st[4])
        print("chain", tag, "accept", acc)
    np.savez_compressed(os.path.join(HERE, "gp_cases.npz"), **data)


if __name__ == "__main__":
    main()
