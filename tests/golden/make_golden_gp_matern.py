"""Golden vectors of the Emulate stage's Matern kernels from scikit-learn (and of oracle/gp_matern_oracle.py's chains).

    python tests/golden/make_golden_gp_matern.py   -> tests/golden/gp_matern_cases.npz

The layout follows tests/golden/make_golden_gp.py (the squared-exponential vectors, gp_cases.npz).  The inputs of a case
are stored once: "<case>/X" (p x n), "<case>/G" (whitened outputs, k x n; the device is fed them with Gamma = I) and
"<case>/U" (test points).  Per family f in Matern12 / Matern32 / Matern52 (GPflow's names; sklearn's Matern(nu=0.5 / 1.5
/ 2.5)) and output y_i = G_i - mean(G_i), sklearn pins under "<f>/<case>/...":
  * theta, and the LML and gradient there: GaussianProcessRegressor(C * Matern(ARD, nu) + WhiteKernel, alpha=1e-10);
  * latent mean / var at U: GaussianProcessRegressor(C * Matern(nu), alpha=sn2 + 1e-10), whose std^2 excludes sn2;
  * (fit cases) the fitted theta and LML from oracle.gp_oracle.default_init / default_bounds, n_restarts_optimizer=0.
Cases: p in {1, 2, 8, 32}, n up to 1000, k up to 64, up to 1000 test points -- the large n, the large k and the many
test points on different cases, which keeps the file near 0.5 MB; "dup_*" repeats training points exactly, so r = 0 off
the diagonal; "cond_*" has near-duplicate points and sn2 = 1e-10 (ill-conditioned K; "<f>/<case>/cond" records cond(K)
of output 0).  The chains "<f>/chain/<tag>/..." are oracle.gp_oracle.emulator_mh runs through the oracle emulator
(oracle.gp_matern_oracle.predict) of p2_n100_k10 with numpy's global generator seeded, and its state afterwards: a
random walk ("rw", then 40 steps resumed from its samples) and pCN ("pcn").
"""
import os
import sys
import warnings

import numpy as np
import sklearn
from scipy.stats import multivariate_normal
from sklearn.gaussian_process import GaussianProcessRegressor as GPR
from sklearn.gaussian_process.kernels import ConstantKernel, Matern, WhiteKernel

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import gp_matern_oracle as gm, gp_oracle as go  # noqa: E402

JITTER = 1e-10
FAMILIES = {"Matern12": 0.5, "Matern32": 1.5, "Matern52": 2.5}
FIT_CASES = ("p1_n37_k1", "p2_n100_k10")


def _outputs(rs, X, k, noise):
    """k functions of the inputs (+ noise): the whitened forward map of a case."""
    p, n = X.shape
    W = rs.normal(size=(k, p)) / np.sqrt(p)
    b = rs.uniform(0, 2 * np.pi, size=k)
    amp = rs.uniform(0.5, 3.0, size=k)
    return amp[:, None] * np.sin(W @ X + b[:, None]) + 0.3 * np.abs(W @ X) + 1.0 + noise * rs.normal(size=(k, n))


def cases():
    rs = np.random.RandomState(2025)
    out = []
    # name, X, G, number of test points
    X = rs.uniform(-2, 2, size=(1, 37))
    out.append(("p1_n37_k1", X, _outputs(rs, X, 1, 0.05), 1000))
    X = np.vstack([rs.normal(-1, 0.3, 100), rs.normal(2, 1.5, 100)])            # anisotropic inputs, notebook scale
    out.append(("p2_n100_k10", X, _outputs(rs, X, 10, 0.05), 100))
    X = rs.normal(size=(8, 1000)) * np.linspace(0.5, 2.0, 8)[:, None]
    out.append(("p8_n1000_k4", X, _outputs(rs, X, 4, 0.1), 33))
    X = rs.normal(size=(8, 150)) * np.linspace(0.5, 2.0, 8)[:, None]
    out.append(("p8_n150_k64", X, _outputs(rs, X, 64, 0.1), 17))
    X = rs.normal(size=(32, 200))
    out.append(("p32_n200_k3", X, _outputs(rs, X, 3, 0.1), 50))
    # 12 of 60 points repeated exactly (and two of them three times): r = 0 off the diagonal
    X = rs.uniform(-1, 1, size=(3, 48))
    X = np.hstack([X, X[:, :10], X[:, :2]])
    out.append(("dup_p3_n60_k2", X, _outputs(rs, X, 2, 0.05), 40))
    # near-duplicate points and sn2 = 1e-10: ill-conditioned K
    X = rs.uniform(-1, 1, size=(2, 60))
    X = np.hstack([X, X[:, :40] + 3e-5 * rs.normal(size=(2, 40))])
    out.append(("cond_p2_n100_k1", X, _outputs(rs, X, 1, 0.0), 40))
    return out


def given_theta(rs, X, Y, name):
    init = go.default_init(X, Y)
    th = init + rs.uniform(-0.5, 0.5, size=init.shape)
    th[:, -1] = np.log(np.maximum(np.exp(th[:, -1]), 1e-3 * np.exp(th[:, 0])))
    if name.startswith("cond"):
        th[:, 1:-1] = np.log(0.7)
        th[:, -1] = np.log(1e-10)
    return th


def sk_kernel(th, p, nu, bounds=None):
    b = bounds if bounds is not None else [(1e-5, 1e5)] * 3 + [(1e-10, 1e1)]
    return (ConstantKernel(np.exp(th[0]), b[0]) * Matern(np.exp(th[1:1 + p]), b[1], nu=nu) + WhiteKernel(np.exp(th[-1]), b[3]))


def main():
    rs = np.random.RandomState(8)
    data = {"sklearn_version": np.array(sklearn.__version__), "jitter": np.array(JITTER),
            "families": np.array(list(FAMILIES))}
    names = []
    for name, X, G, m in cases():
        p, n = X.shape
        k = G.shape[0]
        ybar = G.mean(axis=1)
        Y = G - ybar[:, None]
        U = X[:, rs.randint(0, n, m)] + 0.5 * rs.normal(size=(p, m)) * X.std(axis=1)[:, None]
        data.update({name + "/X": X, name + "/G": G, name + "/U": U})
        for fam, nu in FAMILIES.items():
            th = given_theta(rs, X, Y, name)
            lml, grad, mean, var = np.empty(k), np.empty((k, p + 2)), np.empty((k, m)), np.empty((k, m))
            for i in range(k):
                g = GPR(sk_kernel(th[i], p, nu), alpha=JITTER, optimizer=None).fit(X.T, Y[i])
                lml[i], grad[i] = g.log_marginal_likelihood(th[i], eval_gradient=True)
                latent = ConstantKernel(np.exp(th[i][0]), "fixed") * Matern(np.exp(th[i][1:1 + p]), "fixed", nu=nu)
                gl = GPR(latent, alpha=np.exp(th[i][-1]) + JITTER, optimizer=None).fit(X.T, Y[i])
                mu, sd = gl.predict(U.T, return_std=True)
                mean[i], var[i] = ybar[i] + mu, sd ** 2
            c = {"theta": th, "lml": lml, "grad": grad, "mean": mean, "var": var}
            Kf, _ = gm.kernel_f(X, X, th[0], fam)
            c["cond"] = np.array(np.linalg.cond(Kf + (np.exp(th[0][-1]) + JITTER) * np.eye(n)))
            if name in FIT_CASES:
                init, bounds = go.default_init(X, Y), go.default_bounds(p)
                fth, flml = np.empty((k, p + 2)), np.empty(k)
                for i in range(k):
                    with warnings.catch_warnings():
                        warnings.simplefilter("ignore")
                        g = GPR(sk_kernel(init[i], p, nu, [tuple(np.exp(b)) for b in bounds[[0, 1, 1, p + 1]]]),
                                alpha=JITTER, n_restarts_optimizer=0).fit(X.T, Y[i])
                    fth[i], flml[i] = g.kernel_.theta, g.log_marginal_likelihood_value_
                c.update(fit_theta=fth, fit_lml=flml)
            for key, v in c.items():
                data["%s/%s/%s" % (fam, name, key)] = v
            print(fam, name, "lml", lml[:3], "cond %.1e" % c["cond"], "fit" if name in FIT_CASES else "")
        names.append(name)
    data["names"] = np.array(names)

    # chains through the oracle emulator of the notebook-scale case
    name = "p2_n100_k10"
    X, G = data[name + "/X"], data[name + "/G"]
    ybar = G.mean(axis=1)
    Y = G - ybar[:, None]
    ytil = G[:, 7] + 0.05 * rs.normal(size=G.shape[0])
    Ustar = X[:, :60]
    prior = dict(mean=np.array([-1.0, 2.0]), cov=np.array([[1.0, 0.2], [0.2, 4.0]]))
    data["chain/ytil"], data["chain/Ustar"] = ytil, Ustar
    data["chain/prior_mean"], data["chain/prior_cov"] = prior["mean"], prior["cov"]
    pr = multivariate_normal(prior["mean"], prior["cov"])
    for fam in FAMILIES:
        theta = data["%s/%s/theta" % (fam, name)]

        def predict_one(u, theta=theta, fam=fam):
            mu, v = gm.predict(X, Y, ybar, theta, np.asarray(u, dtype=float).reshape(-1, 1), fam, JITTER)
            return mu[:, 0], v[:, 0]

        for tag, kw in (("rw", dict(delta=0.8, enka_scaling=True)), ("pcn", dict(update="pCN", beta=0.05))):
            pre = "%s/chain/%s/" % (fam, tag)
            np.random.seed(13)
            s, acc = go.emulator_mh(predict_one, 150, pr, Ustar, ytil, **kw)
            st = np.random.get_state()
            data[pre + "samples"], data[pre + "accept"] = s, np.array(acc)
            data[pre + "key"], data[pre + "pos"], data[pre + "gauss"] = st[1], np.array([st[2], st[3]]), np.array(st[4])
            if tag == "rw":                                                  # resume: 40 more from the last sample
                s2, acc2 = go.emulator_mh(predict_one, 40, pr, Ustar, ytil, samples=s, **kw)
                st = np.random.get_state()
                data[pre + "samples_resumed"], data[pre + "accept_resumed"] = s2, np.array(acc2)
                data[pre + "key2"], data[pre + "pos2"], data[pre + "gauss2"] = st[1], np.array([st[2], st[3]]), np.array(st[4])
            print(fam, "chain", tag, "accept", acc)
    np.savez_compressed(os.path.join(HERE, "gp_matern_cases.npz"), **data)


if __name__ == "__main__":
    main()
