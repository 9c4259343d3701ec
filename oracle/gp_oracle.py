"""numpy restatement of the Emulate stage (ces_b200/emulate.py, csrc/emulate.cu) and of ``MCMC.emulator_mh``.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py) -- the checker of the device emulator, never the product.

Parity: PINNED to scikit-learn.  The model is GPflow's ``GPR`` + ``SquaredExponential`` (ARD) + ``Gaussian`` likelihood,
which scikit-learn implements independently as ``GaussianProcessRegressor(ConstantKernel * RBF + WhiteKernel,
alpha=jitter)``; tests/test_gp_oracle.py compares this module with live sklearn and with tests/golden/gp_cases.npz
(tests/golden/make_golden_gp.py, sklearn's LML, gradient, predictions and fitted hyperparameters).

Per output i (whitened and centred training outputs y = Y[i], inputs X (p x n), one point per column):
    theta = [log sf2, log l_1..l_p, log sn2]
    K = sf2 exp(-1/2 |(x - z) / l|^2) + (sn2 + jitter) I,  L = chol(K),  alpha = K^-1 y
    LML = -1/2 y^T alpha - sum log L_jj - n/2 log 2 pi,  dLML/dtheta_j = 1/2 tr(W dK/dtheta_j),  W = alpha alpha^T - K^-1
    mean(u) = ybar + k(u)^T alpha,  var(u) = max(sf2 - |L^-1 k(u)|^2, 0)      (latent f: without sn2)
"""
import numpy as np
import scipy.linalg
import scipy.optimize

LOG_2PI = np.log(2.0 * np.pi)


def whitening(Gamma):
    """T = diag(lam^-1/2) Q^T from Gamma = Q diag(lam) Q^T (numpy.linalg.eigh); T Gamma T^T = I."""
    lam, Q = np.linalg.eigh(np.asarray(Gamma, dtype=float))
    return (Q / np.sqrt(lam)).T


def kernel_f(A, B, theta):
    """sf2 exp(-1/2 sum_d (a_d - b_d)^2 / l_d^2) between the columns of A (p x na) and B (p x nb); also the scaled
    squared differences per dimension (p x na x nb)."""
    theta = np.asarray(theta, dtype=float)
    p = A.shape[0]
    l = np.exp(theta[1:1 + p])
    D = (A / l[:, None])[:, :, None] - (B / l[:, None])[:, None, :]
    D2 = D * D
    return np.exp(theta[0]) * np.exp(-0.5 * D2.sum(axis=0)), D2


def lml(X, y, theta, jitter=1e-10, eval_gradient=False):
    """(LML, dLML/dtheta) of one output; LML = -inf (and a zero gradient) where K is not positive definite, as sklearn."""
    theta = np.asarray(theta, dtype=float)
    n = X.shape[1]
    Kf, D2 = kernel_f(X, X, theta)
    K = Kf + (np.exp(theta[-1]) + jitter) * np.eye(n)
    try:
        L = np.linalg.cholesky(K)
    except np.linalg.LinAlgError:
        return (-np.inf, np.zeros_like(theta)) if eval_gradient else -np.inf
    alpha = scipy.linalg.cho_solve((L, True), y)
    value = -0.5 * y.dot(alpha) - np.log(np.diag(L)).sum() - 0.5 * n * LOG_2PI
    if not eval_gradient:
        return value
    W = np.outer(alpha, alpha) - scipy.linalg.cho_solve((L, True), np.eye(n))
    grad = np.empty_like(theta)
    grad[0] = 0.5 * (W * Kf).sum()
    grad[1:-1] = 0.5 * np.einsum("ab,dab->d", W * Kf, D2)
    grad[-1] = 0.5 * np.exp(theta[-1]) * np.trace(W)
    return value, grad


def default_init(X, Y):
    """Fit start: sf2 = row variance of Y, l_d = row std of X, sn2 = 1e-4 sf2 (log space, k x (p + 2))."""
    sf2 = np.var(Y, axis=1)
    l = np.std(X, axis=1)
    return np.column_stack([np.log(sf2), np.tile(np.log(l), (Y.shape[0], 1)), np.log(1e-4 * sf2)])


def default_bounds(p):
    """sf2, l in [1e-5, 1e5], sn2 in [1e-10, 1e1] (log space, (p + 2) x 2)."""
    return np.log(np.array([[1e-5, 1e5]] * (p + 1) + [[1e-10, 1e1]]))


def minimize(fun_grad, x0, bounds):
    """-LML minimised as sklearn's ``_constrained_optimization('fmin_l_bfgs_b')`` does."""
    res = scipy.optimize.minimize(fun_grad, x0, method="L-BFGS-B", jac=True, bounds=bounds)
    return res.x, -res.fun


def fit(X, Y, jitter=1e-10, init=None, bounds=None):
    """Per-output L-BFGS-B on -LML from ``init`` within ``bounds``; returns (theta (k x (p + 2)), LML (k))."""
    init = default_init(X, Y) if init is None else np.asarray(init, dtype=float)
    bounds = default_bounds(X.shape[0]) if bounds is None else np.asarray(bounds, dtype=float)
    thetas, lmls = [], []
    for i in range(Y.shape[0]):
        def obj(th, y=Y[i]):
            v, g = lml(X, y, th, jitter, eval_gradient=True)
            return -v, -g
        th, v = minimize(obj, init[i], bounds)
        thetas.append(th)
        lmls.append(v)
    return np.array(thetas), np.array(lmls)


def predict(X, Y, ybar, theta, U, jitter=1e-10):
    """(mean, var), each k x m, at the columns of U."""
    k, m = Y.shape[0], U.shape[1]
    mean, var = np.empty((k, m)), np.empty((k, m))
    n = X.shape[1]
    for i in range(k):
        Kf, _ = kernel_f(X, X, theta[i])
        L = np.linalg.cholesky(Kf + (np.exp(theta[i][-1]) + jitter) * np.eye(n))
        alpha = scipy.linalg.cho_solve((L, True), Y[i])
        Ks, _ = kernel_f(X, U, theta[i])
        V = scipy.linalg.solve_triangular(L, Ks, lower=True)
        mean[i] = ybar[i] + Ks.T.dot(alpha)
        var[i] = np.maximum(np.exp(theta[i][0]) - (V * V).sum(axis=0), 0.0)
    return mean, var


def phi(mean, var, ytil, use_variance=True):
    """Emulated misfit of one point (mean, var: k)."""
    r = ytil - mean
    if use_variance:
        return 0.5 * (r * r / (1.0 + var)).sum() + 0.5 * np.log1p(var).sum()
    return 0.5 * (r * r).sum()


def emulator_mh(predict_one, n_mcmc, prior, Ustar, ytil, delta=1.0, enka_scaling=True, update=None, beta=0.5,
                samples=None, use_variance=True, start=None, noise=None):
    """One chain of ``MCMC.emulator_mh``: ``model_mh``'s loop (oracle/mcmc_oracle.py) with Phi the emulated misfit at the
    whitened data ``ytil``; ``predict_one(u) -> (mean (k), var (k))``.  ``start`` and ``noise`` as in
    ``mcmc_oracle.model_mh``.  Returns ``(samples, accept_rate)``."""
    Ustar = np.asarray(Ustar, dtype=float)
    p = Ustar.shape[0]
    if enka_scaling:
        scales = delta * np.linalg.cholesky(np.cov(Ustar).reshape(p, p))
    else:
        scales = delta * np.eye(p)
    if update == "pCN":
        scales = np.linalg.cholesky(prior.cov)

    def Phi(theta):
        v = phi(*predict_one(theta), ytil, use_variance)
        if update != "pCN":
            v -= prior.logpdf(theta)
        return v

    current = Ustar.mean(axis=1) if start is None else np.asarray(start, dtype=float)
    phi_current = Phi(current)
    if samples is not None:
        chain = list(np.asarray(samples).T)
        current = chain[-1]
    else:
        chain = [current.flatten()]
    accept = 0.0
    for it in range(int(n_mcmc)):
        z, u = noise(it) if noise is not None else (np.random.normal(0, 1, p), None)
        if update is None:
            proposal = current + np.matmul(scales, z)
        else:
            proposal = np.sqrt(1 - beta ** 2) * current + np.sqrt(beta) * np.matmul(scales, z)
        phi_proposal = Phi(proposal)
        if u is None:
            u = np.random.uniform()
        if np.log(u) < phi_current - phi_proposal:
            current = np.copy(proposal)
            phi_current = phi_proposal
            accept += 1.0
        chain.append(current.flatten())
    return np.array(chain).T, accept / n_mcmc
