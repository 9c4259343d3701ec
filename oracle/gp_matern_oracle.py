"""numpy restatement of the Emulate stage's Matern kernels (``GPEmulator(kernel="Matern12" / "Matern32" / "Matern52")``,
csrc/emulate.cu).

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py) -- the checker of the device emulator, never the product.

Parity: PINNED to scikit-learn.  The model is GPflow's ``GPR`` + ``Matern12`` / ``Matern32`` / ``Matern52`` (ARD) +
``Gaussian`` likelihood, which scikit-learn implements independently as ``GaussianProcessRegressor(ConstantKernel *
Matern(nu=0.5 / 1.5 / 2.5) + WhiteKernel, alpha=jitter)``; tests/test_gp_matern_oracle.py compares this module with live
sklearn and with tests/golden/gp_matern_cases.npz (tests/golden/make_golden_gp_matern.py).  Everything but the kernel --
theta's layout, whitening, the fit's start and bounds, the misfit and the chains -- is oracle/gp_oracle.py's, which
restates the squared-exponential emulator.

Per output i (whitened and centred training outputs y = Y[i], inputs X (p x n), one point per column):
    theta = [log sf2, log l_1..l_p, log sn2],  D_d = ((x_d - z_d) / l_d)^2,  r = sqrt(sum_d D_d)
    K_f(r) = sf2 exp(-r)                                  (Matern12)
             sf2 (1 + sqrt3 r) exp(-sqrt3 r)              (Matern32)
             sf2 (1 + sqrt5 r + 5 r^2 / 3) exp(-sqrt5 r)  (Matern52)
    K = K_f(X, X) + (sn2 + jitter) I,  L = chol(K),  alpha = K^-1 y
    LML = -1/2 y^T alpha - sum log L_jj - n/2 log 2 pi,  dLML/dtheta_j = 1/2 tr(W dK/dtheta_j),  W = alpha alpha^T - K^-1
    dK/dlog sf2 = K_f,  dK/dlog l_d = sf2 g(r) D_d,  dK/dlog sn2 = sn2 I,  with
        g(r) = exp(-r) / r, and 0 where r = 0 (Matern12; sklearn's convention, duplicate points too),
               3 exp(-sqrt3 r) (Matern32),  5/3 (1 + sqrt5 r) exp(-sqrt5 r) (Matern52)
    mean(u) = ybar + k(u)^T alpha,  var(u) = max(sf2 - |L^-1 k(u)|^2, 0)      (latent f: without sn2)
"""
import numpy as np
import scipy.linalg

from oracle import gp_oracle as go

KERNELS = ("Matern12", "Matern32", "Matern52")


def kernel_f(A, B, theta, kernel):
    """K_f between the columns of A (p x na) and B (p x nb); also the scaled squared differences per dimension
    (p x na x nb)."""
    theta = np.asarray(theta, dtype=float)
    p = A.shape[0]
    l = np.exp(theta[1:1 + p])
    D = (A / l[:, None])[:, :, None] - (B / l[:, None])[:, None, :]
    D2 = D * D
    r = np.sqrt(D2.sum(axis=0))
    if kernel == "Matern12":
        f = np.exp(-r)
    elif kernel == "Matern32":
        t = np.sqrt(3.0) * r
        f = (1.0 + t) * np.exp(-t)
    elif kernel == "Matern52":
        t = np.sqrt(5.0) * r
        f = (1.0 + t + t * t / 3.0) * np.exp(-t)
    else:
        raise ValueError("unknown kernel %r (one of %s)" % (kernel, ", ".join(KERNELS)))
    return np.exp(theta[0]) * f, D2


def kernel_g(D2, kernel):
    """g(r) of dK/dlog l_d = sf2 g(r) D_d, from the scaled squared differences D2 (p x na x nb) of kernel_f."""
    r = np.sqrt(D2.sum(axis=0))
    if kernel == "Matern12":
        pos = r > 0.0
        return np.where(pos, np.exp(-r) / np.where(pos, r, 1.0), 0.0)
    if kernel == "Matern32":
        return 3.0 * np.exp(-np.sqrt(3.0) * r)
    if kernel == "Matern52":
        t = np.sqrt(5.0) * r
        return 5.0 / 3.0 * (1.0 + t) * np.exp(-t)
    raise ValueError("unknown kernel %r (one of %s)" % (kernel, ", ".join(KERNELS)))


def lml(X, y, theta, kernel, jitter=1e-10, eval_gradient=False):
    """(LML, dLML/dtheta) of one output; LML = -inf (and a zero gradient) where K is not positive definite, as sklearn."""
    theta = np.asarray(theta, dtype=float)
    n = X.shape[1]
    Kf, D2 = kernel_f(X, X, theta, kernel)
    K = Kf + (np.exp(theta[-1]) + jitter) * np.eye(n)
    try:
        L = np.linalg.cholesky(K)
    except np.linalg.LinAlgError:
        return (-np.inf, np.zeros_like(theta)) if eval_gradient else -np.inf
    alpha = scipy.linalg.cho_solve((L, True), y)
    value = -0.5 * y.dot(alpha) - np.log(np.diag(L)).sum() - 0.5 * n * go.LOG_2PI
    if not eval_gradient:
        return value
    W = np.outer(alpha, alpha) - scipy.linalg.cho_solve((L, True), np.eye(n))
    grad = np.empty_like(theta)
    grad[0] = 0.5 * (W * Kf).sum()
    grad[1:-1] = 0.5 * np.einsum("ab,dab->d", W * (np.exp(theta[0]) * kernel_g(D2, kernel)), D2)
    grad[-1] = 0.5 * np.exp(theta[-1]) * np.trace(W)
    return value, grad


def fit(X, Y, kernel, jitter=1e-10, init=None, bounds=None):
    """Per-output L-BFGS-B on -LML from ``init`` within ``bounds`` (gp_oracle's defaults); returns (theta, LML)."""
    init = go.default_init(X, Y) if init is None else np.asarray(init, dtype=float)
    bounds = go.default_bounds(X.shape[0]) if bounds is None else np.asarray(bounds, dtype=float)
    thetas, lmls = [], []
    for i in range(Y.shape[0]):
        def obj(th, y=Y[i]):
            v, g = lml(X, y, th, kernel, jitter, eval_gradient=True)
            return -v, -g
        th, v = go.minimize(obj, init[i], bounds)
        thetas.append(th)
        lmls.append(v)
    return np.array(thetas), np.array(lmls)


def predict(X, Y, ybar, theta, U, kernel, jitter=1e-10):
    """(mean, var), each k x m, at the columns of U."""
    k, m = Y.shape[0], U.shape[1]
    mean, var = np.empty((k, m)), np.empty((k, m))
    n = X.shape[1]
    for i in range(k):
        Kf, _ = kernel_f(X, X, theta[i], kernel)
        L = np.linalg.cholesky(Kf + (np.exp(theta[i][-1]) + jitter) * np.eye(n))
        alpha = scipy.linalg.cho_solve((L, True), Y[i])
        Ks, _ = kernel_f(X, U, theta[i], kernel)
        V = scipy.linalg.solve_triangular(L, Ks, lower=True)
        mean[i] = ybar[i] + Ks.T.dot(alpha)
        var[i] = np.maximum(np.exp(theta[i][0]) - (V * V).sum(axis=0), 0.0)
    return mean, var
