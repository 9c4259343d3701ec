"""Emulate stage: exact Gaussian-process emulators of the forward map on the device (csrc/emulate.cu).

The Calibrate -> Emulate -> Sample pipeline trains one GP per output on the calibrated ensemble ``(Ustar, Gstar)`` and then
runs Metropolis-Hastings on the emulator (``MCMC.emulator_mh``) instead of the expensive model.  The model is GPflow's
``GPR`` + ``SquaredExponential`` (ARD) + ``Gaussian`` likelihood -- scikit-learn's ``C * RBF + WhiteKernel`` -- or, with
``kernel="Matern12"`` / ``"Matern32"`` / ``"Matern52"``, GPflow's Matern kernel of that order (sklearn's
``C * Matern(nu=0.5 / 1.5 / 2.5) + WhiteKernel``), with the same hyperparameters:

Whitening (host, once): ``Gamma = Q diag(lam) Q^T`` (``numpy.linalg.eigh``), ``T = diag(lam^-1/2) Q^T``; the training
outputs are ``Y = T G``, each row centred by its mean ``ybar_i`` (a constant mean function).  ``transform`` (T) and
``offset`` (ybar) are stored and never recomputed: with repeated eigenvalues the eigenvectors are not unique.  In whitened
coordinates the noise covariance is I, so the outputs get independent GPs.

Per output i: ``theta_i = [log sf2, log l_1..l_p, log sn2]`` (sklearn's order; GPflow's ``kernel.variance``,
``kernel.lengthscales``, ``likelihood.variance``),
    r = |(x - z) / l|,   k(x, z) = sf2 exp(-r^2/2)                            (SquaredExponential)
                                   sf2 exp(-r)                               (Matern12)
                                   sf2 (1 + sqrt3 r) exp(-sqrt3 r)           (Matern32)
                                   sf2 (1 + sqrt5 r + 5 r^2 / 3) exp(-sqrt5 r)   (Matern52)
    K = k(X, X) + (sn2 + jitter) I,   L = chol(K),   alpha = K^-1 y_i
    LML = -1/2 y_i^T alpha - sum log L_jj - n/2 log 2 pi,   dLML/dtheta = 1/2 tr((alpha alpha^T - K^-1) dK/dtheta)
    mean_i(u) = ybar_i + k_i(u)^T alpha,   var_i(u) = max(sf2 - |L^-1 k_i(u)|^2, 0)       (latent f: GPflow's predict_f)
The emulated misfit of ``MCMC.emulator_mh`` at the whitened data ``ytil = T y_obs`` is
    Phi(u) = 1/2 sum_i (ytil_i - mean_i)^2 / (1 + var_i) + 1/2 sum_i log(1 + var_i)     (use_variance=True)
    Phi(u) = 1/2 sum_i (ytil_i - mean_i)^2  =  (y - G)^T (2 Gamma)^-1 (y - G),  G = T^-1 mean   (use_variance=False)
Limits: p <= 32, k <= 64, n >= 2.
"""
import ctypes

import numpy as np
import scipy.optimize

from . import _lib


class GPEmulator(object):
    """One exact GP per whitened output, trained on ``enka.Ustar`` / ``enka.Gstar`` (or ``U`` (p x n) / ``G`` (k x n))."""

    def __init__(self, enka=None, Gamma=None, U=None, G=None, jitter=1e-10, kernel="SquaredExponential"):
        import torch

        if kernel not in _lib.GP_KERNELS:
            raise ValueError("GPEmulator: kernel must be one of %s, got %r" % (", ".join(_lib.GP_KERNELS), kernel))
        if not torch.cuda.is_available():
            raise RuntimeError("ces_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        if Gamma is None:
            raise ValueError("GPEmulator needs the noise covariance Gamma (the outputs are whitened by it)")
        U = np.asarray(enka.Ustar if U is None else U, dtype=np.float64)
        G = np.asarray(enka.Gstar if G is None else G, dtype=np.float64)
        self.p, self.n = U.shape
        self.k = G.shape[0]
        if G.shape[1] != self.n:
            raise ValueError("U (p x n) and G (k x n) disagree on n")
        lam, Q = np.linalg.eigh(np.asarray(Gamma, dtype=np.float64).reshape(self.k, self.k))
        self.transform = (Q / np.sqrt(lam)).T                       # T Gamma T^T = I
        Yw = self.transform @ G
        self.offset = Yw.mean(axis=1)
        self.X = np.ascontiguousarray(U)
        self.Y = np.ascontiguousarray(Yw - self.offset[:, None])
        self.jitter = float(jitter)
        self._lib = _lib.load()
        self._stream = torch.cuda.current_stream()
        h = ctypes.c_void_p()
        _lib.check(self._lib.ces_gp_create(ctypes.c_void_p(self._stream.cuda_stream), self.p, self.k, self.n,
                                           _lib.host_ptr(self.X), _lib.host_ptr(self.Y),
                                           _lib.host_ptr(np.ascontiguousarray(self.offset)), ctypes.byref(h)))
        self._h = h
        self._kernel = kernel
        _lib.check(self._lib.ces_gp_set_kernel(h, _lib.GP_KERNELS[kernel]))
        self._conditioned = None
        self.theta = self.default_init()

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self._lib.ces_gp_destroy(h)
            self._h = None

    @property
    def kernel(self):
        """The covariance family, by GPflow's class name (fixed at construction)."""
        return self._kernel

    # ---- hyperparameters
    def default_init(self):
        """sf2 = row variance of the outputs, l_d = row std of the inputs, sn2 = 1e-4 sf2 (log space, k x (p + 2))."""
        sf2 = np.var(self.Y, axis=1)
        return np.column_stack([np.log(sf2), np.tile(np.log(np.std(self.X, axis=1)), (self.k, 1)), np.log(1e-4 * sf2)])

    def default_bounds(self):
        """sf2, l in [1e-5, 1e5], sn2 in [1e-10, 1e1] (log space, (p + 2) x 2)."""
        return np.log(np.array([[1e-5, 1e5]] * (self.p + 1) + [[1e-10, 1e1]]))

    @property
    def variance(self):
        return np.exp(self.theta[:, 0])

    @property
    def lengthscales(self):
        return np.exp(self.theta[:, 1:1 + self.p])

    @property
    def noise_variance(self):
        return np.exp(self.theta[:, -1])

    def set_hyperparameters(self, variance, lengthscales, noise_variance):
        """Set theta from GPflow-named values (per output, or one value for every output); e.g. reuse a GPflow training
        whose kernel is this emulator's family: ``kernel.variance``, ``kernel.lengthscales``, ``likelihood.variance``."""
        var = np.broadcast_to(np.asarray(variance, dtype=np.float64), (self.k,))
        ls = np.broadcast_to(np.asarray(lengthscales, dtype=np.float64).reshape(-1, self.p) if np.ndim(lengthscales) else
                             np.full((1, self.p), float(lengthscales)), (self.k, self.p))
        nv = np.broadcast_to(np.asarray(noise_variance, dtype=np.float64), (self.k,))
        self.theta = np.log(np.column_stack([var, ls, nv]))
        self._conditioned = None

    # ---- marginal likelihood and fit
    def _lml(self, i0, i1, theta, eval_gradient):
        th = np.ascontiguousarray(np.asarray(theta, dtype=np.float64).reshape(i1 - i0, self.p + 2))
        lml = np.empty(i1 - i0)
        grad = np.empty((i1 - i0, self.p + 2)) if eval_gradient else None
        _lib.check(self._lib.ces_gp_lml(self._h, i0, i1, _lib.host_ptr(th), self.jitter, _lib.host_ptr(lml),
                                        _lib.host_ptr(grad) if eval_gradient else None))
        return lml, grad

    def log_marginal_likelihood(self, theta=None, eval_gradient=False):
        """LML per output (k) at ``theta`` (k x (p + 2); default: the current one), and its gradient (k x (p + 2)).
        Raises ``numpy.linalg.LinAlgError`` where K is not positive definite."""
        lml, grad = self._lml(0, self.k, self.theta if theta is None else theta, eval_gradient)
        return (lml, grad) if eval_gradient else lml

    def fit(self, init=None, bounds=None):
        """Maximise each output's LML with scipy's L-BFGS-B in log space (sklearn's ``fmin_l_bfgs_b`` procedure); a trial
        point where K is not positive definite scores +inf.  Returns self."""
        init = self.default_init() if init is None else np.asarray(init, dtype=np.float64).reshape(self.k, self.p + 2)
        bounds = self.default_bounds() if bounds is None else np.asarray(bounds, dtype=np.float64)
        theta = np.empty((self.k, self.p + 2))
        self.fit_lml = np.empty(self.k)
        self.fit_evaluations = 0
        for i in range(self.k):
            def obj(th, i=i):
                self.fit_evaluations += 1
                try:
                    v, g = self._lml(i, i + 1, th, True)
                except np.linalg.LinAlgError:
                    return np.inf, np.zeros_like(th)
                return -v[0], -g[0]
            res = scipy.optimize.minimize(obj, init[i], method="L-BFGS-B", jac=True, bounds=bounds)
            theta[i] = res.x
            self.fit_lml[i] = -res.fun
        self.theta = theta
        self._conditioned = None
        return self

    # ---- prediction
    def condition(self):
        """Factor every output's K at the current theta (done on demand by predict / emulator_mh)."""
        key = self.theta.tobytes()
        if self._conditioned != key:
            _lib.check(self._lib.ces_gp_condition(self._h, _lib.host_ptr(np.ascontiguousarray(self.theta)), self.jitter))
            self._conditioned = key
        return self

    def predict_device(self, U):
        """(mean, var) as device tensors (k x m) at the columns of the device tensor U (p x m, float64)."""
        import torch

        self.condition()
        m = U.shape[1]
        mean = torch.empty((self.k, m), dtype=torch.float64, device=U.device)
        var = torch.empty_like(mean)
        _lib.check(self._lib.ces_gp_predict(self._h, ctypes.c_void_p(U.data_ptr()), U.stride(0), m,
                                            ctypes.c_void_p(mean.data_ptr()), mean.stride(0),
                                            ctypes.c_void_p(var.data_ptr()), var.stride(0)))
        return mean, var

    def predict(self, U):
        """Latent prediction at the columns of U (p x m): ``(mean, var)``, each k x m, in whitened coordinates."""
        import torch

        U = np.asarray(U, dtype=np.float64).reshape(self.p, -1)
        ld = -(-U.shape[1] // 16) * 16
        Ud = torch.zeros((self.p, ld), dtype=torch.float64, device="cuda")
        Ud[:, :U.shape[1]] = torch.from_numpy(U)
        mean, var = self.predict_device(Ud[:, :U.shape[1]])
        torch.cuda.current_stream().synchronize()
        return mean.cpu().numpy(), var.cpu().numpy()
