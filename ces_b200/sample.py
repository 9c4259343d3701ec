"""``MCMC`` with the interface of ``ces/sample.py``: the Sample stage that consumes a calibrated ensemble.

``model_mh`` -- random-walk Metropolis-Hastings / pCN on the TRUE forward model (ces/sample.py:121-196) -- runs whole
chains on the GPU (``ces_mcmc_model_mh``, csrc/mcmc.cu): one warp per chain, the proposal / forward map / misfit /
accept loop never leaves the kernel.  Same call signature, same results attributes (``samples`` (p, n + 1), ``accept``),
same resume behaviour (a second call continues from the last sample) and -- for the chain the reference would run -- the
same random numbers: the kernel consumes numpy's global MT19937 stream exactly as ``np.random.normal(0, 1, p)`` followed
by ``np.random.uniform()`` would, and leaves the generator where the reference's loop would leave it.  ``n_chains > 1``
(a new, additive kwarg) runs further independent chains beside it from device noise: ``samples_chains`` /
``accept_chains``.

The forward model must be one of the device maps of ``ces_b200.utils`` (``lineal``, ``lineal_log``, ``elliptic``,
``banana``) with p <= 32, k <= 64, or a Darcy model of ``ces_b200.darcy`` (``model``, ``model_trunc``) with an
``obs_index``: then all chains step in lockstep (``ces_darcy_mh``, csrc/darcy_mh.cu), every step solving each chain's
proposal in one batched Darcy call with the model's ``tol`` / ``max_iter``, and a solve that does not converge makes the
call fail (numpy's generator and ``samples`` untouched) instead of a chain continuing on it.  ``gp_mh`` (Metropolis-Hastings on a GPflow emulator, ces/sample.py:17-119) is not
provided: it needs trained GPflow models (``emulate.predict_gps``, ces/emulate.py:17-79), a third-party library that is
absent here and whose predictions could not be pinned; that half of SURVEY.md section 8f-4 stays out of scope.

``emulator_mh`` (new) is the same sampler on an emulator of the forward model: a ``ces_b200.emulate.GPEmulator`` (exact
GPs on the device, trained on the calibrated ensemble, with any of its kernel families) replaces the model, and the misfit becomes the emulated one in
whitened coordinates (see ces_b200/emulate.py).  Proposals, prior term, accept test, resume behaviour and the random
numbers are ``model_mh``'s.
"""
from __future__ import print_function

import ctypes
import types

import numpy as np

from . import _lib


class MCMC(object):

    def __init__(self):
        self.mute_bar = False

    def gp_mh(self, enka, n_mcmc, prior, delta=1., enka_scaling=True, **kwargs):
        raise NotImplementedError("gp_mh samples a GPflow emulator (ces/sample.py:17-119, ces/emulate.py:17-79); GPflow is "
                                  "not part of this package -- use model_mh on the forward model itself")

    def model_mh(self, model, n_mcmc, prior, enka, Gamma, delta=1., enka_scaling=True, **kwargs):
        """ces/sample.py:121-196.  ``prior``: an object with ``logpdf`` / ``mean`` / ``cov`` (scipy.stats
        multivariate_normal, as in the reference's notebooks).  kwargs: ``update='pCN'``, ``beta`` (reference);
        ``n_chains``, ``seed`` (device chains beside the reference's one)."""
        import torch

        if not torch.cuda.is_available():
            raise RuntimeError("ces_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        kind = getattr(model, 'device_kind', None)
        darcy = kind == 'darcy'
        if getattr(model, 'type', None) != 'map' or (kind not in _lib.MAPS and not darcy) or getattr(model, 'flag_noise', False):
            raise NotImplementedError("model_mh on the device covers the ces_b200.utils maps (lineal, lineal_log, elliptic, "
                                      "banana) and the ces_b200.darcy models without in-model noise; got %r" % (model,))
        p, k = int(enka.p), int(enka.n_obs)
        if darcy:
            obs = getattr(model, 'obs_index', None)
            if obs is None or np.size(obs) == 0:
                raise ValueError("model_mh on a Darcy model needs model.obs_index: the cells whose pressure is observed")
            if int(model.p) != p or np.size(obs) != k:
                raise ValueError("model_mh: the Darcy model has p = %d and %d observed cells, the ensemble p = %d and n_obs = %d"
                                 % (int(model.p), np.size(obs), p, k))
        if kwargs.get('update', None) not in (None, 'pCN'):
            raise ValueError("unknown update %r" % (kwargs.get('update'),))     # the reference would fail on `proposal`
        pcn = kwargs.get('update', None) == 'pCN'
        c = self._chains(p, n_mcmc, prior, enka, delta, enka_scaling, pcn, float(kwargs.get('beta', 0.5)),
                         int(kwargs.get('n_chains', 1)), int(kwargs.get('seed', 0)))
        y = np.ascontiguousarray(np.asarray(self.y_obs, dtype=np.float64).reshape(k))
        Gam = np.asarray(Gamma, dtype=np.float64).reshape(k, k)
        Ginv2 = np.ascontiguousarray(np.linalg.inv(2.0 * Gam))
        if darcy:
            # chains stepped in lockstep through the batched Darcy solver (csrc/darcy_mh.cu), with the model's tol / max_iter
            _lib.check(_lib.load().ces_darcy_mh(model._handle(True), float(model.tol), int(model.max_iter),
                                                _lib.host_ptr(y), _lib.host_ptr(Ginv2), *c.args))
        else:
            A_dev, lda, b_dev, params = model._device_args(torch)
            par = np.ascontiguousarray(params, dtype=np.float64) if params is not None else None
            stream = torch.cuda.current_stream().cuda_stream
            _lib.check(_lib.load().ces_mcmc_model_mh(
                ctypes.c_void_p(stream), _lib.MAPS[kind], p, k,
                ctypes.c_void_p(A_dev.data_ptr()) if A_dev is not None else None, int(lda),
                ctypes.c_void_p(b_dev.data_ptr()) if b_dev is not None else None,
                _lib.host_ptr(par) if par is not None else None, _lib.host_ptr(y), _lib.host_ptr(Ginv2), *c.args))
        self._publish(c, n_mcmc)

    def emulator_mh(self, emulator, n_mcmc, prior, enka, delta=1., enka_scaling=True, update=None, beta=0.5, n_chains=1,
                    seed=0, use_variance=True):
        """``model_mh`` through a ``GPEmulator``: Phi(u) = 1/2 sum_i (ytil_i - mean_i(u))^2 / (1 + var_i(u))
        + 1/2 sum_i log(1 + var_i(u)) (without the variance terms when ``use_variance`` is False), ytil = T y_obs,
        plus -prior.logpdf(u) unless pCN, with mean / var the emulator's latent prediction under its kernel family
        (``emulator.kernel``).  Chains run on the device (csrc/emulate.cu); results as ``model_mh``."""
        p, k = int(emulator.p), int(emulator.k)
        if update not in (None, 'pCN'):
            raise ValueError("unknown update %r" % (update,))
        c = self._chains(p, n_mcmc, prior, enka, delta, enka_scaling, update == 'pCN', float(beta), int(n_chains), int(seed))
        ytil = np.ascontiguousarray(emulator.transform @ np.asarray(self.y_obs, dtype=np.float64).reshape(k))
        emulator.condition()
        _lib.check(_lib.load().ces_gp_mh(emulator._h, _lib.host_ptr(ytil), 1 if use_variance else 0, *c.args))
        self._publish(c, n_mcmc)

    def _chains(self, p, n_mcmc, prior, enka, delta, enka_scaling, pcn, beta, n_chains, seed):
        """The host set-up every device sampler shares (ces/sample.py:123-166): proposal scales, prior mean / precision
        unless pCN, resume, every chain's start and phi_point, numpy's generator state and the output buffers.  ``args``
        are the C arguments from mu_host onwards (include/ces_b200.h)."""
        # RW needs the proposal distribution (:123-129); pCN proposes according to the prior
        if enka_scaling:
            scales = delta * np.linalg.cholesky(np.cov(enka.Ustar).reshape(p, p))
        else:
            scales = delta * np.eye(p)
        if pcn:
            scales = np.linalg.cholesky(np.asarray(prior.cov, dtype=np.float64).reshape(p, p))
        mean = np.asarray(enka.Ustar, dtype=np.float64).mean(axis=1)            # :131
        mu = Pinv = None
        if not pcn:
            mu = np.ascontiguousarray(np.asarray(prior.mean, dtype=np.float64).reshape(p))
            Pinv = np.ascontiguousarray(np.linalg.inv(np.asarray(prior.cov, dtype=np.float64).reshape(p, p)))
        # resume (:156-164): continue from the last sample; Phi_current stays the ensemble mean's, like the reference
        c = types.SimpleNamespace(previous=None)
        if hasattr(self, 'samples'):
            c.previous = np.asarray(self.samples, dtype=np.float64)
            first = c.previous[:, -1].copy()
        else:
            first = mean.copy()
        start = np.tile(first, (n_chains, 1))
        if n_chains > 1:
            # the extra chains start from ensemble members (over-dispersed starts), deterministically chosen
            J = enka.Ustar.shape[1]
            start[1:] = np.asarray(enka.Ustar, dtype=np.float64).T[np.arange(1, n_chains) % J]
        phi_point = np.tile(mean, (n_chains, 1))
        phi_point[1:] = start[1:]
        # numpy's global generator: ('MT19937', key[624], pos, has_gauss, cached_gaussian)
        st = np.random.get_state()
        c.mt = np.empty(626, dtype=np.uint32)
        c.mt[:624], c.mt[624], c.mt[625] = st[1], st[2], st[3]
        c.gauss = np.array([st[4]], dtype=np.float64)
        c.samples = np.empty((n_chains, int(n_mcmc) + 1, p))
        c.accepted = np.zeros(n_chains, dtype=np.int32)
        # the C arguments point into these arrays: they live as long as c
        c.inputs = (mu, Pinv, np.ascontiguousarray(scales, dtype=np.float64), start, phi_point)
        mu_p, Pinv_p, scales_p, start_p, phi_p = (_lib.host_ptr(a) if a is not None else None for a in c.inputs)
        c.args = (mu_p, Pinv_p, scales_p, 1 if pcn else 0, beta, int(n_mcmc), n_chains, start_p, phi_p, c.mt.ctypes.data,
                  _lib.host_ptr(c.gauss), seed, _lib.host_ptr(c.samples), c.accepted.ctypes.data)
        return c

    def _publish(self, c, n_mcmc):
        """After a successful device run: numpy's advanced generator state and the results attributes of model_mh."""
        np.random.set_state(('MT19937', c.mt[:624].copy(), int(c.mt[624]), int(c.mt[625]), float(c.gauss[0])))
        chain0 = c.samples[0]
        if c.previous is not None:
            # the reference appends to list(self.samples.T) WITHOUT repeating the state it resumes from (:158-160)
            chain0 = np.vstack([c.previous.T, c.samples[0][1:]])
        self.samples = np.array(chain0).T                    # (p, n + 1), :195
        self.accept = c.accepted[0] / float(n_mcmc)          # :196
        if len(c.accepted) > 1:
            self.samples_chains = c.samples.transpose(0, 2, 1)     # (n_chains, p, n + 1)
            self.accept_chains = c.accepted / float(n_mcmc)

    def random_walk(self, current, scales, n_dim):
        """ces/sample.py:198-199 (host helper, kept for API parity; the device chains draw their own)."""
        return current + np.matmul(scales, np.random.normal(0, 1, n_dim))

    def pCN(self, current, scales, n_dim, beta=0.5):
        """ces/sample.py:201-202."""
        return np.sqrt(1 - beta ** 2) * current + np.sqrt(beta) * np.matmul(scales, np.random.normal(0, 1, n_dim))
