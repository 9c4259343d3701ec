"""``enka`` / ``sampling`` with the call signatures of ``ces/calibrate.py``, running the
ensemble Kalman update on a B200 through libces_b200.so.

Drop-in for the numpy update: same constructor, same user-set attributes
(``ustar, mu, sigma, T, parallel, mute_bar, directory, nexp``;
examples/scripts/darcy-flow.py:65-83), same ``run`` / ``eks_update*`` /
``timestep_method`` / ``G`` / ``G_ens`` / ``save`` / ``load`` signatures and the same
result attributes (``Uall, Gall, Ustar, Gstar, metrics, radspec, online_path``;
ces/calibrate.py:404-416).  What differs is where the arithmetic runs:

* ``eks_update*`` take and return numpy arrays like the reference; the copies to
  and from the device are inside the call (``ces_step_host``).
* ``run`` keeps the ensemble resident in HBM between iterations.  Forward models
  that carry a ``device_kind`` (``ces_b200.utils``, ``ces_b200.darcy``) are evaluated
  for the whole ensemble on the device; any other ``model.type == 'map'`` callable is
  evaluated particle by particle on the host exactly as ``enka.G_ens`` does
  (ces/calibrate.py:106-130) -- that is the user's model, not a fallback of ours.
* ``model.type == 'pde'`` models (ODE integrators + statistics, ces/calibrate.py:132-168): the Lorenz models of
  ``ces_b200.utils`` are integrated for the whole ensemble on the device (fixed-step RK4; statistics and the state
  carry-over ``W0`` stay in HBM); any other 'pde' model keeps the reference's host
  protocol for the forward pass (``G_pde_ens``: the user's ``model.solve`` / ``model.statistics`` per particle, joblib
  when ``self.parallel``) with the state carry-over ``W0`` / ``ws`` / ``wt`` / ``update_wt`` semantics of ``run``; the
  update still runs on the device.
* Noise: by default ``xi = np.random.normal(0, 1, [p, J])`` is drawn from the global
  numpy RNG at the point where the reference draws it (ces/calibrate.py:447,488,527),
  so a seeded script consumes the same random stream.
* ``formulation='factored'`` (kwarg of ``run`` / ``eks_update*`` or attribute; default ``'interaction'``) computes
  the same update without forming the J x J matrix D: ``(U - ubar) D = (1/J) ((U - ubar) E^T) W`` and ``||D||_F`` from
  two k x k Gram matrices -- identical to rounding (~1e-15), ``O(d k J + k^2 J)`` instead of ``O((k + d) J^2)``.
* ``rng='device'`` (kwarg of ``run`` or attribute, with ``seed``) generates the noise on the GPU (Philox + Box-Muller,
  ``ces_fill_normal``) instead of drawing it with numpy on the host: a different but equally distributed stream.
* ``noise='ensemble'`` (kwarg of ``run`` / ``eks_update*`` or attribute; default ``'cholesky'``, the reference's
  ``sqrt(2h) chol(C^uu) xi``) forms the noise of eks / aldi / aldi_constant from the ensemble itself:
  ``sqrt(2h / n_C) (U - ubar) xi`` with a J x J ``xi`` (n_C = J for eks, J - 1 for the aldi rules; DESIGN.md section 4g).
  Same covariance as the Cholesky form minus its 1e-8 regularisation, but inside span(U - ubar) and without a
  factorisation.  ``xi`` is drawn on the device from ``seed`` at step ``len(self.metrics['t'])`` unless passed as
  ``xi=``; numpy's global generator is not advanced by the update and ``rng`` does not apply.
* Multi-GPU: if ``self.group`` is a ``torch.distributed`` process group, every rank
  calls ``run`` with the same arguments and the ensemble is sharded by particle
  columns (SURVEY.md section 8e).

There is no CPU implementation of the update in this package: without the CUDA
library or without a GPU these classes raise.
"""
from __future__ import print_function

import hashlib
import multiprocessing
import os
import pickle
import zlib

import numpy as np

from .engine import Engine

_METRIC_KEYS = ("self-bias", "self-bias-data", "bias-data", "bias", "t")
# ``update_rule`` the reference records for each rule (its names: not those of the methods)
_UPDATE_RULE = {"eks": "eks_update", "aldi": "eks_update_linear", "aldi_constant": "eks_update_aldi", "eki": "eki_update"}
# options of ``run`` / ``eks_update*`` that may also be set as attributes, with their defaults
_OPTION_DEFAULTS = {"formulation": "interaction", "noise": "cholesky", "rng": "numpy", "seed": 0}


_SMALL_BYTES = 1 << 20
_pool = None


def _digest(a):
    """Content digest of a problem array: every byte is read.  Small arrays: one blake2b; large ones (a dense Gamma at
    k = 4096 is 128 MB): CRC-32 of 64 chunks on a thread pool (zlib releases the GIL) -- ~10 ms instead of 0.3 s."""
    global _pool
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
    raw = memoryview(a.view(np.uint8).reshape(-1))
    if len(raw) <= _SMALL_BYTES:
        return (a.shape, hashlib.blake2b(raw, digest_size=16).digest())
    if _pool is None:
        from concurrent.futures import ThreadPoolExecutor

        _pool = ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1))
    step = -(-len(raw) // 64)
    return (a.shape, tuple(_pool.map(lambda i: zlib.crc32(raw[i * step:(i + 1) * step]), range(64))))


def _identity(a):
    """Which buffer this is (not what it holds): lets an unchanged caller skip the synchronous digest of large arrays."""
    a = np.asarray(a)
    return (id(a), a.__array_interface__['data'][0], a.shape, a.strides, a.dtype.str)


# Largest J of the one-launch run with noise='ensemble': the kernel draws J^2 / 2 Box-Muller pairs per iteration on one SM.
# Measured per iteration (p = 8, k = 16, B200): 0.61x the per-iteration loop on the phases at J = 256, 1.01x at 384
# (DESIGN.md section 4g, profiles/r08_bench_small_ensemble_noise.json).
_FUSED_ENSEMBLE_J_MAX = 256


def _consume_model_rng(model, n_particles):
    """Advance numpy's global generator by what the reference's per-particle loop over ``model`` would have drawn
    (``rng_draws_per_call`` normals per evaluation; only ``banana`` has any, ces/utils.py:122)."""
    draws = int(getattr(model, 'rng_draws_per_call', 0))
    if draws and n_particles:
        np.random.normal(0, 1, [int(n_particles), draws])


def _save_iteration(where, it, U, G):
    """The online files of iteration ``it``: ``ensemble_NNNN.npy`` / ``Gensemble_NNNN.npy`` in the directory ``where``."""
    np.save(where + 'ensemble_' + str(it).zfill(4), U)
    np.save(where + 'Gensemble_' + str(it).zfill(4), G)


class _HostTrace(object):
    """Device -> host copies of the per-iteration ensembles that do not stall the loop (``trace`` / ``save_online`` of
    ``sampling.run``; SURVEY.md section 8f-1).  ``push`` queues an asynchronous copy into fresh page-locked memory on a side
    stream and returns a ticket; ``get`` waits for that copy only.  ``run`` asks for iteration i's arrays while iteration
    i + 1 is already computing (online save) or at the very end (trace), so the forward solves and updates never wait
    for PCIe.  The source tensors are kept alive until their copy has completed."""

    SMALL = 1 << 18         # below 256 KB a plain synchronous copy is cheaper than a page-locked buffer and two events

    def __init__(self, torch):
        self.torch = torch
        self.stream = None
        self.items = []

    def push(self, a, reused=False):
        """``a``: a device tensor, or a host array that is kept as it is.  ``reused``: the caller overwrites the tensor
        before an asynchronous copy may have completed, so that copy reads a private clone."""
        torch = self.torch
        if isinstance(a, np.ndarray):
            self.items.append((a, None, None))
        elif a.numel() * a.element_size() < self.SMALL:
            self.items.append((a.cpu().numpy(), None, None))
        else:
            if reused:
                a = a.clone()
            if self.stream is None:
                self.stream = torch.cuda.Stream()
            host = torch.empty(a.shape, dtype=a.dtype, pin_memory=True)
            self.stream.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(self.stream):
                host.copy_(a, non_blocking=True)
                done = torch.cuda.Event()
                done.record(self.stream)
            self.items.append((host, done, a))
        return len(self.items) - 1

    def get(self, ticket):
        host, done, _ = self.items[ticket]
        if done is not None:
            done.synchronize()
            host = host.numpy()
            self.items[ticket] = (host, None, None)
        return host


class enka(object):
    """State holder of an ensemble Kalman run.  ces/calibrate.py:12-237."""

    def __init__(self, p, n_obs, J):
        self.n_obs = n_obs          # dimension of the observations
        self.p = p                  # dimension of the parameters
        self.J = J                  # ensemble size
        self.epsilon = 1e-7
        self.T = 30                 # maximum number of iterations
        self.num_cores = multiprocessing.cpu_count()
        self.parallel = False
        self.mute_bar = True
        self._engine = None
        self._engine_key = None
        self._problem_key = None

    # ------------------------------------------------------------------ printing
    def __repr__(self):
        return "enka-%s-%s" % (str(self.J).zfill(4), getattr(self, "_update_name", "eks"))

    def __str__(self):
        print(r'Number of parameters ................. %s' % (self.p))
        print(r'Dimension of forward model output .... %s' % (self.n_obs))
        print(r'Ensemble size ........................ %s' % (self.J))
        print(r'Evaluate G in parallel ............... %s' % (self.parallel))
        print(r'Number of iterations to be run ....... %s' % (self.T))
        if not hasattr(self, "directory"):
            self.directory = os.getcwd()
        print('Path to save: ......................... %s' % ('~/.../' + '/'.join(self.directory.split('/')[-2:])))
        if hasattr(self, "Uall"):
            print(r'Number of iterations EKS has run ..... %s' % (len(self.Uall) - 1))
        else:
            print(r'NOTE: EKS has not been run!')
        return str()

    # ------------------------------------------------------------------ stubs kept for API parity
    def run(self, y_obs, U0, model, Gamma, Jnoise):
        """Placeholder in the reference (ces/calibrate.py:50-68); ``sampling.run`` is the algorithm."""
        pass

    def run_sde(self, y_obs, U0, model, Gamma, Jnoise):
        """Placeholder in the reference (ces/calibrate.py:70-87)."""
        pass

    # ------------------------------------------------------------------ forward evaluation
    def G(self, theta, model):
        """One particle through the forward model (ces/calibrate.py:95-104)."""
        return model(theta)

    def G_ens(self, theta, model):
        """Forward model for a (p, N) collection of particles -> (n_obs, N)  (ces/calibrate.py:106-130).

        Device maps run as one batched call on the GPU; other callables keep the reference's
        per-particle host protocol (joblib when ``self.parallel``)."""
        theta = np.asarray(theta, dtype=np.float64)
        if self._is_device_model(model):
            import torch

            n = theta.shape[1]
            if n == 0:
                return np.zeros((self.n_obs, 0))
            width = max(n, 2)                      # a handle needs at least two particles
            padded = np.empty((theta.shape[0], width))
            padded[:, :n] = theta
            padded[:, n:] = theta[:, -1:]
            # forward-only handle, kept between calls of the same shape
            key = (theta.shape[0], int(self.n_obs), width, torch.cuda.current_device())
            cache = getattr(self, "_forward_cache", None)
            if cache is None or cache[0] != key:
                if cache is not None:
                    cache[1].close()
                cache = (key, Engine(theta.shape[0], self.n_obs, width, d_panel_bytes=-1))
                self._forward_cache = cache
            U = torch.from_numpy(padded).cuda()
            G = torch.empty(self.n_obs, width, dtype=torch.float64, device="cuda")
            model.evaluate_ensemble(cache[1], U, G)
            _consume_model_rng(model, n)
            return G[:, :n].cpu().numpy()
        return self._host_G_ens(theta, model)

    def _host_G_ens(self, theta, model):
        if self.parallel:
            from joblib import Parallel, delayed

            cols = Parallel(n_jobs=self.num_cores)(delayed(self.G)(col, model) for col in theta.T)
            return np.asarray(cols).T
        out = np.zeros((self.n_obs, theta.shape[1]))
        for j, col in enumerate(theta.T):
            out[:, j] = model(col)
        return out

    def G_pde(self, k, model, t):
        """One particle of an ODE/PDE-constrained model (ces/calibrate.py:132-154): ``k`` stacks the p parameters
        and the n_state initial condition; returns the statistics followed by the final state."""
        w0 = k[self.p:]
        ws = model.solve(w0, t, args=tuple(k[:self.p]))
        gs = model.statistics(ws)
        return np.concatenate([gs, ws[-1]])

    def G_pde_ens(self, theta, model, t):
        """``G_pde`` for every column of theta (ces/calibrate.py:156-168): rows [:p] are the parameters, rows [p:] the
        initial state of each particle; returns the statistics stacked on the final states.  The Lorenz models of
        ``ces_b200.utils`` integrate the whole set in one device launch; any other model runs the user's (scipy) code on
        the host, one particle at a time or through joblib like the reference."""
        theta = np.asarray(theta, dtype=np.float64)
        if getattr(model, 'device_kind', None) is not None and hasattr(model, 'evaluate_ensemble_pde'):
            import torch

            n = theta.shape[1]
            U = torch.from_numpy(np.ascontiguousarray(theta[:self.p])).cuda()
            W0 = torch.from_numpy(np.ascontiguousarray(theta[self.p:])).cuda()
            G = torch.empty(self.n_obs, n, dtype=torch.float64, device="cuda")
            Wend = torch.empty_like(W0)
            if n:
                model.evaluate_ensemble_pde(None, U, W0, t, G, Wend)
            return np.vstack([G.cpu().numpy(), Wend.cpu().numpy()])
        if self.parallel:
            from joblib import Parallel, delayed

            cols = Parallel(n_jobs=self.num_cores)(delayed(self.G_pde)(col, model, t) for col in theta.T)
            return np.asarray(cols).T
        out = np.zeros((self.n_obs + model.n_state, theta.shape[1]))
        for j, col in enumerate(theta.T):
            out[:, j] = self.G_pde(col, model, t)
        return out

    @staticmethod
    def _is_device_model(model):
        return getattr(model, "device_kind", None) is not None and not getattr(model, "flag_noise", False)

    # ------------------------------------------------------------------ persistence (ces/calibrate.py:170-237)
    def save(self, path='./', file='ces/', all=False, reset=True, online=False, counter=0):
        """Same files as the reference: ``ensemble.npy``, ``Gensemble.npy``, ``metrics.pkl``
        (+ ``*_path.npy`` with ``all``), or ``ensemble_NNNN.npy`` / ``Gensemble_NNNN.npy`` online."""
        try:
            os.makedirs(path + file)
        except OSError:
            pass
        if not hasattr(self, "Uall"):
            print('There is nothing to save')
            return
        if online:
            _save_iteration(path + file, counter, self.Uall[-1], self.Gall[-1])
        else:
            np.save(path + file + 'ensemble', self.Ustar)
            np.save(path + file + 'Gensemble', self.Gstar)
            if all:
                np.save(path + file + 'ensemble_path', self.Uall)
                np.save(path + file + 'Gensemble_path', self.Gall)
        self._save_metrics(path + file)

    def _save_metrics(self, where):
        with open(where + 'metrics.pkl', "wb") as fh:
            pickle.dump(self.metrics, fh)

    def load(self, path='./', eks_dir='ces/', ix_ensemble=False, flag_metrics=False):
        """Rebuild ``Uall, Gall, Ustar, Gstar, J, metrics`` from a directory written by ``save``."""
        where = path + eks_dir
        os.listdir(where)               # FileNotFoundError for a missing directory, like the reference (:203)
        try:
            with open(where + 'metrics.pkl', 'rb') as fh:
                self.metrics = pickle.load(fh)
        except FileNotFoundError:
            print('Metrics object not found. Could not load EKS object.')
            return False
        if not ix_ensemble:
            try:
                self.Uall = np.load(where + 'ensemble_path.npy')
                self.Gall = np.load(where + 'Gensemble_path.npy')
            except FileNotFoundError:
                print('EKS trajectory files not found.')
                return False
            return True
        if flag_metrics:
            count = len(self.metrics['self-bias'])
        else:
            count = sum(1 for name in os.listdir(where) if name.split('_')[0] == 'ensemble')
        try:
            Us = [np.load(where + 'ensemble_' + str(i).zfill(4) + '.npy') for i in range(count)]
            Gs = [np.load(where + 'Gensemble_' + str(i).zfill(4) + '.npy') for i in range(count)]
        except FileNotFoundError:
            return False
        self.Uall, self.Gall = np.asarray(Us), np.asarray(Gs)
        self.Ustar, self.Gstar = self.Uall[-1], self.Gall[-1]
        self.J = self.Uall.shape[-1]
        return True

    # ------------------------------------------------------------------ device plumbing
    def _get_engine(self, J, group=None):
        key = (self.p, self.n_obs, int(J), id(group))
        if self._engine is None or self._engine_key != key:
            if self._engine is not None:
                self._engine.close()
            self._engine = Engine(self.p, self.n_obs, int(J), group=group,
                                  d_panel_bytes=int(getattr(self, "d_panel_bytes", 0)))
            self._engine_key = key
            self._problem_key = None
        return self._engine

    def _sync_problem(self, eng, y_obs, Gamma, defer_large=False):
        """Make the device copies of y_obs / Gamma / sigma / mu / ustar (and the cached factorisations) current.

        The cache is keyed on the *content* of the five arrays (``_digest`` reads every byte), so an in-place edit is
        never missed.  Small arrays are digested on the spot.  With ``defer_large`` (the per-call path of
        ``eks_update*``), a large array whose buffer identity is unchanged is digested on a thread pool while the GPU
        step runs; the returned callable reports afterwards whether its content had changed after all, in which case
        the caller re-synchronises and repeats the step."""
        # AttributeError when mu / sigma / ustar are unset, like the reference (:433, :443)
        mu, sigma, ustar = self.mu, self.sigma, self.ustar
        arrays = (y_obs, Gamma, sigma, mu, ustar)
        idents = tuple(_identity(a) for a in arrays)
        prev = self._problem_key
        deferred = []
        digests = []
        for i, a in enumerate(arrays):
            large = np.asarray(a).nbytes > _SMALL_BYTES
            if defer_large and large and prev is not None and prev[0][i] == idents[i]:
                digests.append(prev[1][i])
                deferred.append(i)
            else:
                digests.append(_digest(a))
        digests = tuple(digests)
        if prev is None or prev[1] != digests:
            eng.set_problem(y_obs, Gamma, sigma, mu, ustar)
        self._problem_key = (idents, digests)
        if not deferred:
            return None
        global _pool
        if _pool is None:
            _digest(arrays[deferred[0]])          # creates the pool
        futures = [(i, _pool.submit(_digest, arrays[i])) for i in deferred]

        def stale():
            changed = False
            new = list(self._problem_key[1])
            for i, fut in futures:
                dg = fut.result()
                if dg != new[i]:
                    new[i], changed = dg, True
            if changed:
                eng.set_problem(y_obs, Gamma, sigma, mu, ustar)
                self._problem_key = (idents, tuple(new))
            return changed

        return stale


class sampling(enka):
    """Ensemble Kalman sampler (EKS / ALDI).  ces/calibrate.py:241-529."""

    # ------------------------------------------------------------------ step-size rule
    def timestep_method(self, D, Geval, y_obs, Gamma, Jnoise, **kwargs):
        """hk from an explicit interaction matrix D (ces/calibrate.py:243-267), with the same cumulative
        time bookkeeping in ``self.metrics['t']``.  The update methods below compute the same quantity on
        the device without materialising D on the host; this entry point serves callers that own a D."""
        kind = kwargs.get('time_step', None)
        const = kwargs.get('delta_t', 1. / (self.T / 2))
        if kind is None or (kind == 'mix' and (len(self.metrics['t']) == 0 or
                                               self.metrics['t'][-1] < kwargs.get('spinup', 4.))):
            hk = 1. / (self._frobenius(D) + 1e-8)
        elif kind in ('constant', 'mix'):
            hk = const
        elif kind == 'spectral':
            # ces/calibrate.py:249-251 on a caller-owned (non-symmetric) D: radspec = eigvals(D).real.max().  The update
            # methods never come here (they get lambda_max from the ensemble, csrc/eig.cu); this compatibility entry
            # point has only the J x J matrix, so it runs the general eigenvalue routine on the device (cuSOLVER geev
            # through torch.linalg.eigvals -- library code, off the hot path).
            self._ensure_metrics()
            radspec = self._eigvals_real_max(D)
            self.radspec.append(radspec)
            hk = 1. / radspec
        else:
            raise NotImplementedError("time_step=%r: 'adaptive' calls a method the reference does not define "
                                      "(ces/calibrate.py:255)" % (kind,))
        self._advance_time(hk)
        return hk

    @staticmethod
    def _frobenius(D):
        import ctypes
        import torch
        from . import _lib

        Dd = torch.from_numpy(np.ascontiguousarray(D, dtype=np.float64)).cuda()
        out = ctypes.c_double()
        _lib.check(_lib.load().ces_frobenius(ctypes.c_void_p(torch.cuda.current_stream().cuda_stream),
                                             ctypes.c_void_p(Dd.data_ptr()), int(Dd.stride(0)), int(Dd.shape[0]),
                                             int(Dd.shape[1]), ctypes.byref(out)))
        return out.value

    @staticmethod
    def _eigvals_real_max(D):
        import torch

        if not torch.cuda.is_available():
            raise RuntimeError("ces_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        Dd = torch.from_numpy(np.ascontiguousarray(D, dtype=np.float64)).cuda()
        return float(torch.linalg.eigvals(Dd).real.max().item())

    def _advance_time(self, hk):
        # ces/calibrate.py:262-265 (first step <=> no time recorded yet)
        t = self.metrics['t']
        t.append(hk if len(t) == 0 else hk + t[-1])

    def _ensure_metrics(self):
        if not hasattr(self, 'metrics'):
            self.radspec = []
            self.metrics = dict((key, []) for key in _METRIC_KEYS)

    def _option(self, kwargs, name):
        """An option of the call: the keyword argument, else the attribute of that name, else its default."""
        return kwargs.get(name, getattr(self, name, _OPTION_DEFAULTS[name]))

    def _step_options(self, rule, kwargs):
        """(fixed_h, resolve) for Engine.step from the reference's ``time_step`` kwargs
        (ces/calibrate.py:247-260 for hk; :439-441 / :470-473 for the hk C^pp + Gamma re-solve of D)."""
        kind = kwargs.get('time_step', None)
        if kind is None or rule == 'aldi_constant':          # aldi_constant sets its own hk (:519)
            return None, None
        const = kwargs.get('delta_t', 1. / (self.T / 2))
        if kind == 'constant':
            return const, ('always' if rule in ('eks', 'aldi') else None)
        if kind == 'mix':
            t = self.metrics['t'] if hasattr(self, 'metrics') else []
            spun_up = not (len(t) == 0 or t[-1] < kwargs.get('spinup', 4.))
            resolve = ((t[-1] if len(t) else 0.0), 1.0) if rule == 'aldi' else None     # eks never re-solves for 'mix'
            return (const if spun_up else None), resolve
        if kind == 'spectral':
            # hk = 1 / eigvals(D).real.max() (:249-251), no re-solve of D; aldi_constant never gets here (:519)
            return None, 'spectral'
        if kind == 'adaptive':
            raise NotImplementedError(
                "time_step='adaptive' calls a method the reference does not define (ces/calibrate.py:255)")
        raise ValueError("unknown time_step %r" % (kind,))

    def _noise_options(self, rule, kwargs, J, cols=None):
        """(ensemble?, explicit J x J xi or None) from the ``noise`` kwarg / attribute, checked before any device work.
        ``cols``: this rank's column count when the caller may pass only its own columns of xi (``local_shard``)."""
        mode = self._option(kwargs, 'noise')
        if mode not in ('cholesky', 'ensemble'):
            raise ValueError("noise must be 'cholesky' or 'ensemble', got %r" % (mode,))
        if mode == 'cholesky' or rule == 'eki':                  # eki has no noise term
            return False, None
        if self._option(kwargs, 'formulation') == 'factored':
            raise ValueError("noise='ensemble' needs formulation='interaction': the factored formulation never gathers "
                             "U - ubar")
        xi = kwargs.get('xi', None)
        if xi is None:
            return True, None
        xi = np.asarray(xi, dtype=np.float64)
        shapes = [(J, J)] + ([(J, cols)] if cols is not None else [])
        if xi.ndim != 2 or xi.shape not in shapes:
            raise ValueError("noise='ensemble' takes xi of shape %s, got %s" % (" or ".join(map(str, shapes)), xi.shape))
        return True, xi

    # ------------------------------------------------------------------ single updates on numpy arrays
    def _start_step(self, rule, kwargs, noise):
        """Begin a step of ``rule``: set ``update_rule`` to the reference's name of it and return the keywords of
        ``Engine.step`` / ``step_host``.  ``noise``: (ensemble?, J x J xi or None) from ``_noise_options``; the ensemble
        noise is keyed by the step count ``len(self.metrics['t'])``."""
        self.update_rule = _UPDATE_RULE[rule]
        fixed, resolve = self._step_options(rule, kwargs)     # 'mix' depends on the time reached so far
        ensemble, xi = noise
        return dict(fixed_h=fixed, switch=kwargs.get('switch', 1.), resolve=resolve,
                    formulation=self._option(kwargs, 'formulation'),
                    noise=('ensemble', int(self._option(kwargs, 'seed')), len(self.metrics['t']), xi) if ensemble else None)

    def _record(self, met, hk, resolve):
        """A step's metrics and cumulative time; with time_step='spectral' also lambda_max = 1 / hk (ces/calibrate.py:250)."""
        for key in ('self-bias', 'bias', 'self-bias-data', 'bias-data'):
            self.metrics[key].append(met[key])
        self._advance_time(hk)
        if resolve == 'spectral':
            self.radspec.append(1. / hk)

    def _update_host(self, rule, y_obs, U0, Geval, Gamma, kwargs):
        self._ensure_metrics()
        self._step_options(rule, kwargs)            # validates time_step before any work
        U0 = np.asarray(U0, dtype=np.float64)
        group = getattr(self, 'group', None)
        local = bool(kwargs.get('local_shard', False)) and group is not None
        Jg = self.J if local else U0.shape[1]
        cols = None
        if local:
            import torch.distributed as dist

            from .engine import shard_range

            lo, hi = shard_range(Jg, dist.get_rank(group), dist.get_world_size(group))
            cols = hi - lo
        ensemble, xi_ens = self._noise_options(rule, kwargs, Jg, cols)
        eng = self._get_engine(Jg, group)
        stale = self._sync_problem(eng, y_obs, Gamma, defer_large=True)
        Gk = np.asarray(Geval, dtype=np.float64)[:self.n_obs]
        xi = None
        if ensemble:
            # the J x J xi: this rank's columns of the caller's array, or the device's Philox stream keyed by the step
            if xi_ens is not None and xi_ens.shape[1] == eng.J and eng.cols != eng.J:
                xi_ens = xi_ens[:, eng.col_lo:eng.col_hi]
        elif rule != 'eki':
            # the full (p, J) draw on every rank -- the same global stream as the reference -- unless the caller
            # passes its own (possibly sharded) noise
            xi = self._draw_noise((U0.shape[0], eng.J), kwargs)
        if eng.nranks > 1 and not local:
            # every rank was called with the full arrays (the reference's calling convention): take this rank's columns;
            # the full U_next is gathered below
            lo, hi = eng.col_lo, eng.col_hi
            U0, Gk = U0[:, lo:hi], Gk[:, lo:hi]
            if xi is not None and xi.shape[1] == eng.J:
                xi = xi[:, lo:hi]
        elif local and xi is not None and xi.shape[1] == eng.J and eng.J != eng.cols:
            xi = xi[:, eng.col_lo:eng.col_hi]
        opts = self._start_step(rule, kwargs, (ensemble, xi_ens))
        Uk, hk, met = eng.step_host(rule, U0, Gk, xi, **opts)
        if stale is not None and stale():
            # a large problem array was edited in place since the previous call: the device copy has just been
            # refreshed; repeat the step with the current data (the noise already drawn is reused)
            Uk, hk, met = eng.step_host(rule, U0, Gk, xi, **opts)
        if eng.nranks > 1 and not local:
            Uk = eng.gather_columns(eng.torch.from_numpy(Uk).cuda(), Uk.shape[0]).cpu().numpy()
        self._record(met, hk, opts['resolve'])
        return Uk

    def _draw_noise(self, shape, kwargs):
        xi = kwargs.get('xi', None)
        if xi is not None:
            return np.asarray(xi, dtype=np.float64)
        return np.random.normal(0, 1, [shape[0], shape[1]])

    def eks_update(self, y_obs, U0, Geval, Gamma, iter, **kwargs):
        """Semi-implicit EKS step (ces/calibrate.py:418-449).

        ``noise='ensemble'`` (here and in the aldi updates) replaces the reference's ``sqrt(2h) chol(C^uu) xi`` by
        ``sqrt(2h / n_C) (U - ubar) xi`` with a J x J ``xi``: ``xi=`` an explicit (J, J) array ((J, cols) with
        ``local_shard=True``), or by default the device's Philox stream keyed by ``seed`` and the step count
        ``len(self.metrics['t'])``.  The update then draws nothing from numpy's global generator (``rng`` does not apply);
        a forward model's own draws, such as ``banana``'s, are unaffected."""
        return self._update_host('eks', y_obs, U0, Geval, Gamma, kwargs)

    def eks_update_aldi(self, y_obs, U0, Geval, Gamma, iter, **kwargs):
        """ALDI step, the default (ces/calibrate.py:451-490)."""
        return self._update_host('aldi', y_obs, U0, Geval, Gamma, kwargs)

    def eks_update_aldi_constant(self, y_obs, U0, Geval, Gamma, iter, **kwargs):
        """ALDI step with h = 0.1 / max|drift| (ces/calibrate.py:492-529)."""
        return self._update_host('aldi_constant', y_obs, U0, Geval, Gamma, kwargs)

    def eki_update(self, y_obs, U0, Geval, Gamma, iter, **kwargs):
        """Deterministic ensemble Kalman inversion step U - h (U - ubar) D: the part every EKS rule shares
        (first two terms of ces/calibrate.py:444 / :484).  The reference ships no EKI class (SURVEY.md F3)."""
        return self._update_host('eki', y_obs, U0, Geval, Gamma, kwargs)

    # ------------------------------------------------------------------ the run loop
    def _ensembles_dir(self, model, tag=''):
        """``directory/ensembles/<model_name><tag>-JJJJ[-NN]/`` (NN: ``nexp``): ``online_path`` without a tag, and the
        directory of the online save with the tag ``-eks-LLL`` (LLL: ``model.l_window``)."""
        return (self.directory + '/ensembles/' + model.model_name + tag + '-' + str(self.J).zfill(4)
                + ('-' + str(self.nexp).zfill(2) if hasattr(self, 'nexp') else '') + '/')

    def _online_dir(self, model):
        """The directory of ``run``'s online save, created: the files of ``enka.save(online=True)`` (ces/calibrate.py:371-385;
        the reference reads ``model.l_window`` there, which its own Darcy model lacks: defaulted to 0)."""
        where = self._ensembles_dir(model, '-eks-' + str(getattr(model, 'l_window', 0)).zfill(3))
        try:
            os.makedirs(where)
        except OSError:
            pass
        return where

    def _end_run(self, model, Us, Gs, U, G):
        """The results of ``run`` (ces/calibrate.py:404-416) from the final ensemble ``U`` and forward output ``G`` ('pde':
        the statistics stacked on the final states).  With a trace (``Us`` / ``Gs``: each iteration's ensemble and output
        before its update; None without), ``Uall`` / ``Gall`` continue those of an earlier run and end with U / G."""
        if Us is not None:
            self.Uall = np.asarray(list(getattr(self, 'Uall', [])) + list(Us) + [U])
            self.Gall = np.asarray(list(getattr(self, 'Gall', [])) + list(Gs) + [G])
        self.Ustar = U
        self.Gstar = G[:self.n_obs, :]
        self.online_path = self._ensembles_dir(model)

    def _carry_state(self, ws_pool, W_end, final):
        """The next initial states ``W0`` of a 'pde' model (ces/calibrate.py:317-327, 390-396): a draw from the ``ws`` pool,
        appended to ``Wall`` except after the final pass; without a pool, the final states ``W_end`` of the pass (a host
        array, or None while they are kept on the device only).  Returns True when the final states carry over."""
        if ws_pool is not None:
            widx = np.random.randint(ws_pool.shape[0], size=self.J)
            if not final:
                self.Wall.append(widx)
            self.W0 = ws_pool[widx].T
            return False
        if W_end is not None:
            self.W0 = np.copy(W_end)
        return True

    def _fused_small_run(self, eng, U0, model, rule, kwargs, first, noise, save_online, trace):
        """The whole loop in ONE kernel launch (``ces_small_run``) when the problem fits a single CTA (p <= 8, k <= 16,
        J <= 512 -- BASELINE config 1) and the forward model is one of the ``ces_b200.utils`` maps: forward, update,
        cumulative time and the ``t_tol`` stopping rule run back to back on the device, the trace is the chain of
        ensembles the kernel leaves in HBM, and the host downloads everything once.  Same results as the iteration-by-
        iteration loop below (same arithmetic per step; the noise is the numpy stream the reference would consume: all T
        draws are taken in one call and the generator is rewound to where an early stop leaves it).  ``noise='ensemble'``
        runs here too up to J = _FUSED_ENSEMBLE_J_MAX: the kernel draws the device stream keyed by ``seed`` at step
        ``len(self.metrics['t']) + i``, or reads the one (J, J) ``xi``, as the general loop does.  ``first``: the
        ``_step_options`` of the first step, ``noise``: the ``_noise_options``.  Returns False when the configuration
        needs the general loop."""
        import ctypes

        from . import _lib

        kind = getattr(model, 'device_kind', None)
        ensemble = noise[0]
        if not (eng.nranks == 1 and kind in _lib.MAPS and self.p <= 8 and self.n_obs <= 16
                and 2 <= eng.J <= (_FUSED_ENSEMBLE_J_MAX if ensemble else 512) and self.T >= 1
                and first == (None, None) and self._option(kwargs, 'formulation') == 'interaction'
                and getattr(self, 'fused_run', True) and (ensemble or kwargs.get('xi', None) is None)):
            return False
        p, k, J, T = self.p, self.n_obs, eng.J, int(self.T)
        if (T + 1) * ((p if ensemble else 2 * p) + k) * J * 8 > (1 << 28):     # traces (+ the T x p x J Cholesky xi)
            return False
        torch = eng.torch
        A_dev, lda, b_dev, params = model._device_args(torch)
        par = np.ascontiguousarray(params, dtype=np.float64) if params is not None else None
        device_rng = self._option(kwargs, 'rng') == 'device'
        xi_all, state = None, None
        fdraws = int(getattr(model, 'rng_draws_per_call', 0)) * J    # normals the reference's forward loop draws per pass
        host_noise = rule != 'eki' and not device_rng and not ensemble
        if host_noise or fdraws:
            # per iteration the reference draws [forward pass: fdraws][update: p * J] (:351-352 then :447,488,527), and
            # fdraws once more for the final forward pass; all T iterations are drawn in one call (the same stream)
            state = np.random.get_state()
            per = fdraws + (p * J if host_noise else 0)
            raw = np.random.normal(0, 1, [T, per])
            if host_noise:
                xi_all = np.ascontiguousarray(raw[:, fdraws:]).reshape(T, p, J)
        t_hist = self.metrics['t']
        Ut = np.empty((T + 1, p, J))
        Gt = np.empty((T + 1, k, J))
        S = np.empty((T, 16))
        tv = np.empty(T)
        n = ctypes.c_int64()
        opts = self._start_step(rule, kwargs, noise)
        with eng.on_stream():
            eng._apply_noise(opts['noise'])
            _lib.check(eng.lib.ces_small_run(
                eng.h, _lib.RULES[rule], _lib.TS_FROBENIUS, 0.0, float(opts['switch']), _lib.MAPS[kind],
                ctypes.c_void_p(A_dev.data_ptr()) if A_dev is not None else None, int(lda),
                ctypes.c_void_p(b_dev.data_ptr()) if b_dev is not None else None,
                _lib.host_ptr(par) if par is not None else None, _lib.host_ptr(U0),
                _lib.host_ptr(xi_all) if xi_all is not None else None, int(self._option(kwargs, 'seed')),
                len(t_hist), T, float(t_hist[-1]) if len(t_hist) else 0.0, 1 if len(t_hist) else 0,
                float(kwargs.get('t_tol', 2.)), _lib.host_ptr(Ut), _lib.host_ptr(Gt), _lib.host_ptr(S), _lib.host_ptr(tv),
                ctypes.byref(n)))
        n = int(n.value)
        if state is not None:
            if n < T:
                np.random.set_state(state)                       # an early stop consumed only n iterations' draws
                np.random.normal(0, 1, [n, fdraws + (p * J if host_noise else 0)])
            if fdraws:
                np.random.normal(0, 1, fdraws)                   # the final forward pass
        # step scalars -> metrics (sums over particles / J), cumulative times
        for name, col in (('self-bias', 1), ('bias', 2), ('self-bias-data', 3), ('bias-data', 4)):
            self.metrics[name].extend((S[:n, col] / J).tolist())
        self.metrics['t'].extend(tv[:n].tolist())
        if save_online:
            where = self._online_dir(model)
            for it in range(n):
                _save_iteration(where, it, Ut[it], Gt[it])
            self._save_metrics(where)
        self._end_run(model, Ut[:n] if trace else None, Gt[:n] if trace else None, Ut[n].copy(), Gt[n].copy())
        return True

    def run(self, y_obs, U0, model, Gamma, Jnoise, save_online=False, trace=True, **kwargs):
        """Ensemble Kalman sampler loop (ces/calibrate.py:270-416): forward -> trace -> update -> (save) ->
        stop when the cumulative pseudo-time exceeds ``t_tol`` (default 2.0) or after ``self.T`` iterations.
        ``Jnoise`` is accepted and ignored like in the reference (it recomputes cholesky(Gamma), :437).
        ``noise='ensemble'``: the ensemble form of the noise (see ``eks_update``), drawn on the device from ``seed`` at
        step ``len(self.metrics['t'])`` -- a resumed run continues the stream -- or ``xi=`` one (J, J) array used at every
        iteration; numpy's global generator is then advanced only by the forward model's own draws."""
        import torch

        mtype = model.type          # AttributeError if absent, like :294-297
        if not hasattr(self, 'directory'):
            self.directory = os.getcwd()
        rule = kwargs.get('update', 'aldi')
        self._update_name = rule
        if mtype not in ('map', 'pde'):
            raise ValueError("model.type must be 'map' or 'pde'")
        is_pde = (mtype == 'pde')
        self._ensure_metrics()
        first = self._step_options(rule, kwargs)            # validates time_step before any work
        group = getattr(self, 'group', None)

        U0 = np.ascontiguousarray(U0, dtype=np.float64)
        J = U0.shape[1]
        ensemble, xi_ens = self._noise_options(rule, kwargs, J)     # validates noise / xi before any work
        eng = self._get_engine(J, group)
        self._sync_problem(eng, y_obs, Gamma)
        lo, hi = eng.col_lo, eng.col_hi
        dev = torch.device("cuda", torch.cuda.current_device())
        known = rule in _UPDATE_RULE
        device_model = (not is_pde) and self._is_device_model(model)
        if known and device_model and self._fused_small_run(eng, U0, model, rule, kwargs, first, (ensemble, xi_ens),
                                                            save_online, trace):
            return

        U_dev = torch.from_numpy(U0[:, lo:hi].copy()).to(dev)
        if xi_ens is not None:
            xi_ens = torch.from_numpy(np.ascontiguousarray(xi_ens[:, lo:hi])).to(dev)     # the same xi every iteration
        G_dev = torch.empty(self.n_obs, hi - lo, dtype=torch.float64, device=dev)
        if is_pde:
            # initial conditions of the integrator, one per particle (ces/calibrate.py:317-327)
            t_ode, ws_pool, update_wt = kwargs.get('t', None), kwargs.get('ws', None), kwargs.get('update_wt', True)
            if ws_pool is not None:
                self.Wall = []
                self._carry_state(ws_pool, None, final=False)
            else:
                self.W0 = np.tile(kwargs.get('wt', None), self.J).reshape(self.J, model.n_state).T
        device_pde = is_pde and getattr(model, 'device_kind', None) is not None and hasattr(model, 'evaluate_ensemble_pde')
        W_dev = []                      # device 'pde' models: this rank's [W0, final states] in HBM

        def gather_host(local, rows):
            """Full (rows, J) host array from the column shards (synchronous)."""
            return eng.gather_columns(local, rows).cpu().numpy()

        def forward(U_dev, final=False):
            """G(U_dev) into G_dev (ces/calibrate.py:342-352, 390-396).  Returns the full host array of the outputs when
            the pass has one, else None: a host map's on a single GPU; a 'pde' model's statistics stacked on the final
            states, which the device integrators assemble on the host only for the trace or the final pass."""
            if not is_pde:
                if device_model:
                    model.evaluate_ensemble(eng, U_dev, G_dev)
                    _consume_model_rng(model, J)                # (every rank: the stream is global)
                    return None
                G_host = self._host_G_ens(U_dev.cpu().numpy(), model)
                G_dev.copy_(torch.from_numpy(np.ascontiguousarray(G_host[:self.n_obs])))
                return G_host if eng.nranks == 1 else None      # several ranks: this rank's columns only
            if device_pde:
                # the ces_b200.utils Lorenz models: the ensemble integrated on the device
                if not W_dev or ws_pool is not None:
                    W0 = torch.from_numpy(np.ascontiguousarray(self.W0[:, lo:hi])).to(dev)
                    W_dev[:] = [W0, torch.empty_like(W0)]
                model.evaluate_ensemble_pde(eng, U_dev, W_dev[0], t_ode, G_dev, W_dev[1])
                G_full = None
                if trace or final:
                    G_full = np.vstack([gather_host(G_dev, self.n_obs), gather_host(W_dev[1], model.n_state)])
            else:
                # the user's integrator on the host for this rank's particles; every rank needs the full array (next W0)
                G_full = self.G_pde_ens(np.vstack([U_dev.cpu().numpy(), self.W0[:, lo:hi]]), model, t_ode)
                if eng.nranks > 1:
                    G_full = gather_host(torch.from_numpy(np.ascontiguousarray(G_full)).to(dev), G_full.shape[0])
                G_dev.copy_(torch.from_numpy(np.ascontiguousarray(G_full[:self.n_obs, lo:hi])))
            if update_wt:
                carried = self._carry_state(ws_pool, None if G_full is None else G_full[self.n_obs:], final)
                if carried and device_pde:
                    W_dev.reverse()                     # the final states become the next W0 without leaving HBM
            return G_full

        # trace / save_online: asynchronous device->host copies into page-locked memory (no stall of the loop); the
        # arrays of iteration i are materialised when iteration i + 1 has been queued (online save) or after the loop
        host_trace = _HostTrace(torch) if (trace or save_online) else None
        tickets = []                    # per iteration: (U ticket, G ticket)
        online = save_online and eng.rank == 0
        device_rng = self._option(kwargs, 'rng') == 'device'
        for i in range(self.T):
            G_host = forward(U_dev)
            if host_trace is not None:
                tu = host_trace.push(eng.gather_columns(U_dev, self.p))        # every update returns a new tensor
                G_i = G_host if G_host is not None else eng.gather_columns(G_dev, self.n_obs)
                tickets.append((tu, host_trace.push(G_i, reused=G_i is G_dev)))
            if known:
                opts = self._start_step(rule, kwargs, (ensemble, xi_ens))
                xi_dev = None
                if not ensemble and rule != 'eki':
                    if device_rng:
                        # production mode: Philox noise generated on the device, nothing crosses PCIe
                        xi_dev = eng.normal_noise(self.p, self._option(kwargs, 'seed'), len(self.metrics['t']))
                    else:
                        xi = self._draw_noise((self.p, J), kwargs)      # same stream on every rank
                        xi_dev = torch.from_numpy(np.ascontiguousarray(xi[:, lo:hi])).to(dev)
                U_dev, hk, met = eng.step(rule, U_dev, G_dev, xi_dev, **opts)
                self._record(met, hk, opts['resolve'])
            # an unknown ``update`` leaves the ensemble unchanged and records nothing, like :364-369 --
            # the reference then fails on the empty ``metrics['t']``; so do we
            if online:
                # iteration i - 1's files are written now, while iteration i's copies are still in flight; metrics.pkl
                # follows the latest completed update like the reference's
                where = self._online_dir(model)
                if i:
                    _save_iteration(where, i - 1, *map(host_trace.get, tickets[i - 1]))
                self._save_metrics(where)
            if self.metrics['t'][-1] > kwargs.get('t_tol', 2.):
                break
        if online:
            where = self._online_dir(model)
            if tickets:
                _save_iteration(where, len(tickets) - 1, *map(host_trace.get, tickets[-1]))
        Us = [host_trace.get(tu) for tu, _ in tickets] if trace else None
        Gs = [host_trace.get(tg) for _, tg in tickets] if trace else None

        G_host = forward(U_dev, final=True)
        self._end_run(model, Us, Gs, gather_host(U_dev, self.p),
                      G_host if G_host is not None else gather_host(G_dev, self.n_obs))
