"""The device's Philox4x32-10 streams against oracle/philox_oracle.py, value for value: ces_fill_normal (the EKS noise of
sampling.run(rng='device'), fused and general paths, resumed runs), and every chain c >= 1 of the three
Metropolis-Hastings samplers -- map models (ces_mcmc_model_mh), emulator (ces_gp_mh) and Darcy (ces_darcy_mh) -- against
the oracle chain started where MCMC._chains starts it and driven by the restated chain noise.  Also chain 0 of each
sampler when the caller passes no MT19937 state: it is then the Philox chain c = 0.

Tolerances: the noise passes through CUDA's log / sincospi against numpy's log / cos / sin (1e-13 absolute; any indexing
error moves a value by O(1)); the chains use chain 0's tolerances (1e-9 of the sample scale for the map and Darcy
samplers, 1e-10 for the emulator) and equal acceptance counts."""
import ctypes
import os

import numpy as np
import pytest
import torch
from scipy.stats import multivariate_normal

pytestmark = pytest.mark.gpu

from ces_b200 import _lib, calibrate, sample as csample, utils as cutils  # noqa: E402
from ces_b200.emulate import GPEmulator  # noqa: E402
from oracle import eks_oracle as eo, forward_oracle as fo, gp_matern_oracle as gmo, gp_oracle as go  # noqa: E402
from oracle import mcmc_oracle as mo, philox_oracle as po  # noqa: E402
from test_gpu_darcy_mh import device_model as darcy_device_model, problem as darcy_problem  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
NOISE_TOL = 1e-13


# ---------------------------------------------------------------------------------------------- ces_fill_normal
@pytest.mark.parametrize("seed", [0, 7, 2 ** 40 + 3])
@pytest.mark.parametrize("step", [0, 5, 2 ** 31])
def test_fill_normal_is_the_restated_stream(seed, step):
    lib = _lib.load()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for rows in (1, 7, 64):
        for cols in (1, 2, 255, 256, 257, 1001):
            for off in (0, 1, 4999, 2 ** 32 - 1, 2 ** 33 + 1):
                buf = torch.full((rows, cols + 7), float("nan"), dtype=torch.float64, device="cuda")
                _lib.check(lib.ces_fill_normal(st, seed, step, ctypes.c_void_p(buf.data_ptr()), buf.stride(0), rows, cols,
                                               off))
                got = buf.cpu().numpy()
                want = po.fill_normal(seed, step, rows, cols, off)
                assert np.abs(got[:, :cols] - want).max() <= NOISE_TOL, (rows, cols, off)
                assert np.all(np.isnan(got[:, cols:])), (rows, cols, off)


# ---------------------------------------------------------------------------------------------- sampling.run
def _eks_problem(p, k, J):
    rs = np.random.RandomState(100 * p + k)
    A = rs.normal(size=(k, p)) / np.sqrt(p)
    A[:, 0] = 1.0
    ustar = rs.normal(size=(p, 1))
    Gamma = 0.1 * np.eye(k)
    y = A @ ustar[:, 0] + np.sqrt(0.1) * rs.normal(size=k)
    U0 = 3.0 * rs.normal(size=(p, J))
    return A, ustar, Gamma, y, U0


def _oracle_run(rule, s, A, y, Gamma, U, seed, step0, t, T, t_tol):
    """The oracle loop with the device noise: xi_t = fill_normal(seed, t, p, J, 0) for the run's global step t."""
    p, J = U.shape
    n = 0
    for _ in range(T):
        xi = po.fill_normal(seed, step0 + n, p, J, 0)
        o = eo.step(rule, y, U, fo.lineal(A, U), Gamma, s.mu, s.sigma, s.ustar, xi, t_last=t)
        U, t, n = o["Uk"], o["t"], n + 1
        if t > t_tol:
            break
    return U, t, n


def _rel(a, b):
    return np.abs(a - b).max() / np.abs(b).max()


def _device_runs(rule, p, k, J, fused, seed, T1, t_tol1, T2):
    """sampling.run(rng='device') twice on one object: T1 steps (or until t_tol1; None: until step 9), then T2 more; each
    call against the oracle loop, the second one continuing the step count (the noise's key) and the time of the first."""
    A, ustar, Gamma, y, U0 = _eks_problem(p, k, J)
    s = calibrate.sampling(p, k, J)
    s.ustar, s.mu, s.sigma, s.T, s.fused_run = ustar, np.zeros((p, 1)), 100.0 * np.eye(p), T1, fused
    if t_tol1 is None:
        # stop early, in step 9: t_tol halfway between the oracle's times after 8 and 9 steps
        t8 = _oracle_run(rule, s, A, y, Gamma, U0, seed, 0, None, 8, np.inf)[1]
        t9 = _oracle_run(rule, s, A, y, Gamma, U0, seed, 0, None, 9, np.inf)[1]
        t_tol1 = 0.5 * (t8 + t9)
    state = np.random.get_state()
    s.run(y, U0, cutils.lineal(A), Gamma, None, update=rule, t_tol=t_tol1, rng="device", seed=seed)
    U, t, n = _oracle_run(rule, s, A, y, Gamma, U0, seed, 0, None, T1, t_tol1)
    assert len(s.metrics["t"]) == n and abs(s.metrics["t"][-1] - t) < 1e-9 * t
    assert _rel(s.Ustar, U) < 1e-8, (rule, fused, _rel(s.Ustar, U))
    first = s.Uall.copy()
    s.T = T2
    s.run(y, s.Ustar, cutils.lineal(A), Gamma, None, update=rule, t_tol=1e9, rng="device", seed=seed)
    U2, t2, n2 = _oracle_run(rule, s, A, y, Gamma, s.Uall[n + 1], seed, n, t, T2, 1e9)
    assert n2 == T2 and len(s.metrics["t"]) == n + T2 and abs(s.metrics["t"][-1] - t2) < 1e-9 * t2
    assert _rel(s.Ustar, U2) < 1e-8, (rule, fused, _rel(s.Ustar, U2))
    # numpy's generator is not touched by the device noise
    after = np.random.get_state()
    assert np.array_equal(after[1], state[1]) and after[2] == state[2]
    return first, s.Uall, n


@pytest.mark.parametrize("rule", ["aldi", "eks", "aldi_constant"])
def test_device_noise_run_matches_the_oracle_on_both_paths(rule):
    """p = 2, k = 10, J = 100: the one-launch fused run and the general loop, each against the oracle and against each
    other; the first call stops early on t_tol, the second continues from its step count."""
    seed = 2 ** 33 + 9
    fused = _device_runs(rule, 2, 10, 100, True, seed, 25, None, 6)
    general = _device_runs(rule, 2, 10, 100, False, seed, 25, None, 6)
    n = fused[2]
    assert general[2] == n == 9, n
    assert fused[1].shape == general[1].shape == (n + 1 + 7, 2, 100)
    gap = _rel(fused[1], general[1])
    print("fused vs general trajectory", gap)
    assert gap <= 1e-12, gap


@pytest.mark.parametrize("rule", ["aldi", "eks", "aldi_constant"])
def test_device_noise_run_matches_the_oracle_above_the_small_limits(rule):
    """p = 20, k = 33, J = 1001: the general loop, several blocks of fill_normal and an odd J."""
    first, full, n = _device_runs(rule, 20, 33, 1001, False, 7, 4, 1e9, 3)
    assert n == 4 and full.shape == (4 + 1 + 4, 20, 1001)


# ---------------------------------------------------------------------------------------------- the chains
def _chain_starts(Ustar, C):
    """MCMC._chains: chain c >= 1 starts at ensemble member c mod J, which is also the point of its initial Phi."""
    return [np.asarray(Ustar, dtype=float)[:, c % Ustar.shape[1]] for c in range(C)]


def _assert_chain(got, got_acc, want, want_acc, n, tol, what):
    assert got.shape == want.shape, what
    err = np.abs(got - want).max() / np.abs(want).max()
    assert err <= tol, (what, err)
    assert round(got_acc * n) == round(want_acc * n), (what, got_acc * n, want_acc * n)


G_MCMC = np.load(os.path.join(HERE, "golden", "mcmc_cases.npz"))


def _map_case(name):
    """(forward oracle, device model, prior, Ustar, y, Gamma, kw) of a seeded lineal / lineal_log problem 'p,k,kind,update'
    or of a golden elliptic / banana case."""
    if name in ("elliptic_rw", "banana_rw"):
        g = lambda key: G_MCMC["%s/%s" % (name, key)]
        kind = str(g("kind"))
        fwd = (lambda th: getattr(fo, kind)(np.asarray(th).reshape(2, 1))[:, 0])
        prior = multivariate_normal(g("prior_mean"), g("prior_cov"))
        kw = dict(delta=float(g("delta")), enka_scaling=bool(g("scaling")))
        return fwd, getattr(cutils, kind)(), prior, g("Ustar"), g("y"), g("Gamma"), kw
    p, k, kind, update = name.split(",")
    p, k = int(p), int(k)
    rs = np.random.RandomState(100 * p + k)
    A = rs.normal(size=(k, p)) / np.sqrt(p) * (0.3 if kind == "lineal_log" else 1.0)
    truth = 0.3 * rs.normal(size=p)
    fwd = (lambda th: getattr(fo, kind)(A, np.asarray(th).reshape(-1, 1))[:, 0])
    y = fwd(truth) + 0.05 * rs.normal(size=k)
    Q = rs.normal(size=(k, k))
    Gamma = 0.01 * (np.eye(k) + 0.3 * Q @ Q.T / k)
    S = rs.normal(size=(p, p))
    prior = multivariate_normal(0.1 * rs.normal(size=p) if update == "rw" else np.zeros(p), np.eye(p) + 0.2 * S @ S.T / p)
    J = 3 * p + 8
    Ustar = truth[:, None] + 0.05 * rs.normal(size=(p, J))
    kw = {"delta": 0.6, "enka_scaling": True}
    if update == "pCN":
        kw.update(update="pCN", beta=0.002)
    return fwd, getattr(cutils, kind)(A), prior, Ustar, y, Gamma, kw


MAP_CASES = [("1,1,lineal,rw", 5), ("3,40,lineal,rw", 2 ** 40 + 3), ("17,33,lineal_log,pCN", 11), ("32,64,lineal,rw", 4),
             ("elliptic_rw", 6), ("banana_rw", 2 ** 32)]


@pytest.mark.parametrize("name,seed", MAP_CASES)
def test_model_mh_philox_chains_are_the_oracle_chains(name, seed):
    """C = 9 chains (one warp each, four per CTA: chains 4 and 8 open new CTAs); every chain c >= 1 against the oracle
    chain with chain_noise(seed, 'MH', it, c); the banana's Philox chains draw nothing for the model."""
    fwd, model, prior, Ustar, y, Gamma, kw = _map_case(name)
    p, J = Ustar.shape
    C, n = 9, 150
    enka = calibrate.sampling(p, len(y), J)
    enka.Ustar = Ustar
    mc = csample.MCMC()
    mc.y_obs = y
    np.random.seed(77)
    mc.model_mh(model, n, prior, enka, Gamma, n_chains=C, seed=seed, **kw)
    assert mc.samples_chains.shape == (C, p, n + 1)
    starts = _chain_starts(Ustar, C)
    rates = []
    for c in range(1, C):
        want, acc = mo.model_mh(fwd, n, prior, Ustar, y, Gamma, start=starts[c],
                                noise=lambda it, c=c: po.chain_noise(seed, po.TAG_MH, it, c, p), **kw)
        _assert_chain(mc.samples_chains[c], mc.accept_chains[c], want, acc, n, 1e-9, (name, c))
        rates.append(acc)
    assert 0.0 < np.mean(rates) < 1.0, rates
    # Recorded behaviour: the extra chains are keyed by `seed` alone and restart from the ensemble members at step 0, so a
    # different numpy seed gives the same chains 1..C-1, and a resumed call replays the first call's extra chains.
    first = mc.samples_chains.copy()
    again = csample.MCMC()
    again.y_obs = y
    np.random.seed(78)
    again.model_mh(model, n, prior, enka, Gamma, n_chains=C, seed=seed, **kw)
    assert np.array_equal(again.samples_chains[1:], first[1:])
    mc.model_mh(model, 50, prior, enka, Gamma, n_chains=C, seed=seed, **kw)
    assert mc.samples.shape == (p, n + 51)
    assert np.array_equal(mc.samples_chains[1:], first[1:, :, :51])


GP = np.load(os.path.join(HERE, "golden", "gp_cases.npz"))
GM = np.load(os.path.join(HERE, "golden", "gp_matern_cases.npz"))


def _emulator_case(name, fam):
    """(emulator, enka, prior, ytil): the golden chain set-up of the p = 2 emulators, or a seeded one at p = 32."""
    src = GP if fam == "SquaredExponential" else GM
    X, G = src[name + "/X"], src[name + "/G"]
    emu = GPEmulator(U=X, G=G, Gamma=np.eye(G.shape[0]), jitter=float(src["jitter"]), kernel=fam)
    emu.theta = src[(name if fam == "SquaredExponential" else "%s/%s" % (fam, name)) + "/theta"]
    if name == "p2_n100_k10":
        Ustar, ytil = src["chain/Ustar"], src["chain/ytil"]
        prior = multivariate_normal(src["chain/prior_mean"], src["chain/prior_cov"])
    else:
        rs = np.random.RandomState(32)
        Ustar = src[name + "/U"]
        u0 = Ustar.mean(axis=1)
        mean, _ = go.predict(emu.X, emu.Y, emu.offset, emu.theta, u0[:, None], emu.jitter)
        ytil = mean[:, 0] + 0.05 * rs.normal(size=emu.k)
        prior = multivariate_normal(u0, np.cov(Ustar) + 0.1 * np.eye(emu.p))
    enka = calibrate.sampling(emu.p, emu.k, Ustar.shape[1])
    enka.Ustar = Ustar
    return emu, enka, prior, ytil


def _predict_one(emu, fam):
    if fam == "SquaredExponential":
        return lambda u: tuple(a[:, 0] for a in go.predict(emu.X, emu.Y, emu.offset, emu.theta, u[:, None], emu.jitter))
    return lambda u: tuple(a[:, 0] for a in gmo.predict(emu.X, emu.Y, emu.offset, emu.theta, u[:, None], fam, emu.jitter))


EMU_CASES = [("p2_n100_k10", "SquaredExponential", dict(delta=0.8), True),
             ("p2_n100_k10", "SquaredExponential", dict(delta=0.8), False),
             ("p2_n100_k10", "SquaredExponential", dict(update="pCN", beta=0.05), True),
             ("p2_n100_k10", "Matern52", dict(delta=0.8), True),
             ("p2_n100_k10", "Matern52", dict(update="pCN", beta=0.05), True),
             ("p32_n200_k3", "SquaredExponential", dict(delta=0.3), True)]


@pytest.mark.parametrize("name,fam,kw,use_var", EMU_CASES)
def test_emulator_mh_philox_chains_are_the_oracle_chains(name, fam, kw, use_var):
    """C = 130 chains: the propose and accept kernels run 128 chains per CTA, so chains 127 | 128 sit on either side of a
    CTA edge; chains {1, 2, 63, 127, 128, 129} against the oracle chain with chain_noise(seed, 'GP', it, c)."""
    emu, enka, prior, ytil = _emulator_case(name, fam)
    C, n, seed = 130, 60, 2 ** 35 + 1
    mc = csample.MCMC()
    mc.y_obs = ytil
    np.random.seed(13)
    mc.emulator_mh(emu, n, prior, enka, n_chains=C, seed=seed, use_variance=use_var, **kw)
    assert mc.samples_chains.shape == (C, emu.p, n + 1)
    starts = _chain_starts(enka.Ustar, C)
    predict_one = _predict_one(emu, fam)
    rates = []
    for c in (1, 2, 63, 127, 128, 129):
        want, acc = go.emulator_mh(predict_one, n, prior, enka.Ustar, ytil, use_variance=use_var, start=starts[c],
                                   noise=lambda it, c=c: po.chain_noise(seed, po.TAG_GP, it, c, emu.p), **kw)
        _assert_chain(mc.samples_chains[c], mc.accept_chains[c], want, acc, n, 1e-10, (name, fam, c))
        rates.append(acc)
    assert 0.0 < np.mean(rates) < 1.0, rates


@pytest.mark.parametrize("name,C,n,chains", [("trunc16_rw", 130, 40, (1, 2, 127, 128, 129)), ("full8_pcn", 3, 120, (1, 2))])
def test_darcy_mh_philox_chains_are_the_oracle_chains(name, C, n, chains):
    """The lockstep Darcy chains (128 per CTA in the noise and accept kernels) against the oracle chain through the scipy
    Darcy restatement with chain_noise(seed, 'DR', it, c); full8_pcn has p = 64 (32 Box-Muller pairs) and a dense Gamma."""
    ref, obs, y, Gamma, Ustar, prior, kw, _ = darcy_problem(name)
    p = ref.p
    seed = 2 ** 36 + 5
    enka = calibrate.sampling(p, len(obs), Ustar.shape[1])
    enka.Ustar = Ustar
    mc = csample.MCMC()
    mc.y_obs = y
    np.random.seed(21)
    mc.model_mh(darcy_device_model(name, obs), n, prior, enka, Gamma, n_chains=C, seed=seed, **kw)
    starts = _chain_starts(Ustar, C)
    rates = []
    for c in chains:
        want, acc = mo.model_mh(ref, n, prior, Ustar, y, Gamma, start=starts[c],
                                noise=lambda it, c=c: po.chain_noise(seed, po.TAG_DARCY, it, c, p), **kw)
        _assert_chain(mc.samples_chains[c], mc.accept_chains[c], want, acc, n, 1e-9, (name, c))
        rates.append(acc)
    assert 0.0 < np.mean(rates) < 1.0, rates


# ---------------------------------------------------------------------------------------------- no MT19937 state
def _without_mt(c):
    """The C arguments of MCMC._chains with mt_state_host = mt_gauss_host = NULL."""
    return c.args[:9] + (None, None) + c.args[11:]


def test_chain_zero_without_numpy_state_is_the_philox_chain():
    """Each C entry point, called with no MT19937 state, draws chain 0 from Philox as chain c = 0 (started at the ensemble
    mean, like the stream chain)."""
    lib = _lib.load()
    seed, C = 2 ** 34 + 17, 2
    # map sampler
    fwd, model, prior, Ustar, y, Gamma, kw = _map_case("3,40,lineal,rw")
    p, k, n = 3, 40, 100
    enka = calibrate.sampling(p, k, Ustar.shape[1])
    enka.Ustar = Ustar
    mc = csample.MCMC()
    c = mc._chains(p, n, prior, enka, kw["delta"], kw["enka_scaling"], False, 0.5, C, seed)
    A_dev, lda, b_dev, params = model._device_args(torch)
    assert b_dev is None and params is None
    Ginv2 = np.ascontiguousarray(np.linalg.inv(2.0 * Gamma))
    yc = np.ascontiguousarray(y)
    _lib.check(lib.ces_mcmc_model_mh(ctypes.c_void_p(torch.cuda.current_stream().cuda_stream), _lib.MAPS["lineal"], p, k,
                                     ctypes.c_void_p(A_dev.data_ptr()), int(lda), None, None, _lib.host_ptr(yc),
                                     _lib.host_ptr(Ginv2), *_without_mt(c)))
    want, acc = mo.model_mh(fwd, n, prior, Ustar, y, Gamma, noise=lambda it: po.chain_noise(seed, po.TAG_MH, it, 0, p), **kw)
    _assert_chain(c.samples[0].T, c.accepted[0] / n, want, acc, n, 1e-9, "model_mh")
    # emulator sampler
    emu, enka, prior, ytil = _emulator_case("p2_n100_k10", "SquaredExponential")
    n = 60
    c = mc._chains(emu.p, n, prior, enka, 0.8, True, False, 0.5, C, seed)
    emu.condition()
    yt = np.ascontiguousarray(ytil)
    _lib.check(lib.ces_gp_mh(emu._h, _lib.host_ptr(yt), 1, *_without_mt(c)))
    want, acc = go.emulator_mh(_predict_one(emu, "SquaredExponential"), n, prior, enka.Ustar, ytil, delta=0.8,
                               noise=lambda it: po.chain_noise(seed, po.TAG_GP, it, 0, emu.p))
    _assert_chain(c.samples[0].T, c.accepted[0] / n, want, acc, n, 1e-10, "emulator_mh")
    # Darcy sampler
    ref, obs, y, Gamma, Ustar, prior, kw, _ = darcy_problem("trunc16_rw")
    n = 40
    enka = calibrate.sampling(ref.p, len(obs), Ustar.shape[1])
    enka.Ustar = Ustar
    m = darcy_device_model("trunc16_rw", obs)
    c = mc._chains(ref.p, n, prior, enka, kw["delta"], kw["enka_scaling"], False, 0.5, C, seed)
    Ginv2 = np.ascontiguousarray(np.linalg.inv(2.0 * Gamma))
    yc = np.ascontiguousarray(y)
    _lib.check(lib.ces_darcy_mh(m._handle(True), float(m.tol), int(m.max_iter), _lib.host_ptr(yc), _lib.host_ptr(Ginv2),
                                *_without_mt(c)))
    want, acc = mo.model_mh(ref, n, prior, Ustar, y, Gamma,
                            noise=lambda it: po.chain_noise(seed, po.TAG_DARCY, it, 0, ref.p), **kw)
    _assert_chain(c.samples[0].T, c.accepted[0] / n, want, acc, n, 1e-9, "darcy_mh")
