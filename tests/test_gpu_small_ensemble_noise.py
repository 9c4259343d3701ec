"""noise='ensemble' on the single-CTA path (DESIGN.md sections 4c, 4g): small problems (p <= 8, k <= 16) take the one-kernel
step (J <= 128) and the one-launch sampling.run (J <= 256) with the ensemble noise sqrt(2h / n_C) (U - ubar) xi, xi J x J.

* one step (Engine.step on device tensors, eks_update* on numpy arrays) against oracle/ensemble_noise_oracle.step and against
  the phase path (CES_NO_SMALL_PATH=1), with an explicit xi and with the device stream, in one launch like a Cholesky step
  up to the J limit, on the phases above it;
* the stream drawn inside the kernel equals, bit for bit, the same step fed ces_fill_ensemble_noise as its explicit xi;
* sampling.run in one launch against the per-iteration loop and the oracle loop: t_tol stops, resumed runs, an explicit
  xi, numpy's generator, and a launch count that does not grow with T;
* ces_small_run refuses a host xi in ensemble mode before any device work; eki keeps its noiseless one-kernel step."""
import ctypes
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from ces_b200 import _lib, calibrate, utils as cutils  # noqa: E402
from ces_b200.engine import Engine  # noqa: E402
from oracle import ensemble_noise_oracle as eno, forward_oracle as fo  # noqa: E402

STEP_J_MAX = 128           # csrc/api.cu kSmallEnsembleJMax: the one-kernel step with ensemble noise; the phases above it
RUN_J_MAX = calibrate._FUSED_ENSEMBLE_J_MAX
UPDATE = {"eks": "eks_update", "aldi": "eks_update_aldi", "aldi_constant": "eks_update_aldi_constant"}
RULES = ("eks", "aldi", "aldi_constant")


def _rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def _problem(p, k, J, dense_gamma=False, dense_sigma=False):
    rs = np.random.RandomState(1000 * p + 10 * k + J)
    A = rs.normal(size=(k, p)) / np.sqrt(p)
    ustar = rs.normal(size=(p, 1))
    Gamma = 0.01 * np.eye(k)
    if dense_gamma:
        Q = rs.normal(size=(k, k))
        Gamma = 0.01 * (np.eye(k) + 0.5 * (Q @ Q.T) / k)
    Sigma0 = 100.0 * np.eye(p)
    if dense_sigma:
        Q = rs.normal(size=(p, p))
        Sigma0 = 50.0 * (np.eye(p) + 0.5 * (Q @ Q.T) / p)
    mu = 0.1 * rs.normal(size=(p, 1))
    y = A @ ustar[:, 0] + 0.1 * rs.normal(size=k)
    U0 = 3.0 * rs.normal(size=(p, J))
    return dict(A=A, ustar=ustar, Gamma=Gamma, Sigma0=Sigma0, mu=mu, y=y, U0=U0, G=fo.lineal(A, U0))


def _engine(pr, small=True):
    p, J = pr["U0"].shape
    k = pr["y"].shape[0]
    if not small:
        os.environ["CES_NO_SMALL_PATH"] = "1"          # read when the handle is created
    try:
        eng = Engine(p, k, J)
    finally:
        os.environ.pop("CES_NO_SMALL_PATH", None)
    eng.set_problem(pr["y"], pr["Gamma"], pr["Sigma0"], pr["mu"], pr["ustar"])
    return eng


def _sampler(pr, T=2):
    p, J = pr["U0"].shape
    s = calibrate.sampling(p, pr["y"].shape[0], J)
    s.ustar, s.mu, s.sigma, s.T = pr["ustar"], pr["mu"], pr["Sigma0"], T
    return s


def _oracle(rule, pr, U, xi, **kw):
    return eno.step(rule, pr["y"], U, fo.lineal(pr["A"], U), pr["Gamma"], pr["mu"], pr["Sigma0"], pr["ustar"], xi, **kw)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _step(eng, rule, pr, noise, xi=None):
    """Engine.step on device tensors; returns (U_next, launches of the step)."""
    torch.cuda.synchronize()
    n0 = eng.launch_count()
    out = eng.step(rule, _dev(pr["U0"]), _dev(pr["G"]), None if xi is None else _dev(xi), noise=noise)[0].cpu().numpy()
    return out, eng.launch_count() - n0


# ---------------------------------------------------------------------------------------------- 1. one step
SHAPES = [
    # p, k, J, dense Gamma, dense Sigma0
    (1, 1, 2, False, False),
    (2, 10, 3, True, True),
    (5, 10, 17, False, True),
    (8, 16, 100, True, False),
    (3, 16, 127, False, False),
    (2, 16, 301, False, True),
    (8, 1, 512, True, True),
    (8, 16, 512, False, False),
]
SEED, STEP = 2 ** 40 + 3, 2 ** 31 + 1


@pytest.mark.parametrize("rule", RULES)
@pytest.mark.parametrize("p,k,J,dense_gamma,dense_sigma", SHAPES)
def test_one_step_matches_the_oracle_and_the_phases(rule, p, k, J, dense_gamma, dense_sigma):
    pr = _problem(p, k, J, dense_gamma, dense_sigma)
    xi = np.random.RandomState(J).normal(size=(J, J))
    small, phases = _engine(pr), _engine(pr, small=False)
    _, chol_launches = _step(small, rule, pr, None, np.random.RandomState(1).normal(size=(p, J)))
    assert chol_launches == 1
    for name, noise, xi_o in (("explicit", ("ensemble", 0, 0, xi), xi),
                              ("stream", ("ensemble", SEED, STEP, None), eno.ensemble_noise(SEED, STEP, J, J))):
        want = _oracle(rule, pr, pr["U0"], xi_o)["Uk"]
        got, launches = _step(small, rule, pr, noise)
        assert (launches == chol_launches) if J <= STEP_J_MAX else (launches > chol_launches), (name, launches)
        assert _rel(got, want) < 1e-10, (name, _rel(got, want))
        ref, ref_launches = _step(phases, rule, pr, noise)
        assert (ref_launches > launches) if J <= STEP_J_MAX else (ref_launches == launches)
        assert _rel(got, ref) < 1e-12, (name, _rel(got, ref))
    small.close()
    phases.close()
    # the numpy-array entry (ces_step_host): explicit xi, then the stream keyed by the step count (0, then 1)
    s = _sampler(pr)
    Ux = getattr(s, UPDATE[rule])(pr["y"], pr["U0"], pr["G"], pr["Gamma"], 0, noise="ensemble", xi=xi)
    assert _rel(Ux, _oracle(rule, pr, pr["U0"], xi)["Uk"]) < 1e-10
    Us = getattr(s, UPDATE[rule])(pr["y"], pr["U0"], pr["G"], pr["Gamma"], 1, noise="ensemble", seed=SEED)
    assert _rel(Us, _oracle(rule, pr, pr["U0"], eno.ensemble_noise(SEED, 1, J, J))["Uk"]) < 1e-10
    s._engine.close()


# ---------------------------------------------------------------------------------------------- 2. bit-exact stream
@pytest.mark.parametrize("rule", RULES)
@pytest.mark.parametrize("p,k,J", [(2, 10, 2), (5, 10, 17), (8, 16, 100), (3, 16, 127), (8, 16, 128)])
def test_stream_equals_its_fill_bit_for_bit(rule, p, k, J):
    """Odd J: the last particle's partner lane is past J, and still draws its half of the pairs."""
    pr = _problem(p, k, J)
    eng = _engine(pr)
    for seed, step in ((7, 0), (SEED, STEP)):
        xi = torch.empty(J, J, dtype=torch.float64, device="cuda")
        _lib.check(eng.lib.ces_fill_ensemble_noise(ctypes.c_void_p(torch.cuda.current_stream().cuda_stream), seed, step,
                                                   ctypes.c_void_p(xi.data_ptr()), J, J, J, 0, 0))
        drawn, _ = _step(eng, rule, pr, ("ensemble", seed, step, None))
        filled, _ = _step(eng, rule, pr, ("ensemble", 0, 0, xi))
        assert np.array_equal(drawn, filled), (seed, step, np.abs(drawn - filled).max())
    eng.close()


# ---------------------------------------------------------------------------------------------- 3. the one-launch run
def _oracle_loop(rule, pr, U, xis, t=None, t_tol=np.inf):
    n = 0
    for xi in xis:
        o = _oracle(rule, pr, U, xi, t_last=t)
        U, t, n = o["Uk"], o["t"], n + 1
        if t > t_tol:
            break
    return U, t, n


def _run(pr, rule, fused, T, model=None, U0=None, **kw):
    s = _sampler(pr, T)
    s.fused_run = fused
    J = pr["U0"].shape[1]
    eng = s._get_engine(J)
    torch.cuda.synchronize()
    n0 = eng.launch_count()
    s.run(pr["y"], pr["U0"] if U0 is None else U0, model or cutils.lineal(pr["A"]), pr["Gamma"], None, update=rule, **kw)
    return s, eng.launch_count() - n0


def _same_run(a, b, tol=1e-12):
    assert len(a.metrics["t"]) == len(b.metrics["t"])
    assert a.Uall.shape == b.Uall.shape
    assert _rel(a.Uall, b.Uall) < tol and _rel(a.Gall, b.Gall) < tol
    for key in ("self-bias", "bias", "self-bias-data", "bias-data", "t"):
        assert np.allclose(a.metrics[key], b.metrics[key], rtol=tol, atol=0), key


@pytest.mark.parametrize("rule", RULES)
@pytest.mark.parametrize("p,k,J", [(2, 10, 100), (8, 16, RUN_J_MAX - 1), (8, 16, RUN_J_MAX)])
def test_fused_run_with_the_stream_stops_and_resumes(rule, p, k, J):
    """A first call stops on t_tol in its 4th iteration, a resumed call continues the step count of the stream; the one-launch
    run equals the per-iteration loop to 1e-12 and the oracle loop fed ensemble_noise(seed, t, J, J) to 1e-10, and leaves
    numpy's generator untouched (lineal draws nothing)."""
    seed = 2 ** 33 + 7
    pr = _problem(p, k, J)
    xis = lambda t0, n: [eno.ensemble_noise(seed, t0 + i, J, J) for i in range(n)]
    t3 = _oracle_loop(rule, pr, pr["U0"], xis(0, 3))[1]
    t4 = _oracle_loop(rule, pr, pr["U0"], xis(0, 4))[1]
    t_tol = 0.5 * (t3 + t4)
    U, t, n = _oracle_loop(rule, pr, pr["U0"], xis(0, 20), t_tol=t_tol)
    assert n == 4
    U2, t2, _ = _oracle_loop(rule, pr, U, xis(4, 3), t=t)
    runs = {}
    for fused in (True, False):
        state = np.random.get_state()
        s, launches = _run(pr, rule, fused, 20, t_tol=t_tol, noise="ensemble", seed=seed)
        assert len(s.metrics["t"]) == 4 and abs(s.metrics["t"][-1] - t) <= 1e-10 * t
        assert _rel(s.Ustar, U) < 1e-10, _rel(s.Ustar, U)
        s.T = 3
        s.run(pr["y"], s.Ustar, cutils.lineal(pr["A"]), pr["Gamma"], None, update=rule, t_tol=1e9, noise="ensemble",
              seed=seed)
        assert len(s.metrics["t"]) == 7 and abs(s.metrics["t"][-1] - t2) <= 1e-10 * t2
        assert _rel(s.Ustar, U2) < 1e-10, _rel(s.Ustar, U2)
        after = np.random.get_state()
        assert np.array_equal(after[1], state[1]) and after[2:] == state[2:]
        runs[fused] = (s, launches)
    _same_run(runs[True][0], runs[False][0])
    assert runs[True][1] < runs[False][1]


@pytest.mark.parametrize("rule", RULES)
def test_fused_run_with_an_explicit_xi(rule):
    """One (J, J) xi at every iteration (odd J: the device copy is padded to an even leading dimension)."""
    p, k, J, T = 3, 7, 45, 5
    pr = _problem(p, k, J, dense_gamma=True)
    xi = np.random.RandomState(5).normal(size=(J, J))
    a, la = _run(pr, rule, True, T, t_tol=1e9, noise="ensemble", xi=xi)
    b, lb = _run(pr, rule, False, T, t_tol=1e9, noise="ensemble", xi=xi)
    _same_run(a, b)
    assert la < lb
    U, t, n = _oracle_loop(rule, pr, pr["U0"], [xi] * T)
    assert len(a.metrics["t"]) == n == T and abs(a.metrics["t"][-1] - t) <= 1e-10 * t
    assert _rel(a.Ustar, U) < 1e-10, _rel(a.Ustar, U)


@pytest.mark.parametrize("rule", ["aldi", "eks"])
def test_fused_run_with_banana_consumes_numpys_stream_as_the_loop_does(rule):
    """banana draws two normals per particle per forward pass from numpy's global generator; the update draws nothing."""
    J = 64
    model = cutils.banana()
    ustar = np.array([[0.5], [1.0]])
    rs = np.random.RandomState(2)
    pr = dict(ustar=ustar, Gamma=0.01 * np.eye(2), Sigma0=25.0 * np.eye(2), mu=np.zeros((2, 1)),
              y=np.asarray(model(ustar[:, 0]), dtype=float), U0=ustar + rs.normal(size=(2, J)))
    out = {}
    for fused in (True, False):
        np.random.seed(11)
        s, launches = _run(pr, rule, fused, 8, model=model, t_tol=1e9, noise="ensemble", seed=4)
        out[fused] = (s, np.random.get_state(), launches)
    (a, sa, la), (b, sb, lb) = out[True], out[False]
    _same_run(a, b)
    assert np.array_equal(sa[1], sb[1]) and sa[2:] == sb[2:]
    assert la < lb
    np.random.seed(11)
    untouched = np.random.get_state()
    assert not np.array_equal(sa[1], untouched[1]) or sa[2] != untouched[2]      # banana did draw


def test_fused_run_launch_count_does_not_depend_on_T():
    pr = _problem(2, 10, 100)
    counts = [_run(pr, "aldi", True, T, t_tol=1e30, noise="ensemble", seed=1)[1] for T in (5, 50)]
    assert counts[0] == counts[1], counts
    s, _ = _run(pr, "aldi", True, 50, t_tol=1e30, noise="ensemble", seed=1)
    assert len(s.metrics["t"]) == 50
    # above the J limit the run takes the per-iteration loop
    big = _problem(2, 10, RUN_J_MAX + 1)
    assert _run(big, "aldi", True, 5, t_tol=1e30, noise="ensemble", seed=1)[1] > 5


# ---------------------------------------------------------------------------------------------- 4. refusals, eki
def test_small_run_refuses_a_host_xi_in_ensemble_mode():
    p, k, J, T = 2, 10, 100, 3
    pr = _problem(p, k, J)
    eng = _engine(pr)
    lib, h = eng.lib, eng.h
    Ad = _dev(pr["A"])
    U0 = np.ascontiguousarray(pr["U0"])
    xi_host = np.zeros((T, p, J))
    Ut, Gt, S, tv = np.full((T + 1, p, J), 7.0), np.full((T + 1, k, J), 7.0), np.full((T, 16), 7.0), np.full(T, 7.0)
    n = ctypes.c_int64(7)
    assert lib.ces_set_noise(h, _lib.NOISES["ensemble"], 3, 0, None, 0) == 0
    torch.cuda.synchronize()
    before = eng.launch_count()
    rc = lib.ces_small_run(h, _lib.RULES["aldi"], _lib.TS_FROBENIUS, 0.0, 1.0, _lib.MAPS["lineal"],
                           ctypes.c_void_p(Ad.data_ptr()), p, None, None, _lib.host_ptr(U0), _lib.host_ptr(xi_host), 0, 0, T,
                           0.0, 0, 2.0, _lib.host_ptr(Ut), _lib.host_ptr(Gt), _lib.host_ptr(S), _lib.host_ptr(tv),
                           ctypes.byref(n))
    assert rc == _lib.CES_ERR_INVALID
    assert b"ces_small_run: ensemble noise takes its xi from ces_set_noise" in lib.ces_last_error(), lib.ces_last_error()
    torch.cuda.synchronize()
    assert eng.launch_count() == before
    for out in (Ut, Gt, S, tv, np.array([n.value])):
        assert (out == 7).all()
    eng.close()


def test_eki_under_ensemble_noise_keeps_the_noiseless_one_kernel_step():
    pr = _problem(5, 10, 17)
    eng = _engine(pr)
    ref, ref_launches = _step(eng, "eki", pr, None)
    got, launches = _step(eng, "eki", pr, ("ensemble", 4, 0, None))
    assert ref_launches == launches == 1
    assert np.array_equal(got, ref)
    eng.close()
