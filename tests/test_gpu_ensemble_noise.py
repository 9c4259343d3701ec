"""noise='ensemble' on the device (DESIGN.md section 4g): sqrt(2h / n_C) (U - ubar) xi with a J x J xi.

* explicit xi against oracle/ensemble_noise_oracle.step within the suite's 1e-10 bar: every noisy rule, diagonal and
  dense Gamma, J < p and J > p, odd J and J off the 16-column grid, several D panels, every time_step rule, the device
  path (sampling.run) and the pipelined host path (eks_update* on numpy arrays, with the chunked download);
* ces_fill_ensemble_noise value for value against oracle/ensemble_noise_oracle.ensemble_noise, and sampling.run with the device
  stream against the oracle loop fed the restated xi (resumed runs, a problem small enough for the fused path);
* the statistics of the increments: covariance C^uu - 1e-8 I, and no component outside span(U - ubar) when J < p;
* column-sharded steps (2-4 GPUs) against the single-GPU step;
* refusals before any device work."""
import ctypes
import os
import socket
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from ces_b200 import _lib, calibrate, utils as cutils  # noqa: E402
from ces_b200.engine import Engine  # noqa: E402
from oracle import ensemble_noise_oracle as eno, forward_oracle as fo  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NOISE_TOL = 1e-13
UPDATE = {"eks": "eks_update", "aldi": "eks_update_aldi", "aldi_constant": "eks_update_aldi_constant"}


def _rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def _problem(p, k, J, dense=False, seed=0):
    rs = np.random.RandomState(1000 * p + 10 * k + J + seed)
    A = rs.normal(size=(k, p)) / np.sqrt(p)
    ustar = rs.normal(size=(p, 1))
    if dense:
        Q = rs.normal(size=(k, k))
        Gamma = 0.01 * (np.eye(k) + 0.5 * (Q @ Q.T) / k)
    else:
        Gamma = 0.01 * np.eye(k)
    y = A @ ustar[:, 0] + 0.1 * rs.normal(size=k)
    U0 = 3.0 * rs.normal(size=(p, J))
    return A, ustar, Gamma, y, U0


def _sampler(p, k, J, ustar, T=2, d_panel_bytes=0):
    s = calibrate.sampling(p, k, J)
    s.ustar, s.mu, s.sigma, s.T = ustar, np.zeros((p, 1)), 100.0 * np.eye(p), T
    if d_panel_bytes:
        s.d_panel_bytes = d_panel_bytes
    return s


def _oracle_loop(rule, s, A, y, Gamma, U, xis, ts_kw, t=None, t_tol=np.inf):
    """ensemble_noise_oracle.step iteration by iteration with G = A U and the given J x J xi per step."""
    n = 0
    for xi in xis:
        o = eno.step(rule, y, U, fo.lineal(A, U), Gamma, s.mu, s.sigma, s.ustar, xi, t_last=t, **ts_kw)
        U, t, n = o["Uk"], o["t"], n + 1
        if t > t_tol:
            break
    return U, t, n


def _ts_kw(time_step):
    return {} if time_step is None else {"time_step": time_step, "spinup": 0.0, "delta_t": 0.05}


# ---------------------------------------------------------------------------------------------- 1. explicit xi
CASES = [
    # rule, dense Gamma, p, k, J, time_step, panels (0: one panel)
    ("aldi", False, 24, 40, 13, None, 0),             # J < p, odd
    ("eks", True, 24, 40, 13, None, 0),
    ("aldi_constant", False, 24, 40, 13, None, 0),
    ("aldi", True, 8, 30, 100, None, 0),              # J > p, not a multiple of 16
    ("eks", False, 8, 30, 301, None, 3),              # three 128-column panels of D
    ("aldi_constant", True, 8, 30, 301, None, 3),
    ("aldi", False, 16, 30, 77, "constant", 0),
    ("eks", False, 16, 30, 77, "constant", 0),
    ("aldi", False, 16, 30, 77, "mix", 0),
    ("eks", True, 16, 30, 77, "mix", 0),
    ("aldi", False, 16, 30, 77, "spectral", 0),
    ("eks", False, 16, 30, 77, "spectral", 0),
]


def _panel_bytes(J, panels):
    return 8 * (-(-J // 16) * 16) * 128 if panels else 0


@pytest.mark.parametrize("rule,dense,p,k,J,time_step,panels", CASES)
def test_explicit_xi_device_run_matches_the_oracle(rule, dense, p, k, J, time_step, panels):
    """sampling.run (device-resident loop, Engine.step) with one explicit J x J xi used at both iterations."""
    A, ustar, Gamma, y, U0 = _problem(p, k, J, dense)
    xi = np.random.RandomState(J).normal(size=(J, J))
    s = _sampler(p, k, J, ustar, T=2, d_panel_bytes=_panel_bytes(J, panels))
    state = np.random.get_state()
    s.run(y, U0, cutils.lineal(A), Gamma, None, update=rule, t_tol=1e9, noise="ensemble", xi=xi, **_ts_kw(time_step))
    U, t, n = _oracle_loop(rule, s, A, y, Gamma, U0, [xi, xi], _ts_kw(time_step))
    assert n == 2 and len(s.metrics["t"]) == 2 and abs(s.metrics["t"][-1] - t) <= 1e-10 * t
    assert _rel(s.Ustar, U) < 1e-10, (rule, dense, J, time_step, _rel(s.Ustar, U))
    after = np.random.get_state()
    assert np.array_equal(after[1], state[1]) and after[2] == state[2]


@pytest.mark.parametrize("rule,dense,p,k,J,time_step,panels", CASES + [("aldi", False, 8, 16, 4500, None, 0),
                                                                       ("aldi_constant", False, 8, 16, 4500, None, 0)])
def test_explicit_xi_host_updates_match_the_oracle(rule, dense, p, k, J, time_step, panels):
    """eks_update* on numpy arrays (ces_step_host, or the phases for the non-default step sizes), two steps; J = 4500
    downloads U_next in overlapped column chunks, each chunk's noise finished before its copy is queued."""
    A, ustar, Gamma, y, U0 = _problem(p, k, J, dense)
    rs = np.random.RandomState(J + 1)
    xis = [rs.normal(size=(J, J)), rs.normal(size=(J, J))]
    s = _sampler(p, k, J, ustar, d_panel_bytes=_panel_bytes(J, panels))
    U = U0
    for i, xi in enumerate(xis):
        U = getattr(s, UPDATE[rule])(y, U, fo.lineal(A, U), Gamma, i, noise="ensemble", xi=xi, **_ts_kw(time_step))
    Uo, t, _ = _oracle_loop(rule, s, A, y, Gamma, U0, xis, _ts_kw(time_step))
    assert abs(s.metrics["t"][-1] - t) <= 1e-10 * t
    assert _rel(U, Uo) < 1e-10, (rule, dense, J, time_step, _rel(U, Uo))


# ---------------------------------------------------------------------------------------------- 2. the device stream
@pytest.mark.parametrize("seed", [0, 2 ** 32 + 5, 2 ** 40 + 3])
@pytest.mark.parametrize("step", [0, 3, 2 ** 31 + 1])
def test_fill_ensemble_noise_is_the_restated_stream(seed, step):
    lib = _lib.load()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for rows, r0 in ((1, 0), (7, 65535), (300, 1)):
        for cols in (1, 2, 511, 512, 513):
            for c0 in (0, 1, 511, 512, 2 ** 32 + 1):
                buf = torch.full((rows, cols + 5), float("nan"), dtype=torch.float64, device="cuda")
                _lib.check(lib.ces_fill_ensemble_noise(st, seed, step, ctypes.c_void_p(buf.data_ptr()), buf.stride(0), rows,
                                                       cols, r0, c0))
                got = buf.cpu().numpy()
                want = eno.ensemble_noise(seed, step, rows, cols, r0, c0)
                assert np.abs(got[:, :cols] - want).max() <= NOISE_TOL, (rows, r0, cols, c0)
                assert np.all(np.isnan(got[:, cols:])), (rows, r0, cols, c0)
    # more rows than gridDim.y can hold: the grid-stride loop covers all of them
    rows = 65536 + 3
    buf = torch.empty((rows, 2), dtype=torch.float64, device="cuda")
    _lib.check(lib.ces_fill_ensemble_noise(st, seed, step, ctypes.c_void_p(buf.data_ptr()), 2, rows, 2, 0, 6))
    assert np.abs(buf.cpu().numpy() - eno.ensemble_noise(seed, step, rows, 2, 0, 6)).max() <= NOISE_TOL


@pytest.mark.parametrize("rule", ["aldi", "eks", "aldi_constant"])
@pytest.mark.parametrize("p,k,J,panels", [(2, 10, 100, 0), (24, 40, 301, 3)])
def test_device_stream_run_matches_the_oracle_and_resumes(rule, p, k, J, panels):
    """sampling.run(noise='ensemble', seed) against the oracle loop fed xi_t = ensemble_noise(seed, t, J, J): a first call
    that stops on t_tol in step 4, then a resumed call continuing the step count.  p = 2, k = 10, J = 100 fits the fused
    single-launch path, which must not be taken (it has no ensemble noise).  Numpy's generator is untouched."""
    seed = 2 ** 33 + 7
    A, ustar, Gamma, y, U0 = _problem(p, k, J)
    s = _sampler(p, k, J, ustar, T=20, d_panel_bytes=_panel_bytes(J, panels))
    xis = lambda t0, n: [eno.ensemble_noise(seed, t0 + i, J, J) for i in range(n)]
    t3 = _oracle_loop(rule, s, A, y, Gamma, U0, xis(0, 3), {})[1]
    t4 = _oracle_loop(rule, s, A, y, Gamma, U0, xis(0, 4), {})[1]
    t_tol = 0.5 * (t3 + t4)
    state = np.random.get_state()
    s.run(y, U0, cutils.lineal(A), Gamma, None, update=rule, t_tol=t_tol, noise="ensemble", seed=seed)
    U, t, n = _oracle_loop(rule, s, A, y, Gamma, U0, xis(0, 20), {}, t_tol=t_tol)
    assert n == 4 and len(s.metrics["t"]) == 4 and abs(s.metrics["t"][-1] - t) <= 1e-10 * t
    assert _rel(s.Ustar, U) < 1e-10, _rel(s.Ustar, U)
    s.T = 3
    s.run(y, s.Ustar, cutils.lineal(A), Gamma, None, update=rule, t_tol=1e9, noise="ensemble", seed=seed)
    U2, t2, n2 = _oracle_loop(rule, s, A, y, Gamma, U, xis(4, 3), {}, t=t)
    assert n2 == 3 and len(s.metrics["t"]) == 7 and abs(s.metrics["t"][-1] - t2) <= 1e-10 * t2
    assert _rel(s.Ustar, U2) < 1e-10, _rel(s.Ustar, U2)
    after = np.random.get_state()
    assert np.array_equal(after[1], state[1]) and after[2] == state[2]


def test_host_update_with_the_device_stream_matches_the_oracle():
    p, k, J, seed = 8, 20, 150, 12
    A, ustar, Gamma, y, U0 = _problem(p, k, J)
    s = _sampler(p, k, J, ustar)
    s.noise, s.seed = "ensemble", seed                  # as attributes
    state = np.random.get_state()
    U = U0
    for i in range(2):
        U = s.eks_update_aldi(y, U, fo.lineal(A, U), Gamma, i)
    Uo = _oracle_loop("aldi", s, A, y, Gamma, U0, [eno.ensemble_noise(seed, t, J, J) for t in range(2)], {})[0]
    assert _rel(U, Uo) < 1e-10
    after = np.random.get_state()
    assert np.array_equal(after[1], state[1]) and after[2] == state[2]


# ---------------------------------------------------------------------------------------------- 3. statistics
def _one_step(eng, rule, U, G, noise, xi=None):
    Ud = torch.from_numpy(U).cuda()
    Gd = torch.from_numpy(G).cuda()
    xd = torch.from_numpy(xi).cuda() if xi is not None else None
    out, hk, _ = eng.step(rule, Ud, Gd, xd, noise=noise)
    return out.cpu().numpy(), hk


def test_increments_have_the_ensemble_covariance():
    """p = 8, J = 8192: Delta = (U+_Philox - U+_{xi=0}) / sqrt(2h) has E[Delta Delta^T / J | U] = U~ U~^T / n_C = C^uu - 1e-8 I;
    every entry within 5 standard errors sqrt((C_ii C_jj + C_ij^2) / J)."""
    p, k, J = 8, 12, 8192
    A, ustar, Gamma, y, U0 = _problem(p, k, J)
    eng = Engine(p, k, J)
    eng.set_problem(y, Gamma, 100.0 * np.eye(p), np.zeros(p), ustar)
    G = fo.lineal(A, U0)
    base, hk0 = _one_step(eng, "aldi", U0, G, None, np.zeros((p, J)))
    noisy, hk = _one_step(eng, "aldi", U0, G, ("ensemble", 5, 0, None))
    assert hk == hk0
    D = (noisy - base) / np.sqrt(2 * hk)
    Ut = U0 - U0.mean(axis=1)[:, None]
    C = Ut @ Ut.T / (J - 1)
    emp = D @ D.T / J
    se = np.sqrt((np.outer(np.diag(C), np.diag(C)) + C ** 2) / J)
    z = np.abs(emp - C) / se
    assert z.max() < 5.0, z.max()
    eng.close()


@pytest.mark.parametrize("rule", ["aldi", "eks", "aldi_constant"])
def test_increments_stay_in_the_ensemble_span(rule):
    """J = 16 < p = 64: the ensemble noise has no component outside span(U - ubar) (1e-12 relative); the Cholesky noise
    of the same step puts ~1e-4 sqrt(2h) there (rank-deficient C^uu + 1e-8 I), so the check can tell the two apart."""
    p, k, J = 64, 30, 16
    A, ustar, Gamma, y, U0 = _problem(p, k, J)
    eng = Engine(p, k, J)
    eng.set_problem(y, Gamma, 100.0 * np.eye(p), np.zeros(p), ustar)
    G = fo.lineal(A, U0)
    base, _ = _one_step(eng, rule, U0, G, None, np.zeros((p, J)))
    Q = np.linalg.qr(U0 - U0.mean(axis=1)[:, None])[0][:, :J - 1]
    out_of_span = lambda d: np.linalg.norm(d - Q @ (Q.T @ d)) / np.linalg.norm(d)
    ens, _ = _one_step(eng, rule, U0, G, ("ensemble", 9, 1, None))
    chol, _ = _one_step(eng, rule, U0, G, None, np.random.RandomState(3).normal(size=(p, J)))
    assert out_of_span(ens - base) <= 1e-12, out_of_span(ens - base)
    assert out_of_span(chol - base) >= 1e-6, out_of_span(chol - base)
    eng.close()


# ---------------------------------------------------------------------------------------------- 4. sharding
def _free_port():
    with socket.socket() as sock:
        sock.bind(("127.0.0.1", 0))
        return sock.getsockname()[1]


def _shard_worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist

    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    errs = []
    try:
        for rule, p, k, J in (("aldi", 24, 40, 301), ("eks", 24, 40, 130), ("aldi_constant", 16, 272, 4300)):
            A, ustar, Gamma, y, U0 = _problem(p, k, J)
            G = fo.lineal(A, U0)
            xi = np.random.RandomState(J).normal(size=(J, J))
            single = Engine(p, k, J)
            single.set_problem(y, Gamma, 100.0 * np.eye(p), np.zeros(p), ustar)
            refs = {"philox": single.step_host(rule, U0, G, None, noise=("ensemble", 77, 3, None))[0],
                    "explicit": single.step_host(rule, U0, G, None, noise=("ensemble", 0, 0, xi))[0]}
            single.close()
            for gather in ("1", "0"):                        # peer pulls over CUDA IPC, NCCL all-gathers
                os.environ["CES_PEER_GATHER"] = gather
                eng = Engine(p, k, J, group=dist.group.WORLD)
                eng.set_problem(y, Gamma, 100.0 * np.eye(p), np.zeros(p), ustar)
                sl = slice(eng.col_lo, eng.col_hi)
                dev = lambda a: torch.from_numpy(np.ascontiguousarray(a[:, sl])).cuda()
                for which, noise in (("philox", ("ensemble", 77, 3, None)), ("explicit", ("ensemble", 0, 0, xi[:, sl]))):
                    ref = refs[which][:, sl]
                    if eng.cols:
                        out = eng.step(rule, dev(U0), dev(G), None, noise=noise)[0].cpu().numpy()
                        errs.append((rule, gather, which, "device", _rel(out, ref)))
                    host = eng.step_host(rule, np.ascontiguousarray(U0[:, sl]), np.ascontiguousarray(G[:, sl]), None,
                                         noise=noise)[0]
                    if eng.cols:
                        errs.append((rule, gather, which, "host", _rel(host, ref)))
                eng.close()
        q.put((rank, errs))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3, 4])
def test_sharded_ensemble_noise_matches_one_gpu(world):
    """Each rank holds every U~ block after the gathers and adds sum_s U~_s xi[s, its columns]: the sharded step equals the
    single-GPU step to 1e-12, on the device phases with both gather paths and on the pipelined host path."""
    import torch.multiprocessing as mp

    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_shard_worker, args=(r, world, port, q)) for r in range(world)]
    for pr in procs:
        pr.start()
    for pr in procs:
        pr.join(600)
        assert pr.exitcode == 0
    for rank, errs in sorted(q.get(timeout=10) for _ in range(world)):
        for e in errs:
            assert e[-1] < 1e-12, (rank, e)


# ---------------------------------------------------------------------------------------------- 5. refusals
def test_invalid_settings_are_refused_before_device_work():
    p, k, J = 4, 6, 10
    A, ustar, Gamma, y, U0 = _problem(p, k, J)
    G = fo.lineal(A, U0)
    eng = Engine(p, k, J)
    eng.set_problem(y, Gamma, 100.0 * np.eye(p), np.zeros(p), ustar)
    lib = eng.lib
    Ud, Gd = torch.from_numpy(U0).cuda(), torch.from_numpy(G).cuda()
    out = torch.full_like(Ud, 7.0)
    # the factored formulation never gathers U~: refused by ces_step with nothing written
    hk, met = ctypes.c_double(), (ctypes.c_double * 4)()
    assert lib.ces_set_noise(eng.h, 1, 0, 0, None, 0) == 0
    assert lib.ces_step(eng.h, 1, 0, 0.0, 1.0, 1, ctypes.c_void_p(Ud.data_ptr()), J, ctypes.c_void_p(Gd.data_ptr()), J,
                        None, 0, ctypes.c_void_p(out.data_ptr()), J, ctypes.byref(hk), met) == _lib.CES_ERR_INVALID
    assert b"factored" in lib.ces_last_error()
    torch.cuda.synchronize()
    assert bool((out == 7.0).all())
    # explicit xi: 16-byte base, even ld >= cols
    xi = torch.zeros(J, J + 2, dtype=torch.float64, device="cuda")
    assert lib.ces_set_noise(eng.h, 1, 0, 0, ctypes.c_void_p(xi.data_ptr() + 8), J + 2) == _lib.CES_ERR_ALIGN
    assert lib.ces_set_noise(eng.h, 1, 0, 0, ctypes.c_void_p(xi.data_ptr()), J + 1) == _lib.CES_ERR_ALIGN
    assert lib.ces_set_noise(eng.h, 1, 0, 0, ctypes.c_void_p(xi.data_ptr()), J - 2) == _lib.CES_ERR_ALIGN
    assert lib.ces_set_noise(eng.h, 2, 0, 0, None, 0) == _lib.CES_ERR_INVALID
    with pytest.raises(ValueError):
        eng.set_noise("ensemble", 0, 0, torch.zeros(J, J - 1, dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        eng.set_noise("gaussian")
    # eki has no noise term: the ensemble setting changes nothing (it takes the phases instead of the one-kernel path)
    ref = eng.step("eki", Ud, Gd, None)[0].cpu().numpy()
    ens = eng.step("eki", Ud, Gd, None, noise=("ensemble", 4, 0, None))[0].cpu().numpy()
    assert _rel(ens, ref) < 1e-12
    eng.close()
    # sampling: bad settings raise ValueError before the engine exists and before numpy's generator moves
    s = _sampler(p, k, J, ustar)
    state = np.random.get_state()
    for kw in ({"noise": "gaussian"}, {"noise": "ensemble", "formulation": "factored"},
               {"noise": "ensemble", "xi": np.zeros((p, J))}, {"noise": "ensemble", "xi": np.zeros((J, J - 1))}):
        with pytest.raises(ValueError):
            s.eks_update(y, U0, G, Gamma, 0, **kw)
        with pytest.raises(ValueError):
            s.run(y, U0, cutils.lineal(A), Gamma, None, update="aldi", **kw)
    assert s._engine is None
    after = np.random.get_state()
    assert np.array_equal(after[1], state[1]) and after[2] == state[2]
