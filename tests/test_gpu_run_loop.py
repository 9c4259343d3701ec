"""sampling.run's state carry-over of 'pde' models (``ws`` pool, ``update_wt``) on the device and through the reference's
per-particle host protocol, and the names of the online-save directory and ``online_path`` on both run paths."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from ces_b200 import calibrate, utils as cu  # noqa: E402
from oracle import eks_oracle as eo  # noqa: E402


def _lorenz63_case():
    model = cu.lorenz63(l_window=1, freq=50)
    model.substeps = 8
    t = np.arange(0, 2.0 + 1e-9, 0.02)
    wt = np.array([1.0, 2.0, 25.0])
    y = model.statistics(model.solve(wt, t, args=(28.0, 8.0 / 3)))
    J, p = 16, 2
    rng = np.random.default_rng(1)
    U0 = np.array([[30.0], [3.0]]) + np.array([[3.0], [0.5]]) * rng.standard_normal((p, J))
    xi = rng.standard_normal((p, J))                # explicit update noise: the pool is numpy's only consumer
    pool = wt + rng.standard_normal((40, 3))

    class HostProtocol(object):                     # the same model through the reference's per-particle interface only
        type, n_state, n_obs, model_name = 'pde', 3, model.n_obs, 'lorenz63'
        solve, statistics = staticmethod(model.solve), staticmethod(model.statistics)

    def run(m, **kw):
        s = calibrate.sampling(p, model.n_obs, J)
        s.ustar, s.mu, s.sigma, s.T = np.array([[28.0], [8.0 / 3]]), np.array([[30.0], [3.0]]), np.diag([25.0, 1.0]), 3
        s.run(y, U0, m, np.diag((0.05 * np.abs(y) + 0.1) ** 2), None, t=t, xi=xi, t_tol=1e9, **kw)
        return s

    return model, HostProtocol(), run, pool, wt, J


def test_ws_pool_draws_replay_numpy_on_both_pde_paths():
    """With ``ws=``: one randint over the pool before the loop and one after every forward pass; every draw but the final
    pass's is appended to Wall, and the final pass's draw gives W0."""
    model, host, run, pool, _, J = _lorenz63_case()
    np.random.seed(5)
    idx = [np.random.randint(pool.shape[0], size=J) for _ in range(1 + 3 + 1)]
    after = np.random.get_state()
    out = []
    for m in (model, host):
        np.random.seed(5)
        s = run(m, ws=pool)
        assert np.array_equal(np.random.get_state()[1], after[1]) and np.random.get_state()[2:] == after[2:]
        assert len(s.Wall) == 4 and all(np.array_equal(w, i) for w, i in zip(s.Wall, idx[:4]))
        assert np.array_equal(s.W0, pool[idx[4]].T)
        out.append(s)
    a, b = out
    assert np.abs(a.Gall - b.Gall).max() < 1e-6 * np.abs(b.Gall).max()
    assert np.abs(a.Ustar - b.Ustar).max() < 1e-6 * np.abs(b.Ustar).max()


def test_update_wt_false_keeps_the_initial_state_on_both_pde_paths():
    model, host, run, _, wt, J = _lorenz63_case()
    out = [run(m, wt=wt, update_wt=False) for m in (model, host)]
    for s in out:
        assert np.array_equal(s.W0, np.tile(wt, J).reshape(J, 3).T)
    a, b = out                                      # the device pass started from the same states as the host's
    assert np.abs(a.Gall - b.Gall).max() < 1e-6 * np.abs(b.Gall).max()


@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("nexp", [None, 3])
def test_online_directory_and_online_path_names(tmp_path, fused, nexp):
    d, k, J = 2, 6, 60
    pr = eo.linear_gaussian_problem(d, k, J)
    s = calibrate.sampling(d, k, J)
    s.ustar, s.mu, s.sigma, s.T, s.fused_run = pr["ustar"], pr["mu"], pr["Sigma0"], 2, fused
    s.directory = str(tmp_path)
    if nexp is not None:
        s.nexp = nexp
    suffix = "-0060" + ("" if nexp is None else "-03")
    np.random.seed(2)
    s.run(pr["y"], pr["U0"], cu.lineal(pr["A"]), pr["Gamma"], None, save_online=True, t_tol=1e9)
    assert s.online_path == str(tmp_path) + "/ensembles/lineal" + suffix + "/"
    assert os.listdir(os.path.join(str(tmp_path), "ensembles")) == ["lineal-eks-000" + suffix]
    where = os.path.join(str(tmp_path), "ensembles", "lineal-eks-000" + suffix)
    assert sorted(os.listdir(where)) == ["Gensemble_0000.npy", "Gensemble_0001.npy", "ensemble_0000.npy",
                                         "ensemble_0001.npy", "metrics.pkl"]
    assert np.array_equal(np.load(os.path.join(where, "ensemble_0001.npy")), s.Uall[1])
