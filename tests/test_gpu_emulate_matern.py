"""GPEmulator(kernel="Matern12" / "Matern32" / "Matern52") and MCMC.emulator_mh through it on the device
(ces_b200/emulate.py, csrc/emulate.cu) against scikit-learn's values in tests/golden/gp_matern_cases.npz and against
oracle/gp_matern_oracle.py: LML and gradient, bit-identical repeats, latent predictions, duplicate points, the ill-conditioned
case, the fit, chains sample for sample with numpy's generator, the conditioned state across a change of family, and the
Darcy Calibrate -> Emulate -> Sample example with Matern 5/2 against the true-model chains."""
import ctypes
import os

import numpy as np
import pytest
from scipy.stats import multivariate_normal

pytestmark = pytest.mark.gpu

from ces_b200 import _lib, calibrate, sample as csample  # noqa: E402
from ces_b200.emulate import GPEmulator  # noqa: E402

GM = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gp_matern_cases.npz"))
NAMES = [str(n) for n in GM["names"]]
FAMILIES = [str(f) for f in GM["families"]]
JITTER = float(GM["jitter"])


def _emulator(name, fam):
    """Golden outputs are already whitened: Gamma = I, whose eigh is exactly the identity, feeds them through unchanged."""
    X, G = GM[name + "/X"], GM[name + "/G"]
    emu = GPEmulator(U=X, G=G, Gamma=np.eye(G.shape[0]), jitter=JITTER, kernel=fam)
    assert np.array_equal(emu.transform, np.eye(G.shape[0])) and emu.kernel == fam
    return emu


@pytest.mark.parametrize("fam", FAMILIES)
@pytest.mark.parametrize("name", NAMES)
def test_lml_and_gradient_match_sklearn_and_repeat_bitwise(fam, name):
    emu = _emulator(name, fam)
    pre = "%s/%s/" % (fam, name)
    theta = GM[pre + "theta"]
    lml, grad = emu.log_marginal_likelihood(theta, eval_gradient=True)
    want, want_g = GM[pre + "lml"], GM[pre + "grad"]
    tol = 1e-6 if name.startswith("cond") else 1e-9          # ill-conditioned K (see tests/test_gp_oracle.py)
    assert np.all(np.abs(lml - want) <= tol * np.abs(want)), (fam, name)
    assert np.all(np.abs(grad - want_g) <= tol * np.maximum(np.abs(want_g).max(axis=1, keepdims=True), 1.0)), (fam, name)
    assert np.all(np.isfinite(grad))
    lml2, grad2 = emu.log_marginal_likelihood(theta, eval_gradient=True)
    assert np.array_equal(lml, lml2) and np.array_equal(grad, grad2)
    assert np.array_equal(emu.log_marginal_likelihood(theta), lml)


@pytest.mark.parametrize("fam", FAMILIES)
@pytest.mark.parametrize("name,m", [("p2_n100_k10", 1), ("p2_n100_k10", 33), ("p2_n100_k10", 100), ("p1_n37_k1", 1000),
                                    ("p8_n1000_k4", 1), ("p8_n1000_k4", 33), ("p8_n150_k64", 17), ("p32_n200_k3", 50),
                                    ("dup_p3_n60_k2", 40), ("cond_p2_n100_k1", 40)])
def test_predict_matches_sklearn(fam, name, m):
    emu = _emulator(name, fam)
    pre = "%s/%s/" % (fam, name)
    theta = GM[pre + "theta"]
    emu.set_hyperparameters(np.exp(theta[:, 0]), np.exp(theta[:, 1:-1]), np.exp(theta[:, -1]))
    emu.theta = theta
    mean, var = emu.predict(GM[name + "/U"][:, :m])
    Y = GM[name + "/G"] - GM[name + "/G"].mean(axis=1, keepdims=True)
    scale = np.abs(Y).max(axis=1)[:, None]
    sf2 = np.exp(theta[:, :1])
    assert mean.shape == var.shape == (Y.shape[0], m)
    tol_v = 1e-8 if name.startswith("cond") else 1e-10     # ill-conditioned K: see tests/test_gp_matern_oracle.py
    assert np.all(np.abs(mean - GM[pre + "mean"][:, :m]) <= tol_v * scale), (fam, name)
    assert np.all(var >= 0.0)
    assert np.all(np.abs(var - GM[pre + "var"][:, :m]) <= tol_v * sf2), (fam, name)


@pytest.mark.parametrize("fam", FAMILIES)
@pytest.mark.parametrize("name", [n for n in NAMES if ("Matern12/%s/fit_lml" % n) in GM.files])
def test_fit_reaches_sklearn_optimum(fam, name):
    emu = _emulator(name, fam)
    emu.fit()
    want = GM["%s/%s/fit_lml" % (fam, name)]
    assert np.all(emu.fit_lml >= want - 1e-8 * np.abs(want)), (fam, emu.fit_lml - want)
    assert np.allclose(emu.log_marginal_likelihood(), emu.fit_lml, rtol=1e-12, atol=0)


def _chain_setup(fam):
    name = "p2_n100_k10"
    emu = _emulator(name, fam)
    emu.theta = GM["%s/%s/theta" % (fam, name)]
    Ustar = GM["chain/Ustar"]
    enka = calibrate.sampling(2, emu.k, Ustar.shape[1])
    enka.Ustar = Ustar
    prior = multivariate_normal(GM["chain/prior_mean"], GM["chain/prior_cov"])
    mc = csample.MCMC()
    mc.y_obs = GM["chain/ytil"]
    return emu, enka, prior, mc


def _state_equal(pre, suffix=""):
    st = np.random.get_state()
    return (np.array_equal(st[1], GM[pre + "key" + suffix]) and [st[2], st[3]] == list(GM[pre + "pos" + suffix])
            and (st[3] == 0 or abs(st[4] - float(GM[pre + "gauss" + suffix])) <= 1e-14 * max(1.0, abs(st[4]))))


@pytest.mark.parametrize("fam", FAMILIES)
@pytest.mark.parametrize("tag,kw", [("rw", dict(delta=0.8, enka_scaling=True)), ("pcn", dict(update="pCN", beta=0.05))])
def test_emulator_mh_chain_zero_is_the_oracle_chain(fam, tag, kw):
    emu, enka, prior, mc = _chain_setup(fam)
    pre = "%s/chain/%s/" % (fam, tag)
    np.random.seed(13)
    mc.emulator_mh(emu, 150, prior, enka, **kw)
    want = GM[pre + "samples"]
    assert mc.samples.shape == want.shape
    assert np.abs(mc.samples - want).max() <= 1e-10 * np.abs(want).max(), (fam, tag)
    assert abs(mc.accept - float(GM[pre + "accept"])) < 1e-12 and _state_equal(pre)
    if tag == "rw":
        mc.emulator_mh(emu, 40, prior, enka, **kw)
        want2 = GM[pre + "samples_resumed"]
        assert mc.samples.shape == want2.shape
        assert np.abs(mc.samples - want2).max() <= 1e-10 * np.abs(want2).max()
        assert abs(mc.accept - float(GM[pre + "accept_resumed"])) < 1e-12 and _state_equal(pre, "2")


def test_changing_the_family_clears_the_conditioned_state():
    """ces_gp_set_kernel after ces_gp_condition: ces_gp_predict and ces_gp_mh refuse until the emulator is conditioned
    again, and the new conditioning predicts with the new family."""
    import torch

    name = "p2_n100_k10"
    emu = _emulator(name, "SquaredExponential")
    theta = GM["Matern52/%s/theta" % name]
    emu.theta = theta
    U = GM[name + "/U"][:, :33]
    se_mean, _ = emu.predict(U)
    lib, h = emu._lib, emu._h
    assert lib.ces_gp_set_kernel(h, _lib.GP_KERNELS["Matern52"]) == _lib.CES_OK
    for kind in (-1, 4):
        assert lib.ces_gp_set_kernel(h, kind) == _lib.CES_ERR_INVALID
    Ud = torch.from_numpy(np.ascontiguousarray(U)).cuda()
    mean = torch.empty((emu.k, 33), dtype=torch.float64, device="cuda")
    var = torch.empty_like(mean)
    st = lib.ces_gp_predict(h, ctypes.c_void_p(Ud.data_ptr()), Ud.stride(0), 33, ctypes.c_void_p(mean.data_ptr()),
                            mean.stride(0), ctypes.c_void_p(var.data_ptr()), var.stride(0))
    assert st == _lib.CES_ERR_STATE and b"ces_gp_condition" in lib.ces_last_error()
    z = np.zeros(emu.p)
    samples, acc = np.empty(emu.p * 2), np.zeros(1, dtype=np.int32)
    st = lib.ces_gp_mh(h, _lib.host_ptr(np.zeros(emu.k)), 1, None, None, _lib.host_ptr(np.eye(emu.p)), 1, 0.5, 1, 1,
                       _lib.host_ptr(z), _lib.host_ptr(z), None, None, 0, _lib.host_ptr(samples), acc.ctypes.data)
    assert st == _lib.CES_ERR_STATE
    th = np.ascontiguousarray(theta)
    _lib.check(lib.ces_gp_condition(h, _lib.host_ptr(th), emu.jitter))
    _lib.check(lib.ces_gp_predict(h, ctypes.c_void_p(Ud.data_ptr()), Ud.stride(0), 33, ctypes.c_void_p(mean.data_ptr()),
                                  mean.stride(0), ctypes.c_void_p(var.data_ptr()), var.stride(0)))
    torch.cuda.current_stream().synchronize()
    Y = GM[name + "/G"] - GM[name + "/G"].mean(axis=1, keepdims=True)
    scale = np.abs(Y).max(axis=1)[:, None]
    assert np.all(np.abs(mean.cpu().numpy() - GM["Matern52/%s/mean" % name][:, :33]) <= 1e-10 * scale)
    assert not np.allclose(se_mean, GM["Matern52/%s/mean" % name][:, :33], rtol=0, atol=1e-6)


def test_emulator_rejects_an_unknown_kernel():
    with pytest.raises(ValueError, match="Matern72"):
        GPEmulator(U=GM["p1_n37_k1/X"], G=GM["p1_n37_k1/G"], Gamma=np.eye(1), kernel="Matern72")
    emu = GPEmulator(U=GM["p1_n37_k1/X"], G=GM["p1_n37_k1/G"], Gamma=np.eye(1))
    assert emu.kernel == "SquaredExponential"
    with pytest.raises(AttributeError):
        emu.kernel = "Matern52"


def _split_rhat(chains):
    """Split-R^ (Gelman et al., BDA3 11.4) per coordinate of chains (n_chains, p, n)."""
    n = chains.shape[2] // 2
    halves = np.concatenate([chains[:, :, :n], chains[:, :, n:2 * n]], axis=0)
    W = halves.var(axis=2, ddof=1).mean(axis=0)
    B = n * halves.mean(axis=2).var(axis=0, ddof=1)
    return np.sqrt(((n - 1) / n * W + B / n) / W)


def test_darcy_example_with_matern52_against_the_true_model():
    """examples/darcy_ces.py --kernel Matern52 at the reduced size of the SE example's test (tests/test_gpu_darcy_mh.py),
    held to the same bounds: split-R^ < 1.1 per mode for the true-model chains, their acceptance in (0.05, 0.9), and the
    emulator's posterior mean within 0.2 true-posterior standard deviations of theirs on every mode."""
    import importlib.util

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("darcy_ces_example", os.path.join(root, "examples", "darcy_ces.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = mod.main(["--n-mcmc", "3000", "--chains", "64", "--kernel", "Matern52"])
    assert out["kernel"] == "Matern52" and out["emulator"].kernel == "Matern52"
    burn = out["burn"]
    rhat = _split_rhat(out["model_mcmc"].samples_chains[:, :, burn:])
    gap = np.abs(out["emulator_mean"] - out["model_mean"]) / out["model_sd"]
    print("split-R^", np.round(rhat, 3), "emulator gap / sd", np.round(gap, 3), "accept", out["model_accept"])
    assert np.all(rhat < 1.1), rhat
    assert 0.05 < out["model_accept"] < 0.9
    assert np.all(gap < 0.2), gap
