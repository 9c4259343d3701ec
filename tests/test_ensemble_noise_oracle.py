"""The ensemble form of the noise (noise='ensemble', DESIGN.md section 4g) on the CPU: the layout of its restated Philox
stream and the algebra of the restated step (oracle/ensemble_noise_oracle.py), the algebra of the oracle step, and the C ABI's refusals of bad settings
before any device work."""
import ctypes

import numpy as np
import pytest

from oracle import eks_oracle as eo, ensemble_noise_oracle as eno, philox_oracle as po

SEEDS = (0, 11, 2 ** 40 + 3)


# ---------------------------------------------------------------------------------------------- stream layout
@pytest.mark.parametrize("seed", SEEDS)
def test_ensemble_stream_is_invariant_to_row_and_column_sharding(seed):
    step, rows, cols = 2 ** 31 + 5, 37, 53
    full = eno.ensemble_noise(seed, step, rows, cols)
    assert full.shape == (rows, cols) and np.all(np.isfinite(full))
    for r0, r1 in ((0, 1), (1, 20), (17, 37), (36, 37)):
        for c0, c1 in ((0, 1), (1, 2), (3, 30), (29, 53), (52, 53)):
            part = eno.ensemble_noise(seed, step, r1 - r0, c1 - c0, r0, c0)
            assert np.array_equal(part, full[r0:r1, c0:c1]), (r0, r1, c0, c1)
    # far offsets: a block drawn at once equals its single rows and columns drawn one by one
    for r0, c0 in ((2 ** 20 + 1, 2 ** 32), (5, 2 ** 32 + 1), (2 ** 31 - 1, 2 ** 33 - 3)):
        block = eno.ensemble_noise(seed, step, 3, 6, r0, c0)
        for i in range(3):
            for j in range(6):
                assert block[i, j] == eno.ensemble_noise(seed, step, 1, 1, r0 + i, c0 + j)[0, 0], (r0, c0, i, j)


def test_ensemble_stream_layout_and_distribution():
    seed, step = 7, 3
    x = eno.ensemble_noise(seed, step, 4, 6)
    # element (s, j): counter (j >> 1, TAG_ENS, s, step); even j the cosine, odd j the sine of one Box-Muller pair
    for s in range(4):
        for j in range(6):
            cs, sn = po.normal_pair(po.philox4x32_10((j >> 1, eno.TAG_ENS, s, step), po._key(seed)))
            assert x[s, j] == (cs if j % 2 == 0 else sn)
    # (seed, step) select different draws; the stream is N(0, 1)
    assert not np.array_equal(x, eno.ensemble_noise(seed, step + 1, 4, 6))
    assert not np.array_equal(x, eno.ensemble_noise(seed + 1, step, 4, 6))
    big = eno.ensemble_noise(seed, step, 256, 256)
    assert abs(big.mean()) < 5 / 256 and abs(big.var() - 1) < 5 * np.sqrt(2) / 256


@pytest.mark.parametrize("seed", SEEDS)
def test_ensemble_stream_is_disjoint_from_fill_normal(seed):
    """Counter word 1 is TAG_ENS here and the high half of the pair index in fill_normal: at the same (seed, step) the two
    streams share no Philox block, so no value of one reappears in the other."""
    step, n = 9, 64
    a = eno.ensemble_noise(seed, step, n, n)
    b = po.fill_normal(seed, step, n, n)
    assert not np.isin(a, b).any()
    assert np.abs(a - b).min() > 0


# ---------------------------------------------------------------------------------------------- oracle algebra
def _problem(p, k, J, seed=4):
    pr = eo.linear_gaussian_problem(p, k, J, seed=seed)
    return pr


@pytest.mark.parametrize("rule", ["eks", "aldi", "aldi_constant"])
def test_oracle_with_zero_xi_is_the_deterministic_part(rule):
    p, k, J = 6, 9, 20
    pr = _problem(p, k, J)
    args = (rule, pr["y"], pr["U0"], pr["G"], pr["Gamma"], pr["mu"], pr["Sigma0"], pr["ustar"])
    ens = eno.step(*args, np.zeros((J, J)))
    chol = eo.step(*args, np.zeros((p, J)))
    assert np.array_equal(ens["Uk"], chol["Uk"]) and ens["hk"] == chol["hk"]
    # and with noise: the ensemble form is exactly sqrt(2h / n_C) (U - ubar) xi on top of it
    xi = np.random.RandomState(1).normal(size=(J, J))
    n_C = J if rule == "eks" else J - 1
    got = eno.step(*args, xi)
    Ut = pr["U0"] - pr["U0"].mean(axis=1)[:, None]
    assert np.allclose(got["Uk"] - ens["Uk"], np.sqrt(2 * got["hk"] / n_C) * (Ut @ xi), rtol=0, atol=1e-12)


@pytest.mark.parametrize("rule", ["eks", "aldi", "aldi_constant"])
def test_oracle_noise_stays_in_the_ensemble_span(rule):
    """J <= p: C^uu has rank <= J - 1, the Cholesky noise leaves span(U - ubar), the ensemble noise does not."""
    p, k, J = 40, 30, 12
    pr = _problem(p, k, J)
    args = (rule, pr["y"], pr["U0"], pr["G"], pr["Gamma"], pr["mu"], pr["Sigma0"], pr["ustar"])
    base = eno.step(*args, np.zeros((J, J)))["Uk"]
    Ut = pr["U0"] - pr["U0"].mean(axis=1)[:, None]
    Q, _ = np.linalg.qr(Ut)
    Q = Q[:, :J - 1]                                   # U - ubar has rank J - 1
    for seed in range(3):
        xi = eno.ensemble_noise(seed, 0, J, J)
        delta = eno.step(*args, xi)["Uk"] - base
        resid = delta - Q @ (Q.T @ delta)
        # delta = U_next(xi) - U_next(0) carries the rounding of U_next itself: 1e-13 of U_next, 1e-12 of delta
        assert np.linalg.norm(resid) <= 1e-13 * np.linalg.norm(base), np.linalg.norm(resid) / np.linalg.norm(base)
        assert np.linalg.norm(resid) <= 1e-12 * np.linalg.norm(delta), np.linalg.norm(resid) / np.linalg.norm(delta)
    chol_delta = eo.step(*args, pr["xi"][:, :J])["Uk"] - eo.step(*args, np.zeros((p, J)))["Uk"]
    resid = chol_delta - Q @ (Q.T @ chol_delta)
    assert np.linalg.norm(resid) > 1e-6 * np.linalg.norm(chol_delta)


def test_oracle_rejects_a_p_by_J_xi_and_leaves_eki_alone():
    pr = _problem(3, 4, 5)
    args = (pr["y"], pr["U0"], pr["G"], pr["Gamma"], pr["mu"], pr["Sigma0"], pr["ustar"])
    with pytest.raises(ValueError):
        eno.step("aldi", *args, pr["xi"])
    assert np.array_equal(eno.step("eki", *args, None)["Uk"], eo.step("eki", *args, None)["Uk"])


# ---------------------------------------------------------------------------------------------- ABI refusals
def test_set_noise_and_fill_refuse_bad_arguments_without_touching_the_gpu():
    from ces_b200 import _lib

    lib = _lib.load()
    # unknown kinds, whatever the handle
    for kind in (-1, 2, 7):
        assert lib.ces_set_noise(None, kind, 0, 0, None, 0) == _lib.CES_ERR_INVALID
        assert b"unknown noise kind" in lib.ces_last_error()
    # a NULL handle, in both modes
    for kind in (0, 1):
        assert lib.ces_set_noise(None, kind, 0, 0, None, 0) == _lib.CES_ERR_INVALID
        assert b"null handle" in lib.ces_last_error()
    # an explicit xi needs a 16-byte base and an even leading dimension
    buf = (ctypes.c_double * 64)()
    base = ctypes.addressof(buf)
    aligned = base + (-base) % 16
    assert lib.ces_set_noise(None, 1, 0, 0, ctypes.c_void_p(aligned + 8), 8) == _lib.CES_ERR_ALIGN
    assert lib.ces_set_noise(None, 1, 0, 0, ctypes.c_void_p(aligned), 7) == _lib.CES_ERR_ALIGN
    assert lib.ces_set_noise(None, 1, 0, 0, ctypes.c_void_p(aligned), 0) == _lib.CES_ERR_ALIGN
    # the fill: NULL output, ld below the width, negative sizes or offsets
    assert lib.ces_fill_ensemble_noise(None, 0, 0, None, 4, 2, 2, 0, 0) == _lib.CES_ERR_INVALID
    for ld, rows, cols, r0, c0 in ((1, 2, 2, 0, 0), (4, -1, 2, 0, 0), (4, 2, -1, 0, 0), (4, 2, 2, -1, 0), (4, 2, 2, 0, -3)):
        assert lib.ces_fill_ensemble_noise(None, 0, 0, ctypes.c_void_p(aligned), ld, rows, cols, r0, c0) == \
            _lib.CES_ERR_INVALID, (ld, rows, cols, r0, c0)
    with pytest.raises(ValueError):
        _lib.check(lib.ces_set_noise(None, 5, 0, 0, None, 0))


def test_sampling_refuses_bad_noise_settings_before_any_device_work():
    """The Python checks run before the engine is created, so they hold without a GPU."""
    from ces_b200 import calibrate

    p, k, J = 3, 4, 6
    pr = _problem(p, k, J)
    s = calibrate.sampling(p, k, J)
    s.mu, s.sigma, s.ustar = pr["mu"], pr["Sigma0"], pr["ustar"]
    upd = lambda **kw: s.eks_update_aldi(pr["y"], pr["U0"], pr["G"], pr["Gamma"], 0, **kw)
    with pytest.raises(ValueError, match="noise"):
        upd(noise="spherical")
    with pytest.raises(ValueError, match="factored"):
        upd(noise="ensemble", formulation="factored")
    for shape in ((p, J), (J, J + 1), (J,), (J - 1, J)):
        with pytest.raises(ValueError, match="xi"):
            upd(noise="ensemble", xi=np.zeros(shape))
    s.noise = "gaussian"
    with pytest.raises(ValueError, match="noise"):
        s.run(pr["y"], pr["U0"], type("Model", (), {"type": "map"})(), pr["Gamma"], None, update="eks")
    assert s._engine is None
