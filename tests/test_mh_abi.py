"""ces_mcmc_model_mh and ces_gp_mh refuse bad arguments with the limits every sampler shares (n_mcmc < 2^31 - 1,
n_chains <= 2^24, mt_gauss with mt_state), before any device work, so on a machine without a GPU too."""
import numpy as np

from ces_b200 import _lib

V, MT, GAUSS = np.zeros(64), np.zeros(626, dtype=np.uint32), np.zeros(1)
ACC = np.zeros(4, dtype=np.int32)
OK = dict(mu=V.ctypes.data, Pinv=V.ctypes.data, scales=V.ctypes.data, pcn=0, beta=0.5, n_mcmc=10, n_chains=2,
          start=V.ctypes.data, phi=V.ctypes.data, mt=MT.ctypes.data, gauss=GAUSS.ctypes.data, seed=0,
          samples=V.ctypes.data, accepted=ACC.ctypes.data)
TAIL = ("mu", "Pinv", "scales", "pcn", "beta", "n_mcmc", "n_chains", "start", "phi", "mt", "gauss", "seed", "samples",
        "accepted")
SHARED_LIMITS = (dict(gauss=None), dict(n_mcmc=2 ** 31), dict(n_mcmc=0), dict(n_chains=(1 << 24) + 1), dict(n_chains=0))


def _mcmc(**kw):
    """The banana map (p = k = 2, parameters on the host): no device pointer is needed."""
    lib = _lib.load()
    a = dict(OK, **kw)
    return lib.ces_mcmc_model_mh(None, _lib.MAPS["banana"], 2, 2, None, 0, None, V.ctypes.data, V.ctypes.data,
                                 V.ctypes.data, *(a[n] for n in TAIL))


def _gp(model=None, **kw):
    lib = _lib.load()
    a = dict(OK, **kw)
    return lib.ces_gp_mh(model, V.ctypes.data, 1, *(a[n] for n in TAIL))


def test_model_mh_abi_refuses_the_shared_limits_without_a_gpu():
    lib = _lib.load()
    for bad in SHARED_LIMITS:
        assert _mcmc(**bad) == _lib.CES_ERR_INVALID, bad
        assert b"ces_mcmc_model_mh" in lib.ces_last_error() and b"n_mcmc" in lib.ces_last_error(), bad


def test_gp_mh_abi_checks_the_shared_limits_before_the_model():
    lib = _lib.load()
    assert _gp() == _lib.CES_ERR_INVALID
    assert b"ces_gp_mh: null model" in lib.ces_last_error()
    for bad in SHARED_LIMITS:
        assert _gp(**bad) == _lib.CES_ERR_INVALID, bad
        assert b"ces_gp_mh" in lib.ces_last_error() and b"n_mcmc" in lib.ces_last_error(), bad
