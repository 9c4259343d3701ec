"""ces_darcy_mh (MCMC.model_mh on the Darcy models) refuses bad arguments before any device work, so on a machine without a
GPU too."""
import numpy as np

from ces_b200 import _lib


def test_darcy_mh_abi_rejects_bad_arguments_without_a_gpu():
    lib = _lib.load()
    v, mt, g = np.zeros(64), np.zeros(626, dtype=np.uint32), np.zeros(1)
    acc = np.zeros(4, dtype=np.int32)
    ok = dict(y=v.ctypes.data, Ginv2=v.ctypes.data, mu=v.ctypes.data, Pinv=v.ctypes.data, scales=v.ctypes.data, pcn=0,
              beta=0.5, n_mcmc=10, n_chains=2, start=v.ctypes.data, phi=v.ctypes.data, mt=mt.ctypes.data, gauss=g.ctypes.data,
              seed=0, samples=v.ctypes.data, accepted=acc.ctypes.data)

    def call(model=None, **kw):
        a = dict(ok, **kw)
        return lib.ces_darcy_mh(model, 1e-10, 0, a["y"], a["Ginv2"], a["mu"], a["Pinv"], a["scales"], a["pcn"], a["beta"],
                                a["n_mcmc"], a["n_chains"], a["start"], a["phi"], a["mt"], a["gauss"], a["seed"], a["samples"],
                                a["accepted"])

    assert call() == _lib.CES_ERR_INVALID                                   # no model
    for bad in (dict(n_mcmc=0), dict(n_mcmc=-3), dict(n_chains=0), dict(n_chains=(1 << 24) + 1), dict(y=None),
                dict(Ginv2=None), dict(scales=None), dict(start=None), dict(phi=None), dict(samples=None), dict(accepted=None),
                dict(mu=None), dict(Pinv=None), dict(gauss=None)):
        assert call(**bad) == _lib.CES_ERR_INVALID, bad
        assert b"ces_darcy_mh" in lib.ces_last_error()
    # pCN needs no prior mean / precision, numpy's stream is optional: still refused here only for the missing model
    assert call(pcn=1, mu=None, Pinv=None, mt=None, gauss=None) == _lib.CES_ERR_INVALID
    assert b"null model" in lib.ces_last_error()
