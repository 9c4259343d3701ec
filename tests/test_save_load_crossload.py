"""enka.save / enka.load against the REAL reference's (ces/calibrate.py:170-237): files written by one are read by the
other, in every mode (last, all, online).  Host-side code only; the cross-loads need a checkout of the reference
(oracle/reference_loader.py)."""
import os

import numpy as np
import pytest

from ces_b200 import calibrate
from oracle import reference_loader as rl

needs_reference = pytest.mark.skipif(not rl.available(), reason="needs a checkout of the reference (CES_REFERENCE_ROOT)")


def _filled(cls, d=3, k=5, J=11, T=4, seed=0):
    rs = np.random.RandomState(seed)
    obj = cls(d, k, J)
    obj.Uall = rs.normal(size=(T + 1, d, J))
    obj.Gall = rs.normal(size=(T + 1, k, J))
    obj.Ustar, obj.Gstar = obj.Uall[-1], obj.Gall[-1]
    obj.metrics = {key: list(rs.uniform(size=T)) for key in ("self-bias", "self-bias-data", "bias-data", "bias", "t")}
    return obj


@needs_reference
@pytest.mark.parametrize("writer", ["reference", "ours"])
def test_last_and_all_modes_cross_load(tmp_path, writer):
    ref_cls, our_cls = rl.load_calibrate().sampling, calibrate.sampling
    src = _filled(ref_cls if writer == "reference" else our_cls)
    path = str(tmp_path) + "/"
    src.save(path=path, file="run/", all=True)
    assert sorted(os.listdir(path + "run")) == ["Gensemble.npy", "Gensemble_path.npy", "ensemble.npy", "ensemble_path.npy", "metrics.pkl"]
    dst = (our_cls if writer == "reference" else ref_cls)(3, 5, 11)
    assert dst.load(path=path, eks_dir="run/") in (True, None)       # the reference's load returns None on success
    assert np.array_equal(dst.Uall, src.Uall) and np.array_equal(dst.Gall, src.Gall) and dst.metrics == src.metrics
    assert np.array_equal(np.load(path + "run/ensemble.npy"), src.Ustar)
    assert np.array_equal(np.load(path + "run/Gensemble.npy"), src.Gstar)


@needs_reference
@pytest.mark.parametrize("writer", ["reference", "ours"])
def test_online_mode_cross_load(tmp_path, writer):
    ref_cls, our_cls = rl.load_calibrate().sampling, calibrate.sampling
    src = _filled(ref_cls if writer == "reference" else our_cls)
    full_U, full_G = src.Uall, src.Gall
    path = str(tmp_path) + "/"
    for i in range(4):                                               # what run(save_online=True) does per iteration
        src.Uall, src.Gall = list(full_U[:i + 1]), list(full_G[:i + 1])
        src.save(path=path, file="online/", online=True, counter=i)
    names = sorted(os.listdir(path + "online"))
    assert names == sorted(["ensemble_%04d.npy" % i for i in range(4)] + ["Gensemble_%04d.npy" % i for i in range(4)] + ["metrics.pkl"])
    for flag in (False, True):
        dst = (our_cls if writer == "reference" else ref_cls)(3, 5, 11)
        dst.load(path=path, eks_dir="online/", ix_ensemble=True, flag_metrics=flag)
        assert np.array_equal(np.asarray(dst.Uall), full_U[:4]) and np.array_equal(np.asarray(dst.Gall), full_G[:4])
        assert np.array_equal(dst.Ustar, full_U[3]) and dst.J == 11 and dst.metrics == src.metrics


def test_missing_files_behave_like_the_reference(tmp_path, capsys):
    """The reference's load without files, as recorded from it (and compared with it again when a checkout is present):
    an empty directory prints "Metrics object not found" and returns False, a missing one raises FileNotFoundError."""
    objs = [calibrate.sampling(3, 5, 11)] + ([rl.load_calibrate().sampling(3, 5, 11)] if rl.available() else [])
    os.makedirs(str(tmp_path) + "/empty")
    for obj in objs:
        assert obj.load(path=str(tmp_path) + "/", eks_dir="empty/") is False
        with pytest.raises(FileNotFoundError):
            obj.load(path=str(tmp_path) + "/", eks_dir="nothing/")       # os.listdir of a missing directory (:203)
    out = capsys.readouterr().out
    assert out.count("Metrics object not found") == len(objs)
