"""Host-side logic of the drop-in classes that needs no GPU: sharding arithmetic, time bookkeeping,
persistence format, loud failure without CUDA."""
import os
import pickle

import numpy as np
import pytest
import torch

from ces_b200 import calibrate
from ces_b200.engine import Engine, shard_range, shard_width

no_cuda = not torch.cuda.is_available()


@pytest.mark.parametrize("J,n", [(100, 1), (100, 8), (17, 2), (17, 4), (5, 8), (65536, 8)])
def test_shards_partition_the_ensemble(J, n):
    w = shard_width(J, n)
    assert w * n >= J
    cols = []
    for r in range(n):
        lo, hi = shard_range(J, r, n)
        assert 0 <= hi - lo <= w
        cols.extend(range(lo, hi))
    assert cols == list(range(J))


def test_time_bookkeeping_matches_reference_rule():
    s = calibrate.sampling(2, 3, 10)
    s._ensure_metrics()
    assert set(s.metrics) == {"self-bias", "self-bias-data", "bias-data", "bias", "t"} and s.radspec == []
    s._advance_time(0.5)
    s._advance_time(0.25)
    assert s.metrics["t"] == [0.5, 0.75]


def test_time_step_kwargs_map_to_step_options():
    """time_step semantics of ces/calibrate.py:247-260 (hk) and :439-441 / :470-473 (re-solve of D)."""
    s = calibrate.sampling(2, 3, 10)
    s.T = 30
    with pytest.raises(NotImplementedError):
        s._step_options("aldi", {"time_step": "adaptive"})         # undefined in the reference (:255)
    assert s._step_options("aldi", {"time_step": "spectral"}) == (None, "spectral")
    assert s._step_options("aldi_constant", {"time_step": "spectral"}) == (None, None)
    with pytest.raises(ValueError):
        s._step_options("aldi", {"time_step": "bogus"})
    assert s._step_options("aldi", {}) == (None, None)
    assert s._step_options("aldi", {"time_step": "constant"}) == (1. / 15, "always")
    assert s._step_options("eks", {"time_step": "constant", "delta_t": 0.5}) == (0.5, "always")
    assert s._step_options("aldi_constant", {"time_step": "constant"}) == (None, None)
    s._ensure_metrics()
    assert s._step_options("aldi", {"time_step": "mix"}) == (None, (0.0, 1.0))        # first step: default rule
    s.metrics["t"] = [0.5, 2.0]
    assert s._step_options("aldi", {"time_step": "mix"}) == (None, (2.0, 1.0))        # before spin-up (4.0)
    assert s._step_options("eks", {"time_step": "mix"}) == (None, None)               # eks never re-solves for mix
    s.metrics["t"] = [0.5, 4.5]
    assert s._step_options("aldi", {"time_step": "mix", "delta_t": 0.1}) == (0.1, (4.5, 1.0))


def test_save_load_round_trip(tmp_path):
    """File names and contents of enka.save / enka.load (ces/calibrate.py:170-237)."""
    s = calibrate.sampling(2, 3, 4)
    rng = np.random.default_rng(0)
    s.Uall = rng.standard_normal((3, 2, 4))
    s.Gall = rng.standard_normal((3, 3, 4))
    s.Ustar, s.Gstar = s.Uall[-1], s.Gall[-1]
    s.metrics = {"self-bias": [1.0, 2.0], "bias": [3.0, 4.0], "self-bias-data": [5.0, 6.0], "bias-data": [7.0, 8.0],
                 "t": [0.1, 0.3]}
    path = str(tmp_path) + "/"
    s.save(path=path, file="ces/", all=True)
    assert sorted(os.listdir(path + "ces/")) == ["Gensemble.npy", "Gensemble_path.npy", "ensemble.npy",
                                                 "ensemble_path.npy", "metrics.pkl"]
    assert pickle.load(open(path + "ces/metrics.pkl", "rb")) == s.metrics
    r = calibrate.sampling(2, 3, 99)
    assert r.load(path=path, eks_dir="ces/") is True
    assert np.array_equal(r.Uall, s.Uall) and np.array_equal(r.Gall, s.Gall) and r.metrics == s.metrics
    for i in range(3):
        s.Uall_i = None
        s.save(path=path, file="online/", online=True, counter=i)
    r2 = calibrate.sampling(2, 3, 99)
    assert r2.load(path=path, eks_dir="online/", ix_ensemble=True) is True
    assert r2.J == 4 and r2.Uall.shape == (3, 2, 4)
    assert calibrate.sampling(2, 3, 4).load(path=path, eks_dir="missing/") is False if os.path.isdir(path + "missing/") else True


def test_model_type_is_required_like_the_reference():
    s = calibrate.sampling(2, 3, 4)

    class NoType(object):
        pass

    with pytest.raises(AttributeError):
        s.run(np.zeros(3), np.zeros((2, 4)), NoType(), np.eye(3), None)


@pytest.mark.skipif(not no_cuda, reason="checks the no-GPU failure mode")
def test_product_fails_loudly_without_cuda():
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        Engine(2, 3, 10)
    s = calibrate.sampling(2, 3, 10)
    s.mu, s.sigma, s.ustar = np.zeros((2, 1)), np.eye(2), np.zeros((2, 1))
    with pytest.raises(RuntimeError):
        s.eks_update_aldi(np.zeros(3), np.zeros((2, 10)), np.zeros((3, 10)), np.eye(3), 0)


def test_product_never_imports_the_oracle():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for dirpath, _, files in os.walk(os.path.join(root, "ces_b200")):
        for name in files:
            if name.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, name)).read()
                assert "import oracle" not in text and "from oracle" not in text, name


class _CountingEngine(object):
    """Stand-in for the device engine: counts how often the problem data is (re-)uploaded."""

    def __init__(self):
        self.uploads = 0

    def set_problem(self, *arrays):
        self.uploads += 1
        self.last = [np.array(a, copy=True) for a in arrays]


def test_problem_cache_is_keyed_on_content():
    """The device copy of (y_obs, Gamma, sigma, mu, ustar) and its factorisations are reused between calls only while the
    CONTENT of the five arrays is unchanged: in-place edits that a strided checksum would miss (a permutation of y_obs, one
    entry of a large Gamma) trigger a re-upload; the deferred check of large arrays (run while the GPU step executes) reports
    the edit afterwards so the caller can repeat the step."""
    k, p = 400, 3                                   # Gamma: 1.28 MB > the 1 MB threshold of the deferred check
    rng = np.random.default_rng(0)
    y, Gamma = rng.standard_normal(k), np.eye(k) * 0.01
    s = calibrate.sampling(p, k, 10)
    s.mu, s.sigma, s.ustar = np.zeros((p, 1)), np.eye(p), np.zeros((p, 1))
    eng = _CountingEngine()
    assert s._sync_problem(eng, y, Gamma) is None and eng.uploads == 1
    assert s._sync_problem(eng, y, Gamma) is None and eng.uploads == 1            # unchanged: no upload
    y[[0, 1]] = y[[1, 0]]                                                         # a permutation keeps every plain sum
    s._sync_problem(eng, y, Gamma)
    assert eng.uploads == 2 and np.array_equal(eng.last[0], y)
    Gamma[123, 77] = Gamma[77, 123] = 1e-4                                        # one entry of a large matrix
    s._sync_problem(eng, y, Gamma)
    assert eng.uploads == 3 and eng.last[1][123, 77] == 1e-4
    s.mu[1, 0] = 0.25                                                             # small arrays: always checked at once
    s._sync_problem(eng, y, Gamma)
    assert eng.uploads == 4
    # deferred mode (the eks_update* path): identical buffers -> the large digest runs in the background
    stale = s._sync_problem(eng, y, Gamma, defer_large=True)
    assert eng.uploads == 4 and callable(stale) and stale() is False and eng.uploads == 4
    Gamma[5, 5] = 0.02                                                            # edited in place, same object
    stale = s._sync_problem(eng, y, Gamma, defer_large=True)
    assert eng.uploads == 4                                                       # not seen yet: the step would run on stale data ...
    assert stale() is True and eng.uploads == 5 and eng.last[1][5, 5] == 0.02     # ... and is reported: the caller repeats it
    assert s._sync_problem(eng, y, Gamma, defer_large=True)() is False
    # a new but equal array (different object, same bytes) does not re-upload
    assert s._sync_problem(eng, y.copy(), Gamma.copy()) is None and eng.uploads == 5


def test_reference_arm_of_bench_runs_on_the_host(tmp_path):
    """bench.py --impl reference needs no GPU: it times the real reference (or the staged copy / the port) on the host and
    prints one JSON line that names the ensemble size it ran."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, OMP_NUM_THREADS="1")                                   # what torch.distributed.run exports
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload", "small", "--steps", "2",
                          "--warmup", "0"], capture_output=True, text=True, timeout=300, cwd=root, env=env)
    assert out.returncode == 0, out.stderr[-1500:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["value"] > 0 and d["config"]["J_sample"] == d["cpu_baseline"]["J_sample"] == 1024
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] == (os.cpu_count() or 1)
    assert d["e2e"] == {"value": d["value"], "unit": "particle-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["steps"] == 2 and d["warmup"] == 0 and d["gpu_launches"] == 0


def test_bench_dump_outputs_keeps_one_seeded_column_sample_within_the_budget(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float64 files, numbers as one-element arrays, and when the outputs exceed the budget the
    same seeded particle columns of every (rows, particles) array, identical from call to call."""
    import importlib.util

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    monkeypatch.setattr(bench, "DUMP_BYTES", 200000)
    rng = np.random.default_rng(3)
    U, G = rng.standard_normal((24, 1000)), rng.standard_normal((7, 1000)).astype(np.float32)
    for name in ("a", "b"):
        bench.dump_outputs(str(tmp_path / name), {"U_next": U, "G": G, "hk": 0.25, "t": [0.5, 0.75]})
    files = sorted(os.listdir(str(tmp_path / "a")))
    assert files == ["G.npy", "U_next.npy", "hk.npy", "t.npy"]
    assert sum(os.path.getsize(str(tmp_path / "a" / f)) for f in files) <= 200000
    a = {f[:-4]: np.load(str(tmp_path / "a" / f)) for f in files}
    assert all(v.dtype == np.float64 for v in a.values()) and a["hk"].tolist() == [0.25] and a["t"].tolist() == [0.5, 0.75]
    ncols = a["U_next"].shape[1]
    assert 0 < ncols < 1000 and a["G"].shape == (7, ncols)
    cols = [int(np.flatnonzero((U == a["U_next"][:, j][:, None]).all(axis=0))[0]) for j in range(ncols)]
    assert cols == sorted(set(cols)) and np.array_equal(a["G"], G[:, cols].astype(np.float64))
    for f in files:
        assert np.array_equal(a[f[:-4]], np.load(str(tmp_path / "b" / f)))


def test_bench_rejects_a_step_count_below_one():
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                         timeout=120, cwd=root)
    assert out.returncode == 2 and "--steps" in out.stderr and out.stdout == ""


def test_bench_flop_models_agree_with_the_oracle():
    """bench.py carries its own copies of the flop models (the GPU arm must not import oracle/ for them): W_step of SURVEY.md
    section 8(d) and the reference-as-written model of BASELINE.md section 3 stay identical to the oracle's."""
    import importlib.util

    from oracle import eks_oracle as eo

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    for (J, d, k) in [(100, 2, 10), (1024, 64, 50), (16384, 1024, 4096), (65536, 1024, 4096)]:
        for dense in (False, True):
            assert bench.algorithmic_flops(J, d, k, dense) == eo.algorithmic_flops(J, d, k, dense)
        assert bench.reference_flops(J, d, k) == eo.reference_flops(J, d, k)
    assert abs(bench.algorithmic_flops(65536, 1024, 4096) - 4.44e13) < 0.02e13          # the target's W_step (DESIGN section 5)
    # the workloads bench.py names are BASELINE.json's
    assert bench.WORKLOADS["target"] == (1024, 4096, 65536) and bench.WORKLOADS["cfg3"] == (1024, 4096, 16384)
    assert bench.DARCY_WORKLOADS["cfg2"][:4] == (64, 64, 50, 1024) and bench.DARCY_WORKLOADS["cfg4"][:4] == (128, 256, 50, 65536)
    pr = bench.cfg1_problem()
    assert pr["U0"].shape == (2, 100) and pr["T"] == 1000 and pr["A"].shape == (10, 2)
