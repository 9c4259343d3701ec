"""The single-GPU schedule that forms only the lower trapezoid of the symmetric part of D (csrc/api.cu symmetric_loops):
the exact contract of its GEMM mode (GEMM_C_LOWER_TRAP with a row term and the mirrored sum-of-squares partials), steps
whose rank-one term dominates D, the constant time-step re-solve over several panels with dense Gamma, and the flops the
D profile reports."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from ces_b200 import calibrate  # noqa: E402
from ces_b200.engine import Engine  # noqa: E402
from oracle import eks_oracle as eo  # noqa: E402
from test_gpu_gemm_contract import A_KM, B_KN, NAN, SENTINEL, Buf, _ints, gemm  # noqa: E402
from test_symmetric_d_schedule import trap_tiles  # noqa: E402

TRAP = 32
TOL = 1e-10


def _rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def test_lower_trapezoid_mode_is_exact():
    """D-shaped launches (A_KM x B_KN, M > N, ragged M / N / K): only the tiles tn <= tm are written, with
    alpha (AB - r 1^T) (+ beta C); the upper tiles keep the sentinel bits; one partial per launched tile in the order of
    the compact enumeration, equal to sum (C + alpha r_m)^2 plus, below the diagonal, sum (C + alpha r_n)^2.  Also in two
    contraction chunks (beta = 1, the row term and the partials on the last chunk only) and on a 2-CTA serpentine walk.
    Entries in {-2..2}: every value is exact."""
    rng = np.random.default_rng(12)
    failures = []
    for M, N, K in [(300, 257, 81), (515, 129, 40), (129, 129, 17), (700, 300, 33), (2100, 300, 20)]:
        tiles = trap_tiles(M, N, 128)
        tm = np.arange(M)[:, None] // 128
        tn = np.arange(N)[None, :] // 128
        comp = tn <= tm
        for mode in ("one", "chunks", "serpentine"):
            A = _ints(rng, (M, K), -2, 2)
            Bm = _ints(rng, (K, N), -2, 2)
            r = _ints(rng, (M,), -3, 3)
            C0 = _ints(rng, (M, N), -2, 2)
            Ab, Bb = Buf(np.ascontiguousarray(A.T)), Buf(Bm)
            init = np.full((M, N), SENTINEL, dtype=np.int64).view(np.float64)
            Cb = Buf(init, fill=SENTINEL)
            rv = torch.from_numpy(r).cuda()
            part = torch.full((len(tiles) + 3,), NAN, dtype=torch.float64, device="cuda")
            part0 = part.clone()
            last = dict(row_vec=rv.data_ptr(), ssq_partials=part.data_ptr(), ssq_partials_elems=len(tiles))
            tag = "M=%d N=%d K=%d %s" % (M, N, K, mode)
            if mode == "chunks":
                s0 = gemm(A_KM, B_KN, M, N, 16, Ab, Bb, Cb, 2.0, 0.0, flags=TRAP)
                s = gemm(A_KM, B_KN, M, N, K - 16, (Ab.ptr + 16 * Ab.ld * 8, Ab.ld), (Bb.ptr + 16 * Bb.ld * 8, Bb.ld),
                         Cb, 2.0, 1.0, flags=TRAP, **last)
                s = s or s0
            else:
                kw = dict(wave_ctas=2, serpentine=1, group_m=3) if mode == "serpentine" else {}
                s = gemm(A_KM, B_KN, M, N, K, Ab, Bb, Cb, 2.0, 0.0, flags=TRAP, **kw, **last)
            if s != 0:
                failures.append("%s: status %d" % (tag, s))
                continue
            ref = 2 * (A.astype(np.int64) @ Bm.astype(np.int64) - r.astype(np.int64)[:, None])
            got = Cb.get()
            if not np.array_equal(got[comp], ref[comp]):
                failures.append("%s: %d trapezoid entries wrong" % (tag, int((got[comp] != ref[comp]).sum())))
            if not np.array_equal(got.view(np.int64)[~comp], init.view(np.int64)[~comp]) or not Cb.outside_intact():
                failures.append("%s: an upper tile or C's surroundings were written" % tag)
            order = trap_tiles(M, N, 128, 3 if mode == "serpentine" else 16)
            want = []
            for a, b in order:
                blk = ref[a * 128:(a + 1) * 128, b * 128:(b + 1) * 128]
                rows = 2 * r[a * 128:(a + 1) * 128].astype(np.int64)[:, None]
                cols = 2 * r[b * 128:b * 128 + blk.shape[1]].astype(np.int64)[None, :]
                want.append(float(((blk + rows) ** 2).sum() + (((blk + cols) ** 2).sum() if a > b else 0)))
            got_p = part.cpu().numpy()
            if not np.array_equal(got_p[:len(tiles)], np.array(want)):
                failures.append("%s: partials %s != %s" % (tag, got_p[:4], want[:4]))
            if not torch.equal(part.view(torch.int64)[len(tiles):], part0.view(torch.int64)[len(tiles):]):
                failures.append("%s: a slot past the launched tiles was written" % tag)
    assert not failures, "\n".join(failures)


@pytest.mark.parametrize("dense", [False, True])
def test_rank_one_dominated_step_matches_oracle(dense):
    """y far outside the ensemble's outputs: c = E^T Gamma^-1 (mean - y) dominates D = (S + c 1^T) / J, and the stored
    S / J = (acc - c_i) / J cancels most of each product.  Several panels and ragged J, host and device steps."""
    d, k, J = 40, 96, 1000
    pr = eo.linear_gaussian_problem(d, k, J, dense_gamma=dense)
    spread = float(np.abs(pr["G"] - pr["G"].mean(axis=1, keepdims=True)).max())
    y = pr["y"] + 100.0 * spread
    eng = Engine(d, k, J, d_panel_bytes=256 * 8 * 1008)        # 256-column panels -> 4 panels
    try:
        eng.set_problem(y, pr["Gamma"], pr["Sigma0"], pr["mu"], pr["ustar"])
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        for rule in ("eks", "aldi", "aldi_constant", "eki"):
            xi = pr["xi"] if rule != "eki" else None
            o = eo.step(rule, y, pr["U0"], pr["G"], pr["Gamma"], pr["mu"], pr["Sigma0"], pr["ustar"], pr["xi"])
            Uk, hk, _ = eng.step_host(rule, pr["U0"], pr["G"], xi)
            assert _rel(Uk, o["Uk"]) < TOL and abs(hk - o["hk"]) <= TOL * o["hk"], rule
            Ud, hd, _ = eng.step(rule, dev(pr["U0"]), dev(pr["G"]), dev(xi) if xi is not None else None)
            assert _rel(Ud.cpu().numpy(), o["Uk"]) < TOL and abs(hd - o["hk"]) <= TOL * o["hk"], rule
    finally:
        eng.close()


def test_constant_time_step_resolve_over_panels_with_dense_gamma():
    """time_step='constant' re-solves D with M = hk C^pp + Gamma (W = M^-1 R, w0 = M^-1 c) on 128-column panels of a ragged
    J, dense Gamma, against the oracle."""
    d, k, J = 20, 40, 600
    pr = eo.linear_gaussian_problem(d, k, J, dense_gamma=True)
    for rule in ("aldi", "eks"):
        for ts in ("constant", "mix"):
            s = calibrate.sampling(d, k, J)
            s.mu, s.sigma, s.ustar = pr["mu"], pr["Sigma0"], pr["ustar"]
            s.d_panel_bytes = 128 * 8 * 608
            s._ensure_metrics()
            np.random.seed(1)
            Uk = getattr(s, {"aldi": "eks_update_aldi", "eks": "eks_update"}[rule])(
                pr["y"], pr["U0"], pr["G"], pr["Gamma"], 0, time_step=ts, delta_t=0.03)
            o = eo.step(rule, pr["y"], pr["U0"], pr["G"], pr["Gamma"], pr["mu"], pr["Sigma0"], pr["ustar"], pr["xi"],
                        time_step=ts, delta_t=0.03, T=s.T, t_last=None)
            assert _rel(Uk, o["Uk"]) < TOL, (rule, ts)


def test_profile_reports_the_flops_of_the_trapezoid():
    """The D profile counts 2 K per output of the launched tiles: sum over panels [a, b) of the lower trapezoid of a
    (J - a) x (b - a) product, not 2 k J^2."""
    d, k, J, panel = 24, 272, 4300, 1536
    pr = eo.linear_gaussian_problem(d, k, J)
    want = 0.0
    for a in range(0, J, panel):
        b = min(a + panel, J)
        for n0 in range(0, b - a, 128):
            want += 2.0 * k * min(128, b - a - n0) * (J - a - n0)
    eng = Engine(d, k, J, d_panel_bytes=panel * 8 * 4304)
    try:
        eng.set_problem(pr["y"], pr["Gamma"], pr["Sigma0"], pr["mu"], pr["ustar"])
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        eng.profile(True)
        eng.step("eks", dev(pr["U0"]), dev(pr["G"]), dev(pr["xi"]))
        ms, n, fl = eng.profile_read()
        assert n == 3 and fl == want and ms > 0, (n, fl, want)
        eng.step_host("eks", pr["U0"], pr["G"], pr["xi"])
        ms, n, fl = eng.profile_read()
        assert n >= 3 and fl == want, (n, fl, want)
        eng.profile(False)
    finally:
        eng.close()
