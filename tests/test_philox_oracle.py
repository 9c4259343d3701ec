"""oracle/philox_oracle.py, the numpy restatement of the device's Philox4x32-10 streams: the Random123 known-answer
vectors, the uniform at the extreme output words, the shard invariance of the restated ces_fill_normal (odd offsets and
widths, the high word of the pair counter), the chain noise's layout, and the ``noise`` / ``start`` arguments of the
oracle chains.  CPU only."""
import numpy as np
import pytest
from scipy.stats import multivariate_normal

from oracle import forward_oracle as fo, gp_oracle as go, mcmc_oracle as mo, philox_oracle as po

# Random123 (Salmon et al., SC'11), kat_vectors: philox4x32 10 rounds
KAT = [((0x00000000, 0x00000000, 0x00000000, 0x00000000), (0x00000000, 0x00000000),
        (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
       ((0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff), (0xffffffff, 0xffffffff),
        (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
       ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
        (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]


@pytest.mark.parametrize("ctr,key,want", KAT)
def test_philox_known_answers(ctr, key, want):
    assert [int(w) for w in po.philox4x32_10(ctr, key)] == list(want)


def test_philox_is_vectorised_over_counters():
    ctr = [np.array([c[i] for c, _, _ in KAT]) for i in range(4)]
    out = po.philox4x32_10(ctr, (0, 0))
    for n, (c, _, _) in enumerate(KAT):
        assert [int(w[n]) for w in out] == [int(w) for w in po.philox4x32_10(c, (0, 0))]


def test_u53_stays_inside_the_open_interval():
    lo, hi = po.u53(0, 0), po.u53(0xffffffff, 0xffffffff)
    assert lo == 2.0 ** -54 and 0.0 < lo
    assert hi == 1.0 - 2.0 ** -53 and hi < 1.0
    # the min touches only the top value: its neighbour keeps (n + 1/2) / 2^53 as double arithmetic rounds it
    assert po.u53(0xffffffff, 0xfffff7ff) == ((2.0 ** 53 - 2) + 0.5) * 2.0 ** -53 == 1.0 - 2.0 ** -52
    assert po.u53(0x80000000, 0) == 0.5                     # 2^52 + 1/2 rounds to the even 2^52
    z = po.normal_pair([np.uint64(0), np.uint64(0), np.uint64(0xffffffff), np.uint64(0xffffffff)])
    assert np.all(np.isfinite(z)) and abs(z[0]) > 8.0
    z = po.normal_pair([np.uint64(0xffffffff)] * 4)
    assert np.all(np.isfinite(z)) and np.all(np.abs(z) < 1e-7)


@pytest.mark.parametrize("seed,step", [(0, 0), (7, 3), (2 ** 40 + 3, 2 ** 31)])
def test_fill_normal_is_shard_invariant(seed, step):
    rows, width = 3, 1001
    full = po.fill_normal(seed, step, rows, width, 0)
    assert full.shape == (rows, width) and np.all(np.isfinite(full))
    for off, w in ((0, 1), (1, 1), (1, 2), (125, 125), (499, 1), (7, 994), (998, 3), (0, 1001)):
        assert np.array_equal(po.fill_normal(seed, step, rows, w, off), full[:, off:off + w]), (off, w)
    # beyond 2^32 pairs the high word of the pair counter is used
    far = po.fill_normal(seed, step, rows, 10, 2 ** 33)
    assert np.array_equal(po.fill_normal(seed, step, rows, 9, 2 ** 33 + 1), far[:, 1:])
    assert not np.any(far == full[:, :10])
    # rows, steps and seeds (both key words) each key their own stream
    assert not np.any(po.fill_normal(seed, step + 1, rows, 10, 0) == full[:, :10])
    assert not np.any(po.fill_normal(seed + 2 ** 32, step, rows, 10, 0) == full[:, :10])
    assert not np.any(full[0, :10] == full[1, :10])


def test_fill_normal_pairs_cosine_and_sine():
    seed, step = 5, 2
    out = po.philox4x32_10((3, 0, 1, step), (seed, 0))
    cs, sn = po.normal_pair(out)
    got = po.fill_normal(seed, step, 2, 4, 5)                 # global columns 5..8: pairs 2, 3, 3, 4
    assert got[1, 1] == cs and got[1, 2] == sn
    x = po.fill_normal(11, 0, 8, 20000, 0).ravel()
    assert abs(x.mean()) < 0.01 and abs(x.var() - 1.0) < 0.02


def test_chain_noise_layout():
    seed, it, c = 2 ** 40 + 3, 17, 9
    z5, u5 = po.chain_noise(seed, po.TAG_MH, it, c, 5)
    z6, u6 = po.chain_noise(seed, po.TAG_MH, it, c, 6)
    assert np.array_equal(z5, z6[:5]) and u5 == u6 and 0.0 < u5 < 1.0
    cs, sn = po.normal_pair(po.philox4x32_10((it, c, 2, po.TAG_MH), (3, 256)))
    assert z6[4] == cs and z6[5] == sn
    out = po.philox4x32_10((it, c, 0xffffffff, po.TAG_MH), (3, 256))
    assert u5 == po.u53(out[0], out[1])
    for other in (po.chain_noise(seed, po.TAG_GP, it, c, 6), po.chain_noise(seed, po.TAG_MH, it, c + 1, 6),
                  po.chain_noise(seed, po.TAG_MH, it + 1, c, 6), po.chain_noise(3, po.TAG_MH, it, c, 6)):
        assert not np.any(other[0] == z6) and other[1] != u6


def _noise_from_numpy(p):
    """The default stream of the oracle loops, handed in as ``noise`` (no draws inside the forward model)."""
    return lambda it: (np.random.normal(0, 1, p), np.random.uniform())


def test_oracle_chains_take_start_and_noise():
    rs = np.random.RandomState(4)
    p, k, J = 3, 5, 12
    A = rs.normal(size=(k, p))
    fwd = lambda th: fo.lineal(A, np.asarray(th).reshape(-1, 1))[:, 0]
    y, Gamma = rs.normal(size=k), 0.5 * np.eye(k)
    Ustar = 0.3 * rs.normal(size=(p, J))
    prior = multivariate_normal(np.zeros(p), np.eye(p))
    np.random.seed(3)
    want, acc = mo.model_mh(fwd, 40, prior, Ustar, y, Gamma, delta=0.8)
    np.random.seed(3)
    got, acc2 = mo.model_mh(fwd, 40, prior, Ustar, y, Gamma, delta=0.8, noise=_noise_from_numpy(p))
    assert np.array_equal(got, want) and acc == acc2
    got, _ = mo.model_mh(fwd, 40, prior, Ustar, y, Gamma, delta=0.8, start=Ustar[:, 5],
                         noise=lambda it: po.chain_noise(1, po.TAG_MH, it, 5, p))
    assert np.array_equal(got[:, 0], Ustar[:, 5]) and not np.array_equal(got[:, 1:], want[:, 1:])

    def predict_one(u):
        return A @ u, 0.1 * np.ones(k)

    np.random.seed(3)
    want, acc = go.emulator_mh(predict_one, 40, prior, Ustar, y, delta=0.8)
    np.random.seed(3)
    got, acc2 = go.emulator_mh(predict_one, 40, prior, Ustar, y, delta=0.8, noise=_noise_from_numpy(p))
    assert np.array_equal(got, want) and acc == acc2
    got, _ = go.emulator_mh(predict_one, 40, prior, Ustar, y, delta=0.8, start=Ustar[:, 2],
                            noise=lambda it: po.chain_noise(1, po.TAG_GP, it, 2, p))
    assert np.array_equal(got[:, 0], Ustar[:, 2])
