"""numpy restatement of the device's Philox4x32-10 streams: ``ces_fill_normal`` (csrc/ensemble.cu, the EKS noise of
``sampling.run(rng='device')``) and the per-chain noise of the Metropolis-Hastings samplers (csrc/rng.cuh, every chain
but the one that consumes numpy's MT19937 stream).

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py) -- the checker of the device noise, never the product.

Parity: PINNED.  tests/test_philox_oracle.py checks the block function against the Random123 known-answer vectors of
Philox4x32-10 (Salmon et al., SC'11); tests/test_gpu_philox_streams.py compares the device streams with this module.

Block function: 10 rounds of
    (c0, c1, c2, c3) <- (hi(M1 c2) ^ c1 ^ k0,  lo(M1 c2),  hi(M0 c0) ^ c3 ^ k1,  lo(M0 c0)),  M0 = 0xD2511F53, M1 = 0xCD9E8D57
with the key bumped by (0x9E3779B9, 0xBB67AE85) after every round.  Uniform from a pair of output words:
    u53(hi, lo) = min((((hi << 32 | lo) >> 11) + 1/2) / 2^53, 1 - 2^-53)
in double arithmetic (the top 53-bit value would round to 1.0 without the min).  Normal pair (Box-Muller):
    r = sqrt(-2 log u53(o0, o1)),  (r cos 2 pi u2, r sin 2 pi u2),  u2 = u53(o2, o3).
Counters (words 0..3) and key (words 0, 1):
    fill_normal      (pair g low, pair g high, row, step mod 2^32), key (seed low, seed high); global column 2 g takes the
                     cosine, 2 g + 1 the sine
    chain noise      normal pair j of chain c at step it: (it, c, j, tag); the accept test's uniform: (it, c, 0xffffffff,
                     tag), u53 of output words 0, 1; key (seed low, seed high)
"""
import numpy as np

M32 = np.uint64(0xFFFFFFFF)
PHILOX_M = (np.uint64(0xD2511F53), np.uint64(0xCD9E8D57))
PHILOX_W = (np.uint64(0x9E3779B9), np.uint64(0xBB67AE85))
U53_MAX = 1.0 - 2.0 ** -53

# the Philox counter word of each sampler's chain noise
TAG_MH = 0x4D48         # ces_mcmc_model_mh (csrc/mcmc.cu)
TAG_GP = 0x4750         # ces_gp_mh (csrc/emulate.cu)
TAG_DARCY = 0x4452      # ces_darcy_mh (csrc/darcy_mh.cu)


def _words(x):
    return np.asarray(x, dtype=np.uint64) & M32


def philox4x32_10(ctr, key):
    """Philox4x32-10 of the counter words ``ctr`` (4 arrays or scalars, broadcast together) under the key words ``key``
    (2); returns the 4 output words as uint64 arrays of the broadcast shape."""
    c = [_words(w) for w in np.broadcast_arrays(*[np.asarray(w, dtype=np.uint64) for w in ctr])]
    k0, k1 = _words(key[0]), _words(key[1])
    for _ in range(10):
        p0 = PHILOX_M[0] * c[0]                     # 32 x 32 -> 64-bit products: exact in uint64
        p1 = PHILOX_M[1] * c[2]
        c = [((p1 >> np.uint64(32)) ^ c[1] ^ k0) & M32, p1 & M32, ((p0 >> np.uint64(32)) ^ c[3] ^ k1) & M32, p0 & M32]
        k0 = (k0 + PHILOX_W[0]) & M32
        k1 = (k1 + PHILOX_W[1]) & M32
    return c


def u53(hi, lo):
    """Uniform in (0, 1) from two output words."""
    x = (_words(hi) << np.uint64(32)) | _words(lo)
    return np.minimum(((x >> np.uint64(11)).astype(np.float64) + 0.5) * 2.0 ** -53, U53_MAX)


def normal_pair(out):
    """The Box-Muller pair (cosine, sine) of the four output words ``out``."""
    rad = np.sqrt(-2.0 * np.log(u53(out[0], out[1])))
    ang = np.pi * (2.0 * u53(out[2], out[3]))
    return rad * np.cos(ang), rad * np.sin(ang)


def _key(seed):
    seed = int(seed)
    return seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF


def fill_normal(seed, step, rows, cols, col_offset=0):
    """(rows, cols) block of ``ces_fill_normal``: rows 0..rows-1, global columns col_offset .. col_offset + cols - 1."""
    gc = np.uint64(col_offset) + np.arange(cols, dtype=np.uint64)
    g = gc >> np.uint64(1)
    row = np.arange(rows, dtype=np.uint64)[:, None]
    out = philox4x32_10((g & M32, g >> np.uint64(32), row, int(step) & 0xFFFFFFFF), _key(seed))
    cs, sn = normal_pair(out)
    return np.where((gc & np.uint64(1)) == 0, cs, sn)


def chain_noise(seed, tag, it, c, p):
    """``(z (p), u)``: the proposal's normals and the accept test's uniform of chain ``c`` at step ``it``."""
    j = np.arange((p + 1) // 2, dtype=np.uint64)
    cs, sn = normal_pair(philox4x32_10((it, c, j, tag), _key(seed)))
    z = np.empty(2 * len(j))
    z[0::2], z[1::2] = cs, sn
    out = philox4x32_10((it, c, 0xFFFFFFFF, tag), _key(seed))
    return z[:p], float(u53(out[0], out[1]))
