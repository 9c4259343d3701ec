"""numpy restatement of ``noise='ensemble'`` (DESIGN.md section 4g): the J x J Philox stream of
``ces_fill_ensemble_noise`` and the update step with the ensemble form of the noise.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py) -- the checker of the device path, never the product.

The step is not part of the reference, so there is nothing to pin it to there: it is built from the pinned pieces.  The
deterministic part is ``eks_oracle.step`` with xi = 0 (its noise term sqrt(2h) chol(C) 0 is exactly 0, so the result is
bit for bit the reference's update without noise), and the noise term is added last, as the reference adds its own:

    noise term = sqrt(2h / n_C) (U - ubar) xi,   xi (J, J),   n_C = J for eks (bias=True), J - 1 for aldi / aldi_constant

Stream: xi[s, j] is Philox4x32-10 keyed by (seed low, seed high) at the counter (j >> 1, TAG_ENS, s, step mod 2^32), the
cosine of the Box-Muller pair for even j and the sine for odd j (the block function, u53 and Box-Muller of
oracle/philox_oracle.py, which tests/test_philox_oracle.py pins to the Random123 known-answer vectors).
"""
import numpy as np

from . import eks_oracle
from .philox_oracle import M32, _key, normal_pair, philox4x32_10

TAG_ENS = 0x454E        # counter word 1 of the ensemble noise (csrc/ensemble.cu: fill_ensemble_noise_kernel)
NOISY_RULES = ("eks", "aldi", "aldi_constant")


def ensemble_noise(seed, step, rows, cols, row_offset=0, col_offset=0):
    """(rows, cols) block of ``ces_fill_ensemble_noise``: source particles row_offset .. row_offset + rows - 1, target
    particles col_offset .. col_offset + cols - 1 of the J x J xi at (seed, step)."""
    gc = np.uint64(col_offset) + np.arange(cols, dtype=np.uint64)
    s = (np.uint64(row_offset) + np.arange(rows, dtype=np.uint64))[:, None]
    out = philox4x32_10(((gc >> np.uint64(1)) & M32, TAG_ENS, s & M32, int(step) & 0xFFFFFFFF), _key(seed))
    cs, sn = normal_pair(out)
    return np.where((gc & np.uint64(1)) == 0, cs, sn)


def n_c(rule, J):
    """Normalisation of the rule's own C^uu: np.cov(U, bias=True) for eks (:424), np.cov(U) for the aldi rules (:476, :512)."""
    return J if rule == "eks" else J - 1


def step(rule, y, U, G, Gamma, mu, Sigma0, ustar, xi, **kwargs):
    """``eks_oracle.step`` with the ensemble noise: xi is (J, J).  Same keyword arguments and return value; eki has no
    noise term and is returned unchanged."""
    U = np.asarray(U, dtype=float)
    p, J = U.shape
    out = eks_oracle.step(rule, y, U, G, Gamma, mu, Sigma0, ustar, np.zeros((p, J)), **kwargs)
    if rule in NOISY_RULES:
        xi = np.asarray(xi, dtype=float)
        if xi.shape != (J, J):
            raise ValueError("the ensemble noise takes xi of shape (J, J) = (%d, %d), got %s" % (J, J, xi.shape))
        Ut = U - U.mean(axis=1)[:, None]
        out["Uk"] = out["Uk"] + np.sqrt(2 * out["hk"] / n_c(rule, J)) * (Ut @ xi)
    return out
