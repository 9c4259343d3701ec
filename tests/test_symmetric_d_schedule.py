"""The single-GPU interaction schedule restated in numpy (csrc/api.cu symmetric_loops): D column panels [a, b) form only the
lower trapezoid of S / J (J D = S + c 1^T, S = E^T B E, c = E^T w0, w0 = B (mean - y)), the strictly lower tiles of each
panel's diagonal block are mirrored, V is the sum of the two panel products plus (U~ c / J) 1^T, and ||D||_F^2 comes from
the stored values.  It must reproduce U~ D and ||D||_F of the direct formula to rounding.  The tile edge is a parameter:
the index math is the same in units of tiles, and small tiles put many of them into small shapes.  The new GEMM mode's
argument checks are pinned here too (no GPU needed: they run before any device work)."""
import ctypes

import numpy as np
import pytest

from ces_b200 import _lib


def trap_tiles(M, N, T, group_m=16):
    """(tm, tn) of the lower trapezoid in the order of the kernel (gemm.cuh trap_tile)."""
    tiles_m, tiles_n = -(-M // T), -(-N // T)
    out = []
    for f in range(0, tiles_m, group_m):
        gs = min(tiles_m - f, group_m)
        for tn in range(min(f + gs, tiles_n)):
            for tm in range(max(f, tn), f + gs):
                out.append((tm, tn))
    return out


def schedule(E, W, w0, Ut, panel, T):
    k, J = E.shape
    c = E.T @ w0
    V = np.full((Ut.shape[0], J), np.nan)
    ssq = 0.0
    for a in range(0, J, panel):
        b = min(a + panel, J)
        nc, M = b - a, J - a
        Dws = np.full((M, nc), np.nan)
        acc = E[:, a:].T @ W[:, a:b]
        for tm, tn in trap_tiles(M, nc, T):                       # step 1: lower trapezoid, row term
            r, q = slice(tm * T, min((tm + 1) * T, M)), slice(tn * T, min((tn + 1) * T, nc))
            s = (acc[r, q] - c[a:][r, None]) / J
            Dws[r, q] = s
            ssq += ((s + c[a:][r, None] / J) ** 2).sum()           # step 6
            if tm > tn:
                ssq += ((s + c[a:][None, q] / J) ** 2).sum()
        for i in range(nc):                                        # step 2: mirror across tiles of the diagonal block
            for j in range(i + 1, nc):
                if i // T < j // T:
                    assert np.isnan(Dws[i, j])
                    Dws[i, j] = Dws[j, i]
        assert not np.isnan(Dws[:nc]).any()
        own = Ut[:, a:] @ Dws                                      # step 3
        V[:, a:b] = own if a == 0 else V[:, a:b] + own
        if b < J:                                                  # step 4
            later = Ut[:, a:b] @ Dws[nc:].T
            V[:, b:] = later if a == 0 else V[:, b:] + later
    V += (Ut @ c / J)[:, None]                                     # step 5
    return V, ssq


@pytest.mark.parametrize("seed", range(6))
def test_schedule_reproduces_the_direct_formula(seed):
    rng = np.random.default_rng(seed)
    T = int(rng.choice([4, 8]))
    J = int(rng.integers(3 * T, 12 * T)) | 1                       # ragged: J % T != 0
    k, p = int(rng.integers(2, 9)), int(rng.integers(1, 6))
    G = rng.standard_normal((k, J)) + 3.0
    y = rng.standard_normal(k)
    A = rng.standard_normal((k, k))
    B = np.linalg.inv(A @ A.T + k * np.eye(k))                     # dense symmetric Gamma^-1 (or M^-1)
    E = G - G.mean(axis=1, keepdims=True)
    R = G - y[:, None]
    W = B @ R
    w0 = B @ (G.mean(axis=1) - y)
    Ut = rng.standard_normal((p, J))
    D = E.T @ W / J
    for tiles_per_panel in (1, 2, 3):
        V, ssq = schedule(E, W, w0, Ut, tiles_per_panel * T, T)
        ref = Ut @ D
        assert np.abs(V - ref).max() <= 1e-12 * np.abs(ref).max(), tiles_per_panel
        assert abs(np.sqrt(ssq) - np.linalg.norm(D)) <= 1e-12 * np.linalg.norm(D), tiles_per_panel


def test_trapezoid_enumeration_is_the_full_grid_without_the_upper_tiles():
    """The kernel's compact enumeration visits exactly the tiles tn <= tm, in the order of the grouped full grid."""
    for tiles_m, tiles_n in [(1, 1), (5, 5), (17, 3), (40, 33), (512, 128), (33, 33)]:
        full = []
        for L in range(tiles_m * tiles_n):
            per = 16 * tiles_n
            first = (L // per) * 16
            gs = min(tiles_m - first, 16)
            r = L - (L // per) * per
            full.append((first + r % gs, r // gs))
        want = [t for t in full if t[1] <= t[0]]
        got = trap_tiles(tiles_m * 128, tiles_n * 128, 128)
        assert got == want and len(got) == tiles_m * tiles_n - tiles_n * (tiles_n - 1) // 2


A, B, C, PART, VEC = 0x10008, 0x20000, 0x30000, 0x50000, 0x70000
NOT_REACHED = (_lib.CES_ERR_ALIGN, _lib.CES_ERR_CUDA)
TRAP = 32


def _ex(**kw):
    base = dict(a_mode=1, b_mode=0, M=300, N=130, K=33, A=A, lda=300, B=B, ldb=130, C=C, ldc=130)
    base.update(kw)
    return _lib.load().ces_gemm_ex(None, ctypes.byref(_lib.GemmDesc(**base)))


def test_lower_trapezoid_mode_argument_checks():
    # 3 x 2 tiles, 5 in the trapezoid: the partials capacity is that of the launched tiles
    ok = [dict(flags=TRAP), dict(flags=TRAP, row_vec=VEC, ssq_partials=PART, ssq_partials_elems=5),
          dict(M=130, flags=TRAP), dict(row_vec=VEC), dict(flags=TRAP, row_vec=VEC, beta=1.0, serpentine=1, wave_ctas=2)]
    for kw in ok:
        assert _ex(**kw) in NOT_REACHED, (kw, _lib.load().ces_last_error())
    ws = dict(splitk_ws=0x40000, splitk_ws_elems=8 * 300 * 130)
    refused = [(b"needs M >= N", dict(M=129, flags=TRAP)),
               (b"GEMM_C_LOWER_TRAP excludes", dict(flags=TRAP, splits=2, **ws)),
               (b"GEMM_C_LOWER_TRAP excludes", dict(flags=TRAP, batch=2, c_batch_elems=300 * 130)),
               (b"GEMM_C_LOWER_TRAP excludes", dict(flags=TRAP | 2, M=130)),
               (b"row_vec needs the direct epilogue", dict(row_vec=VEC, splits=2, **ws)),
               (b"smaller than", dict(flags=TRAP, ssq_partials=PART, ssq_partials_elems=4))]
    for msg, kw in refused:
        assert _ex(**kw) == _lib.CES_ERR_INVALID, (msg, kw)
        assert msg in _lib.load().ces_last_error(), (msg, _lib.load().ces_last_error())
    assert _ex(flags=16) == _lib.CES_ERR_INVALID
