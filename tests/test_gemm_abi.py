"""ces_gemm, ces_gemm_ex and ces_potri refuse bad arguments with CES_ERR_INVALID before any device work, so on a machine
without a GPU too.  Every call below passes a 16-byte misaligned A: a call that got past the argument checks would stop at
the tensor-map encoding with CES_ERR_ALIGN (or CES_ERR_CUDA without a driver), never launch a kernel."""
import ctypes

from ces_b200 import _lib

A, B, C, WS, PART, DEV = 0x10008, 0x20000, 0x30000, 0x40000, 0x50000, 0x60000
NOT_REACHED = (_lib.CES_ERR_ALIGN, _lib.CES_ERR_CUDA)


def _ex(**kw):
    base = dict(a_mode=0, b_mode=0, M=200, N=130, K=33, A=A, lda=34, B=B, ldb=130, C=C, ldc=130)
    base.update(kw)
    d = _lib.GemmDesc(**base)
    return _lib.load().ces_gemm_ex(None, ctypes.byref(d))


def _last():
    return _lib.load().ces_last_error()


def test_valid_descriptors_get_past_the_argument_checks():
    """The baseline of every rejection below is accepted: each rejection is caused by the one field it changes."""
    ok = [dict(), dict(a_mode=1, lda=200), dict(b_mode=1, ldb=34), dict(splits=3, splitk_ws=WS, splitk_ws_elems=3 * 200 * 130),
          dict(splits=100, splitk_ws=WS, splitk_ws_elems=3 * 200 * 130),           # clamped to the 3 k-blocks
          dict(M=130, flags=2, splits=2, splitk_ws=WS, splitk_ws_elems=2 * 130 * 130, diag_add=1.0),
          dict(ssq_partials=PART, ssq_partials_elems=4), dict(batch=3, ssq_partials=PART, ssq_partials_elems=12),
          dict(batch=3, splitk_ws=WS, splitk_ws_elems=3 * 200 * 130, a_batch_rows=200),
          dict(a_mode=1, lda=200, batch=2, a_batch_rows=33, c_batch_elems=200 * 130),
          dict(a_mode=1, lda=200, K=32, batch=2, a_batch_rows=32, b_batch_rows=32, c_batch_elems=200 * 130),
          dict(flags=1 | 4, alpha_dev=DEV, group_m=3, wave_ctas=2, serpentine=1), dict(serpentine=0)]
    for kw in ok:
        assert _ex(**kw) in NOT_REACHED, (kw, _last())


def test_gemm_ex_refuses_a_foreign_struct_size():
    for size in (0, ctypes.sizeof(_lib.GemmDesc) - 8, ctypes.sizeof(_lib.GemmDesc) + 8):
        assert _ex(struct_size=size) == _lib.CES_ERR_INVALID, size
        assert b"struct_size" in _last()
    assert _lib.load().ces_gemm_ex(None, None) == _lib.CES_ERR_INVALID


def test_gemm_ex_refuses_capacity_overflows():
    cases = [dict(splits=3, splitk_ws=WS, splitk_ws_elems=3 * 200 * 130 - 1),
             dict(splits=100, splitk_ws=WS, splitk_ws_elems=3 * 200 * 130 - 1),
             dict(splitk_ws=WS, splitk_ws_elems=200 * 130 - 1),
             dict(batch=4, splitk_ws=WS, splitk_ws_elems=3 * 200 * 130, a_batch_rows=200),
             dict(ssq_partials=PART, ssq_partials_elems=3),
             dict(batch=3, ssq_partials=PART, ssq_partials_elems=11),
             dict(M=64, N=257, ssq_partials=PART, ssq_partials_elems=2)]
    for kw in cases:
        assert _ex(**kw) == _lib.CES_ERR_INVALID, kw
        assert b"smaller than" in _last(), kw


def test_gemm_ex_refuses_bad_modes_sizes_and_flags():
    for kw in (dict(a_mode=2), dict(b_mode=-1), dict(M=0), dict(K=0), dict(N=(1 << 30) + 1), dict(batch=0),
               dict(batch=65536), dict(a_batch_rows=-1), dict(c_batch_elems=-1), dict(splits=-1), dict(splits=65536),
               dict(group_m=-1), dict(flags=8), dict(flags=16), dict(wave_ctas=-1), dict(serpentine=2), dict(serpentine=-2),
               dict(A=None), dict(C=None)):
        assert _ex(**kw) == _lib.CES_ERR_INVALID, kw


def test_gemm_refuses_the_unsupported_feature_combinations():
    ws = dict(splitk_ws=WS, splitk_ws_elems=8 * 200 * 200)
    cases = {
        b"diag_add needs the workspace": dict(M=130, flags=2, diag_add=1e-8),
        b"GEMM_C_LOWER_ONLY cannot produce sum-of-squares": dict(M=130, flags=2, ssq_partials=PART, ssq_partials_elems=64),
        b"GEMM_C_LOWER_ONLY needs a square C": dict(flags=2),
        b"needs K % 16 == 0": dict(a_mode=1, lda=200, batch=2, a_batch_rows=33, b_batch_rows=33, c_batch_elems=200 * 130),
        b"split-K needs a workspace": dict(splits=2),
        b"workspace path cannot produce": dict(ssq_partials=PART, ssq_partials_elems=64, **ws),
        b"batching excludes split-K": dict(batch=2, splits=2, **ws),
    }
    for msg, kw in cases.items():
        assert _ex(**kw) == _lib.CES_ERR_INVALID, (msg, kw)
        assert msg in _last(), (msg, _last())
    # the batched hazard is specific to A_KM x B_KN with both operands batched
    for kw in (dict(a_mode=1, lda=200, batch=2, a_batch_rows=33, c_batch_elems=200 * 130),
               dict(a_mode=1, lda=200, b_mode=1, ldb=34, batch=2, a_batch_rows=33, b_batch_rows=130, c_batch_elems=200 * 130),
               dict(batch=2, a_batch_rows=200, b_batch_rows=33, c_batch_elems=200 * 130)):
        assert _ex(**kw) in NOT_REACHED, (kw, _last())


def test_leading_dimensions_below_the_operand_widths_are_refused():
    lib = _lib.load()

    def gemm(am, bm, lda, ldb, ldc, M=200, N=130, K=33):
        return lib.ces_gemm(None, am, bm, M, N, K, 1.0, A, lda, B, ldb, 0.0, C, ldc)

    # (a_mode, b_mode) -> the smallest leading dimensions: A_MK K, A_KM M; B_KN N, B_NK K; C N
    smallest = {(0, 0): (33, 130, 130), (1, 0): (200, 130, 130), (0, 1): (33, 33, 130), (1, 1): (200, 33, 130)}
    for (am, bm), (lda, ldb, ldc) in smallest.items():
        assert gemm(am, bm, lda, ldb, ldc) in NOT_REACHED, (am, bm, _last())
        for bad in ((lda - 1, ldb, ldc), (lda, ldb - 1, ldc), (lda, ldb, ldc - 1)):
            assert gemm(am, bm, *bad) == _lib.CES_ERR_INVALID, (am, bm, bad)
            assert b"leading dimension" in _last()
        assert _ex(a_mode=am, b_mode=bm, lda=lda - 1, ldb=ldb, ldc=ldc) == _lib.CES_ERR_INVALID
        assert _ex(a_mode=am, b_mode=bm, lda=lda, ldb=ldb, ldc=ldc - 1) == _lib.CES_ERR_INVALID


def test_potri_refuses_bad_arguments():
    lib = _lib.load()
    assert lib.ces_potri(None, None, 8, 8, C, 8) == _lib.CES_ERR_INVALID
    assert lib.ces_potri(None, A, 8, 8, None, 8) == _lib.CES_ERR_INVALID
    assert lib.ces_potri(None, A, 7, 8, C, 8) == _lib.CES_ERR_INVALID
    assert lib.ces_potri(None, A, 8, 8, C, 7) == _lib.CES_ERR_INVALID
    assert lib.ces_potri(None, A, 8, 0, C, 8) == _lib.CES_ERR_INVALID
    assert b"ces_potri" in _last()
