"""ctypes binding of libces_b200.so (include/ces_b200.h).

The library is the product: if it is missing or fails to load this module raises
-- there is no CPU fallback anywhere in ces_b200.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libces_b200.so")

CES_OK = 0
CES_ERR_INVALID, CES_ERR_STATE, CES_ERR_ALIGN, CES_ERR_NOT_SPD, CES_ERR_CUDA, CES_ERR_NOMEM = -1, -2, -3, -4, -5, -6
RULES = {"eks": 0, "aldi": 1, "aldi_constant": 2, "eki": 3}
TS_FROBENIUS, TS_FIXED, TS_KEEP = 0, 1, 2
FORMULATIONS = {"interaction": 0, "factored": 1}
NOISES = {"cholesky": 0, "ensemble": 1}            # CES_NOISE_*
MAPS = {"lineal": 0, "lineal_log": 1, "elliptic": 2, "banana": 3}
GP_KERNELS = {"SquaredExponential": 0, "Matern12": 1, "Matern32": 2, "Matern52": 3}   # CES_GP_* (GPflow's class names)

# every symbol include/ces_b200.h declares (tests/test_abi.py checks the .so exports them all)
EXPORTS = (
    "ces_version", "ces_last_error", "ces_create", "ces_destroy", "ces_set_problem", "ces_phase1_sums",
    "ces_phase2_centre", "ces_phase3_interact", "ces_phase4a_drift", "ces_phase4_update", "ces_step",
    "ces_step_host", "ces_forward_map", "ces_buffer", "ces_launch_count", "ces_gemm", "ces_potrf", "ces_posv",
    "ces_profile_enable", "ces_profile_read", "ces_darcy_create", "ces_darcy_destroy", "ces_darcy_forward", "ces_darcy_last_stats",
    "ces_peek_step_size", "ces_phase3b_cpp", "ces_phase3c_resolve", "ces_phase3f_products", "ces_phase3f_finish",
    "ces_fill_normal", "ces_phase3_blocks", "ces_frobenius", "ces_phase3d_spectral", "ces_lorenz63_forward",
    "ces_lorenz96_forward", "ces_set_pending_output", "ces_timeline_enable",
    "ces_timeline_mark", "ces_timeline_read", "ces_host_begin", "ces_host_sums_g", "ces_host_centre_g", "ces_host_sums_u",
    "ces_host_centre_u", "ces_host_interact_own", "ces_host_update", "ces_ipc_export", "ces_ipc_import", "ces_peer_gather",
    "ces_peer_gather_wait", "ces_host_interact_chunk", "ces_small_run", "ces_mcmc_model_mh", "ces_host_chunk_schedule",
    "ces_gp_create", "ces_gp_destroy", "ces_gp_lml", "ces_gp_condition", "ces_gp_predict", "ces_gp_mh", "ces_darcy_mh",
    "ces_gp_set_kernel", "ces_set_noise", "ces_fill_ensemble_noise", "ces_potri", "ces_gemm_ex",
)

_i64, _int, _dbl, _vp = ctypes.c_int64, ctypes.c_int, ctypes.c_double, ctypes.c_void_p
_dp = ctypes.c_void_p  # double* (host or device) passed as an address


class GemmDesc(ctypes.Structure):
    """ces_gemm_desc (test support: the whole DMMA GEMM family, see include/ces_b200.h)."""
    _fields_ = [("struct_size", _i64), ("a_mode", ctypes.c_int32), ("b_mode", ctypes.c_int32),
                ("M", _i64), ("N", _i64), ("K", _i64), ("A", _dp), ("lda", _i64), ("B", _dp), ("ldb", _i64),
                ("C", _dp), ("ldc", _i64), ("alpha", _dbl), ("beta", _dbl), ("alpha_dev", _dp),
                ("flags", ctypes.c_int32), ("group_m", ctypes.c_int32), ("splits", ctypes.c_int32),
                ("wave_ctas", ctypes.c_int32), ("serpentine", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("splitk_ws", _dp), ("splitk_ws_elems", _i64), ("diag_add", _dbl), ("ssq_partials", _dp),
                ("ssq_partials_elems", _i64), ("batch", _i64), ("a_batch_rows", _i64), ("b_batch_rows", _i64),
                ("c_batch_elems", _i64), ("row_vec", _dp)]

    def __init__(self, **kw):
        base = dict(struct_size=ctypes.sizeof(GemmDesc), alpha=1.0, serpentine=-1, batch=1)
        base.update(kw)
        super().__init__(**base)


class CesError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("ces_b200 error %d: %s" % (code, message))
        self.code = code


_lib = None


def load():
    """Load libces_b200.so (once).  Raises OSError with build instructions if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise OSError("%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                      "(or `make -C ces_b200/csrc`).  ces_b200 has no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    lib.ces_version.restype = ctypes.c_char_p
    lib.ces_last_error.restype = ctypes.c_char_p
    lib.ces_launch_count.restype = _i64
    lib.ces_launch_count.argtypes = [_vp]
    lib.ces_create.argtypes = [_i64, _i64, _i64, _i64, _int, _int, _i64, _vp, _i64, ctypes.POINTER(_vp)]
    lib.ces_destroy.argtypes = [_vp]
    lib.ces_set_problem.argtypes = [_vp, _dp, _dp, _dp, _dp, _dp]
    lib.ces_phase1_sums.argtypes = [_vp, _dp, _i64, _dp, _i64]
    lib.ces_phase2_centre.argtypes = [_vp, _int, _dp, _i64, _dp, _i64]
    lib.ces_phase3_interact.argtypes = [_vp, _int, _int]
    lib.ces_peek_step_size.argtypes = [_vp, _int, _dbl, ctypes.POINTER(_dbl)]
    lib.ces_phase3_blocks.argtypes = [_vp, _int, _int, _int]
    lib.ces_phase3b_cpp.argtypes = [_vp]
    lib.ces_phase3f_products.argtypes = [_vp, _int]
    lib.ces_phase3f_finish.argtypes = [_vp, _int]
    lib.ces_phase3c_resolve.argtypes = [_vp, _int]
    lib.ces_phase3d_spectral.argtypes = [_vp, ctypes.POINTER(_dbl), ctypes.POINTER(_int)]
    lib.ces_phase4a_drift.argtypes = [_vp, _dbl]
    lib.ces_phase4_update.argtypes = [_vp, _int, _int, _dbl, _dp, _i64, _dp, _i64, _dp, _i64,
                                      ctypes.POINTER(_dbl), ctypes.POINTER(_dbl)]
    lib.ces_step.argtypes = [_vp, _int, _int, _dbl, _dbl, _int, _dp, _i64, _dp, _i64, _dp, _i64, _dp, _i64,
                             ctypes.POINTER(_dbl), ctypes.POINTER(_dbl)]
    lib.ces_step_host.argtypes = [_vp, _int, _int, _dbl, _dbl, _int, _dp, _dp, _dp, _dp,
                                  ctypes.POINTER(_dbl), ctypes.POINTER(_dbl)]
    lib.ces_set_pending_output.argtypes = [_vp, _dp]
    lib.ces_ipc_export.argtypes = [_vp, ctypes.c_char_p, ctypes.c_char_p]
    lib.ces_ipc_import.argtypes = [_vp, _int, ctypes.c_char_p, ctypes.c_char_p]
    lib.ces_peer_gather.argtypes = [_vp]
    lib.ces_peer_gather_wait.argtypes = [_vp]
    lib.ces_host_begin.argtypes = [_vp, _int, _int, _dp, _dp, _dp, ctypes.POINTER(_int), ctypes.POINTER(_i64)]
    lib.ces_host_sums_g.argtypes = [_vp, _int]
    lib.ces_host_centre_g.argtypes = [_vp, _int, _int]
    lib.ces_host_interact_chunk.argtypes = [_vp, _int]
    lib.ces_host_sums_u.argtypes = [_vp]
    lib.ces_host_centre_u.argtypes = [_vp]
    lib.ces_host_interact_own.argtypes = [_vp]
    lib.ces_host_update.argtypes = [_vp, _int, _dbl, _dp, ctypes.POINTER(_dbl), ctypes.POINTER(_dbl)]
    lib.ces_timeline_enable.argtypes = [_vp, _int]
    lib.ces_timeline_mark.argtypes = [_vp, ctypes.c_char_p]
    lib.ces_timeline_read.argtypes = [_vp, ctypes.c_char_p, _i64, ctypes.POINTER(_dbl), _i64, ctypes.POINTER(_i64)]
    lib.ces_small_run.argtypes = [_vp, _int, _int, _dbl, _dbl, _int, _dp, _i64, _dp, _dp, _dp, _dp, ctypes.c_uint64, ctypes.c_uint64,
                                  _i64, _dbl, _int, _dbl, _dp, _dp, _dp, _dp, ctypes.POINTER(_i64)]
    lib.ces_mcmc_model_mh.argtypes = [_vp, _int, _i64, _i64, _dp, _i64, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _int, _dbl, _i64, _i64,
                                      _dp, _dp, _dp, _dp, ctypes.c_uint64, _dp, _dp]
    lib.ces_gp_create.argtypes = [_vp, _i64, _i64, _i64, _dp, _dp, _dp, ctypes.POINTER(_vp)]
    lib.ces_gp_destroy.argtypes = [_vp]
    lib.ces_gp_set_kernel.argtypes = [_vp, _int]
    lib.ces_gp_lml.argtypes = [_vp, _i64, _i64, _dp, _dbl, _dp, _dp]
    lib.ces_gp_condition.argtypes = [_vp, _dp, _dbl]
    lib.ces_gp_predict.argtypes = [_vp, _dp, _i64, _i64, _dp, _i64, _dp, _i64]
    lib.ces_gp_mh.argtypes = [_vp, _dp, _int, _dp, _dp, _dp, _int, _dbl, _i64, _i64, _dp, _dp, _dp, _dp, ctypes.c_uint64,
                              _dp, _dp]
    lib.ces_darcy_mh.argtypes = [_vp, _dbl, _int, _dp, _dp, _dp, _dp, _dp, _int, _dbl, _i64, _i64, _dp, _dp, _dp, _dp,
                                 ctypes.c_uint64, _dp, _dp]
    lib.ces_host_chunk_schedule.argtypes = [_i64, _i64, _i64, _int, _dbl, ctypes.POINTER(_i64)]
    lib.ces_forward_map.argtypes = [_vp, _int, _dp, _i64, _dp, _dp, _dp, _i64, _dp, _i64]
    lib.ces_buffer.argtypes = [_vp, ctypes.c_char_p, ctypes.POINTER(_vp), ctypes.POINTER(_i64),
                               ctypes.POINTER(_i64), ctypes.POINTER(_i64)]
    lib.ces_profile_enable.argtypes = [_vp, _int]
    lib.ces_profile_read.argtypes = [_vp, ctypes.POINTER(_dbl), ctypes.POINTER(_i64), ctypes.POINTER(_dbl)]
    lib.ces_darcy_create.argtypes = [_i64, _i64, _dp, _dp, _dp, _vp, _i64, _vp, ctypes.POINTER(_vp)]
    lib.ces_darcy_destroy.argtypes = [_vp]
    lib.ces_darcy_forward.argtypes = [_vp, _dp, _i64, _i64, _dp, _i64, _int, _dbl, _int, ctypes.POINTER(_int)]
    lib.ces_lorenz63_forward.argtypes = [_vp, _int, _dp, _i64, _i64, _i64, _dp, _i64, _i64, _dbl, _int, _i64, _dp, _i64, _dp, _i64, _dp, _i64]
    lib.ces_lorenz96_forward.argtypes = [_vp, ctypes.POINTER(_int), _int, _int, _dp, _i64, _i64, _i64, _dp, _i64, _i64, _dbl,
                                         _int, _i64, _i64, _int, _int, _dp, _i64, _dp, _i64, _dp, _i64]
    lib.ces_darcy_last_stats.argtypes = [_vp, ctypes.POINTER(_i64), ctypes.POINTER(_i64), ctypes.POINTER(_dbl)]
    lib.ces_frobenius.argtypes = [_vp, _dp, _i64, _i64, _i64, ctypes.POINTER(_dbl)]
    lib.ces_fill_normal.argtypes = [_vp, ctypes.c_uint64, ctypes.c_uint64, _dp, _i64, _i64, _i64, _i64]
    lib.ces_set_noise.argtypes = [_vp, _int, ctypes.c_uint64, ctypes.c_uint64, _dp, _i64]
    lib.ces_fill_ensemble_noise.argtypes = [_vp, ctypes.c_uint64, ctypes.c_uint64, _dp, _i64, _i64, _i64, _i64, _i64]
    lib.ces_gemm.argtypes = [_vp, _int, _int, _i64, _i64, _i64, _dbl, _dp, _i64, _dp, _i64, _dbl, _dp, _i64]
    lib.ces_potrf.argtypes = [_vp, _dp, _i64, _i64]
    lib.ces_posv.argtypes = [_vp, _dp, _i64, _i64, _dp, _i64, _i64]
    lib.ces_potri.argtypes = [_vp, _dp, _i64, _i64, _dp, _i64]
    lib.ces_gemm_ex.argtypes = [_vp, ctypes.POINTER(GemmDesc)]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if fn.restype is ctypes.c_int and name not in ("ces_version", "ces_last_error", "ces_launch_count"):
            fn.restype = _int
    _lib = lib
    return lib


def check(status):
    """Map a C status to the reference's exception conventions (SURVEY.md section 8b)."""
    if status == CES_OK:
        return
    msg = load().ces_last_error().decode("utf-8", "replace")
    if status == CES_ERR_NOT_SPD:
        raise np.linalg.LinAlgError(msg or "Matrix is not positive definite")
    if status == CES_ERR_NOMEM:
        raise MemoryError(msg)
    if status in (CES_ERR_INVALID, CES_ERR_ALIGN):
        raise ValueError(msg)
    raise CesError(status, msg)


def host_ptr(a):
    """Address of a C-contiguous float64 numpy array (kept alive by the caller)."""
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data
