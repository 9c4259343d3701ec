"""The entry points of an update check their arguments before any device work (csrc/api.cu check_step): a refused call
returns its error code and message, leaves its outputs as they were and launches no kernel.

* ces_step and ces_step_host, on the single-CTA path and on the phase path: update rule, step-size rule (CES_TS_KEEP
  included: it belongs to phase 4), formulation, ensemble noise with the factored formulation, null U / G / U_next, and
  a null xi when the rule's Cholesky noise needs one;
* ces_host_begin, ces_small_run, ces_peek_step_size, ces_phase3f_products and ces_phase4_update, which still accepts
  CES_TS_KEEP after ces_peek_step_size."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from ces_b200 import _lib  # noqa: E402
from ces_b200.engine import Engine  # noqa: E402

INV = _lib.CES_ERR_INVALID
ALDI, EKI, BAD_RULE = _lib.RULES["aldi"], _lib.RULES["eki"], 9
FROB, KEEP, BAD_TS = _lib.TS_FROBENIUS, _lib.TS_KEEP, 7
INTER, FACT, BAD_FORM = _lib.FORMULATIONS["interaction"], _lib.FORMULATIONS["factored"], 5
SHAPES = {"single_cta": (4, 6, 10), "phases": (12, 20, 40)}     # p = 12 > 8 is too large for the single-CTA kernel


def _engine(p, k, J):
    rs = np.random.RandomState(100 * p + J)
    A = rs.normal(size=(k, p)) / np.sqrt(p)
    eng = Engine(p, k, J)
    eng.set_problem(A @ rs.normal(size=p), 0.01 * np.eye(k), 100.0 * np.eye(p), np.zeros(p), rs.normal(size=(p, 1)))
    U = 3.0 * rs.normal(size=(p, J))
    return eng, A, U, A @ U, rs.normal(size=(p, J))


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _refused(eng, call, msg, outputs, code=INV):
    """``call()`` returns ``code`` with ``msg`` in the error, every output still holds 7.0, no kernel was launched."""
    torch.cuda.synchronize()
    before = eng.launch_count()
    assert call() == code
    assert msg in eng.lib.ces_last_error(), eng.lib.ces_last_error()
    torch.cuda.synchronize()
    assert eng.launch_count() == before
    for out in outputs:
        if hasattr(out, "cpu"):
            out = out.cpu().numpy()
        elif isinstance(out, ctypes._SimpleCData):
            out = np.array([out.value])
        elif not isinstance(out, np.ndarray):
            out = np.ctypeslib.as_array(out)
        assert (out == 7).all()


def _poisoned_scalars():
    return ctypes.c_double(7.0), (ctypes.c_double * 4)(*[7.0] * 4)


@pytest.mark.parametrize("shape", SHAPES)
def test_whole_step_entry_points_refuse_before_device_work(shape):
    p, k, J = SHAPES[shape]
    eng, _, U, G, xi = _engine(p, k, J)
    lib, h = eng.lib, eng.h
    Ud, Gd, Xd = _dev(U), _dev(G), _dev(xi)
    out = torch.full_like(Ud, 7.0)
    hk, met = _poisoned_scalars()

    def step(rule=ALDI, ts=FROB, form=INTER, U=Ud, G=Gd, xi=Xd, Uout=out):
        ptr = lambda t: _ptr(t) if t is not None else None
        return lib.ces_step(h, rule, ts, 0.0, 1.0, form, ptr(U), J, ptr(G), J, ptr(xi), J, ptr(Uout), J,
                            ctypes.byref(hk), met)

    Uh, Gh, Xh = (np.ascontiguousarray(a) for a in (U, G, xi))
    out_h = np.full((p, J), 7.0)

    def step_host(rule=ALDI, ts=FROB, form=INTER, U=Uh, G=Gh, xi=Xh, Uout=out_h):
        ptr = lambda a: _lib.host_ptr(a) if a is not None else None
        return lib.ces_step_host(h, rule, ts, 0.0, 1.0, form, ptr(U), ptr(G), ptr(xi), ptr(Uout), ctypes.byref(hk), met)

    outputs = (out, out_h, hk, met)
    for entry, name in ((step, b"ces_step"), (step_host, b"ces_step_host")):
        _refused(eng, lambda: entry(ts=KEEP), b"unknown step-size rule", outputs)
        _refused(eng, lambda: entry(ts=BAD_TS), b"unknown step-size rule", outputs)
        _refused(eng, lambda: entry(rule=BAD_RULE), b"unknown update rule 9", outputs)
        _refused(eng, lambda: entry(form=BAD_FORM), b"unknown formulation", outputs)
        _refused(eng, lambda: entry(xi=None), name + b": null pointer", outputs)
        _refused(eng, lambda: entry(Uout=None), name + b": null pointer", outputs)
        _refused(eng, lambda: entry(U=None), name + b": null pointer", outputs)
        assert lib.ces_set_noise(h, _lib.NOISES["ensemble"], 0, 0, None, 0) == 0
        _refused(eng, lambda: entry(form=FACT), b"factored", outputs)
        assert lib.ces_set_noise(h, _lib.NOISES["cholesky"], 0, 0, None, 0) == 0
    # the same settings are accepted where they are legal: eki needs no xi, and with ensemble noise it may be factored
    assert step(rule=EKI, xi=None) == 0 and step_host(rule=EKI, xi=None) == 0
    assert lib.ces_set_noise(h, _lib.NOISES["ensemble"], 0, 0, None, 0) == 0
    assert step(rule=EKI, form=FACT, xi=None) == 0 and step_host(rule=EKI, form=FACT, xi=None) == 0
    eng.close()


@pytest.mark.parametrize("shape", SHAPES)
def test_host_begin_refuses_before_any_upload(shape):
    p, k, J = SHAPES[shape]
    eng, _, U, G, xi = _engine(p, k, J)
    lib, h = eng.lib, eng.h
    nch, bounds = ctypes.c_int(7), (ctypes.c_int64 * 9)(*[7] * 9)

    def begin(rule=ALDI, form=INTER, U=U, G=G):
        ptr = lambda a: _lib.host_ptr(a) if a is not None else None
        return lib.ces_host_begin(h, rule, form, ptr(U), ptr(G), _lib.host_ptr(xi), ctypes.byref(nch), bounds)

    outputs = (nch, bounds)
    _refused(eng, lambda: begin(rule=BAD_RULE), b"unknown update rule", outputs)
    _refused(eng, lambda: begin(form=BAD_FORM), b"unknown formulation", outputs)
    _refused(eng, lambda: begin(G=None), b"ces_host_begin: null pointer", outputs)
    assert lib.ces_set_noise(h, _lib.NOISES["ensemble"], 0, 0, None, 0) == 0
    _refused(eng, lambda: begin(form=FACT), b"factored", outputs)
    eng.close()


def test_small_run_refuses_before_device_work():
    p, k, J = SHAPES["single_cta"]
    eng, A, U, _, _ = _engine(p, k, J)
    lib, h = eng.lib, eng.h
    Ad = _dev(A)
    T = 3
    U0 = np.ascontiguousarray(U)
    Ut, Gt, S, tv = np.full((T + 1, p, J), 7.0), np.full((T + 1, k, J), 7.0), np.full((T, 16), 7.0), np.full(T, 7.0)
    n = ctypes.c_int64(7)

    def run(rule=ALDI, ts=FROB):
        return lib.ces_small_run(h, rule, ts, 0.0, 1.0, _lib.MAPS["lineal"], _ptr(Ad), p, None, None, _lib.host_ptr(U0), None,
                                 0, 0, T, 0.0, 0, 2.0, _lib.host_ptr(Ut), _lib.host_ptr(Gt), _lib.host_ptr(S),
                                 _lib.host_ptr(tv), ctypes.byref(n))

    for kw, msg in (({"rule": BAD_RULE}, b"unknown update rule"), ({"ts": KEEP}, b"unknown step-size rule"),
                    ({"ts": BAD_TS}, b"unknown step-size rule")):
        _refused(eng, lambda: run(**kw), msg, (Ut, Gt, S, tv, n))
    eng.close()


def test_phase_entry_points_keep_their_rules():
    """ces_peek_step_size refuses CES_TS_KEEP; ces_phase4_update refuses a bad step-size rule or a missing operand and
    accepts CES_TS_KEEP; ces_phase3f_products refuses ensemble noise for a noisy rule."""
    p, k, J = SHAPES["phases"]
    eng, _, U, G, xi = _engine(p, k, J)
    lib, h = eng.lib, eng.h
    Ud, Gd, Xd = _dev(U), _dev(G), _dev(xi)
    out = torch.full_like(Ud, 7.0)
    hk, met = _poisoned_scalars()
    assert lib.ces_phase1_sums(h, _ptr(Ud), J, _ptr(Gd), J) == 0
    assert lib.ces_phase2_centre(h, ALDI, _ptr(Ud), J, _ptr(Gd), J) == 0
    assert lib.ces_phase3_interact(h, ALDI, 0) == 0

    def phase4(ts=FROB, xi=Xd, Uout=out):
        ptr = lambda t: _ptr(t) if t is not None else None
        return lib.ces_phase4_update(h, ALDI, ts, 0.0, _ptr(Ud), J, ptr(xi), J, ptr(Uout), J, ctypes.byref(hk), met)

    _refused(eng, lambda: lib.ces_peek_step_size(h, KEEP, 0.0, ctypes.byref(hk)), b"unknown step-size rule", (hk,))
    _refused(eng, lambda: phase4(ts=BAD_TS), b"unknown step-size rule", (out, hk, met))
    _refused(eng, lambda: phase4(xi=None), b"phase4: null pointer", (out, hk, met))
    _refused(eng, lambda: phase4(Uout=None), b"phase4: null pointer", (out, hk, met))
    assert lib.ces_peek_step_size(h, FROB, 0.0, ctypes.byref(hk)) == 0
    h_peeked = hk.value
    assert phase4(ts=KEEP) == 0
    assert hk.value == h_peeked and not bool((out == 7.0).any())
    # the factored products never gather U~, which ensemble noise needs
    assert lib.ces_set_noise(h, _lib.NOISES["ensemble"], 0, 0, None, 0) == 0
    assert lib.ces_phase2_centre(h, ALDI, _ptr(Ud), J, _ptr(Gd), J) == 0
    _refused(eng, lambda: lib.ces_phase3f_products(h, ALDI), b"factored", ())
    eng.close()
