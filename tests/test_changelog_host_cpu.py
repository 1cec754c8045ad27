"""The host-fed change-log entry points (lstep_pe_step_changelog_host, lstep_pe_steps_changelog_host) reject a NULL stepper,
stream descriptor or change log with LSTEP_ERR_INVALID_ARG before they touch a device."""
import ctypes

from lstep_b200 import _lib

INVALID_ARG = 1


def _step(lib, h, s, cl):
    ticket = ctypes.c_int64(-1)
    src = (ctypes.c_int64 * 4)(1, 2, 3, 4)
    t = (ctypes.c_double * 4)(1.0, 2.0, 3.0, 4.0)
    return lib.lstep_pe_step_changelog_host(h, s, cl, _lib.CSR(), 4, src, src, t, None, 0, 0, 0, None, None, 0, None, 20, _lib.PEMLP(),
                                            _lib.PEMLP(), None, 0, None, None, ctypes.byref(ticket))


def _steps(lib, h, s, cl):
    head, ln, done = ctypes.c_int(0), ctypes.c_int(100), ctypes.c_int64(-1)
    src = (ctypes.c_int64 * 4)(1, 2, 3, 4)
    t = (ctypes.c_double * 4)(1.0, 2.0, 3.0, 4.0)
    res = (ctypes.c_float * 4)()
    rc = lib.lstep_pe_steps_changelog_host(h, s, cl, _lib.CSR(), 4, 4, src, src, t, None, 0, ctypes.byref(head), ctypes.byref(ln), None, 20,
                                           _lib.PEMLP(), _lib.PEMLP(), None, 0, None, None, res, ctypes.byref(done))
    assert done.value == 0 and head.value == 0
    return rc


def test_changelog_host_entry_points_reject_null_arguments():
    lib = _lib.load(require_device=False)
    desc, cl = _lib.PEStreamDesc(), _lib.ChangeLog()
    # (a non-NULL stepper is never dereferenced once another argument is NULL)
    not_null = ctypes.c_void_p(8)
    for fn in (_step, _steps):
        assert fn(lib, None, desc, cl) == INVALID_ARG
        assert fn(lib, not_null, None, cl) == INVALID_ARG
        assert fn(lib, not_null, desc, None) == INVALID_ARG
