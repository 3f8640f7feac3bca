"""ctypes loader for the CPU oracle (TEST INFRASTRUCTURE ONLY).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
arms may import this module.  The product package never does.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def build(force=False):
    so = os.path.join(_HERE, "liblbfgsb_oracle.so")
    src = os.path.join(_HERE, "lbfgsb_oracle.cpp")
    hdr = os.path.join(_HERE, "..", "include", "lbfgsb_b200_shape.h")
    stale = (not os.path.exists(so)) or any(
        os.path.getmtime(p) > os.path.getmtime(so) for p in (src, hdr) if os.path.exists(p))
    if force or stale:
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return so


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
        _LIB.oracle_set_sum_mode.argtypes = [C.c_int]
        _LIB.oracle_get_sum_mode.restype = C.c_int
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class OracleSetulb:
    """Callable with the host-twin calling convention used by tests/harness.py."""

    def __init__(self, dtype=np.float64):
        self.dtype = np.dtype(dtype)
        self.fn = lib().oracle_setulb_f64 if self.dtype == np.float64 else lib().oracle_setulb_f32
        self.fn.restype = None

    def workspace(self, n, m):
        wa = np.zeros(2 * m * n + 5 * n + 11 * m * m + 8 * m, dtype=self.dtype)
        iwa = np.zeros(3 * n, dtype=np.int32)
        return wa, iwa

    def __call__(self, n, m, x, l, u, nbd, f, g, factr, pgtol, wa, iwa, task, iprint, csave,
                 lsave, isave, dsave):
        n64 = C.c_int64(n)
        m32 = C.c_int32(m)
        ip = C.c_int32(iprint)
        fa = np.array([factr], dtype=self.dtype)
        pg = np.array([pgtol], dtype=self.dtype)
        self.fn(C.byref(n64), C.byref(m32), _p(x), _p(l), _p(u), _p(nbd), _p(f), _p(g), _p(fa),
                _p(pg), _p(wa), _p(iwa), _p(task), C.byref(ip), _p(csave), _p(lsave), _p(isave),
                _p(dsave))

    def active_set_hash(self, n, iwa):
        h = C.c_uint64(0)
        c = C.c_int64(0)
        iwhere = iwa[n:2 * n]
        lib().oracle_active_set_hash(C.c_int64(n), _p(iwhere), C.byref(h), C.byref(c))
        return h.value, c.value

    def release(self, isave):
        pass


def rosenbrock_fg(x, g):
    """test/driver1.f90:274-289 in the reference's summation order."""
    n = x.shape[0]
    if x.dtype == np.float64:
        f = C.c_double(0)
        lib().oracle_rosenbrock_fg_f64(C.c_int64(n), _p(x), C.byref(f), _p(g))
    else:
        f = C.c_float(0)
        lib().oracle_rosenbrock_fg_f32(C.c_int64(n), _p(x), C.byref(f), _p(g))
    return f.value


def set_sum_mode(mode):
    lib().oracle_set_sum_mode(int(mode))


def event_counts(reset=True):
    """[subsm backtracks (:2830), ascent directions (:2247), memory resets ("refresh the lbfgs memory"), skipped
    updates (:826-834), 0, 0, 0, 0] seen by the oracle since the last reset."""
    out = (C.c_longlong * 8)()
    lib().oracle_event_counts(out, C.c_int(1 if reset else 0))
    return list(out)


def set_tie_mode(mode):
    """0: equal breakpoints in hpsolb's heap order (the reference); 1: in variable order (stable sort)."""
    lib().oracle_set_tie_mode(int(mode))
