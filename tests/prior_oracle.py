"""ctypes binding of tests/priororacle (the oracle's RANSAC / estimator started from a prior), built on first use with the
oracle's flags.  TEST INFRASTRUCTURE ONLY; the structures are oracle.port's."""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle import port

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "priororacle", "prior_oracle.c")
SO = os.path.join(HERE, "priororacle", "libprior_oracle.so")
ORACLE_SRC = os.path.join(os.path.dirname(HERE), "oracle", "repose_oracle.c")
DP = C.POINTER(C.c_double)

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(SO) or os.path.getmtime(SO) < max(os.path.getmtime(SRC), os.path.getmtime(ORACLE_SRC)):
            subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off",
                                   "-fvisibility=hidden", "-Wall", "-Wno-unused-function", "-o", SO, SRC, "-lm"])
        L = C.CDLL(SO)
        L.ro_ransac_prior.restype = None
        L.ro_ransac_prior.argtypes = [C.c_int, DP, DP, DP, DP, C.c_size_t, C.POINTER(port.RansacOpt),
                                      C.POINTER(port.Model), C.POINTER(port.Model), C.POINTER(port.RansacStats),
                                      C.c_char_p]
        L.ro_estimate_prior.restype = None
        L.ro_estimate_prior.argtypes = [C.c_int, DP, DP, DP, DP, C.c_size_t, DP, DP, C.POINTER(port.RansacOpt),
                                        C.POINTER(port.BundleOpt), C.POINTER(port.Model), C.POINTER(port.Model),
                                        C.POINTER(port.RansacStats), C.c_char_p]
        _lib = L
    return _lib


def _d(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _p(a):
    return a.ctypes.data_as(DP)


def ransac(variant, x1, x2, d1, d2, ropt, prior=None):
    """port.ransac with an optional prior (port.Model, normalised frame) scored and locally optimised before the first
    iteration."""
    x1, x2, d1, d2 = _d(x1), _d(x2), _d(d1), _d(d2)
    m = port.make_model()
    st = port.RansacStats()
    buf = C.create_string_buffer(max(len(x1), 1))
    lib().ro_ransac_prior(variant, _p(x1), _p(x2), _p(d1), _p(d2), len(x1), C.byref(ropt),
                          C.byref(prior) if prior is not None else None, C.byref(m), C.byref(st), buf)
    return m, st, np.frombuffer(buf.raw, dtype=np.uint8)[:len(x1)].astype(bool)


def estimate(variant, x1, x2, d1, d2, cam1, cam2, ropt, bopt, prior=None):
    """port.estimate with an optional prior (port.Model in the caller's frame: the focal variants' f1, f2 in pixels)."""
    x1, x2, d1, d2 = _d(x1), _d(x2), _d(d1), _d(d2)
    c1 = _d(cam1 if cam1 is not None else [1, 1, 0, 0])
    c2 = _d(cam2 if cam2 is not None else [1, 1, 0, 0])
    m = port.make_model()
    st = port.RansacStats()
    buf = C.create_string_buffer(max(len(x1), 1))
    lib().ro_estimate_prior(variant, _p(x1), _p(x2), _p(d1), _p(d2), len(x1), _p(c1), _p(c2), C.byref(ropt),
                            C.byref(bopt), C.byref(prior) if prior is not None else None, C.byref(m), C.byref(st), buf)
    return m, st, np.frombuffer(buf.raw, dtype=np.uint8)[:len(x1)].astype(bool)
