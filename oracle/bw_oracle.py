"""ctypes binding of the Baum-Welch CPU oracle (oracle/libbw_oracle.so, bw_oracle.h).

TEST INFRASTRUCTURE ONLY: the checker of cv_baum_welch in tests/, __graft_entry__.smoke() and tools/bw_bench.py.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from .pyoracle import OracleError

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libbw_oracle.so")

_lib = None


def build(force: bool = False) -> str:
    """Compile the oracle with oracle/bw.mk (gcc -O2, no fast-math, no FMA contraction)."""
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(os.path.join(_HERE, "bw_oracle.c")):
        subprocess.check_call(["make", "-C", _HERE, "-f", "bw.mk", "-s", "-B"])
    return _SO


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        dp, u32p, i64p = C.POINTER(C.c_double), C.POINTER(C.c_uint32), C.POINTER(C.c_int64)
        L.cvo_baum_welch.argtypes = [C.c_int, C.c_int64, dp, dp, dp, u32p, i64p, C.c_int64, C.c_int, C.c_double, dp,
                                     C.POINTER(C.c_int), i64p, C.c_int]
        L.cvo_baum_welch.restype = C.c_int
        _lib = L
    return _lib


def _p(a, ty):
    return a.ctypes.data_as(C.POINTER(ty))


def baum_welch(logA, logB, logPi, obs_flat, seq_off, n_iter: int = 1, tol: float = 0.0, nthreads: int = 1):
    """Baum-Welch with the semantics of cv_baum_welch, in log space.  Returns dict(a, b, pi (log10), loglik[iters],
    iters, skipped (last iteration)).  OracleError(code) on a bad input (codes of cv_oracle.h)."""
    a = np.array(logA, dtype=np.float64, order="C")
    b = np.array(logB, dtype=np.float64, order="C")
    pi = np.array(logPi, dtype=np.float64, order="C")
    K, M = b.shape
    obs = np.ascontiguousarray(obs_flat, dtype=np.uint32)
    off = np.ascontiguousarray(seq_off, dtype=np.int64)
    ll = np.zeros(max(n_iter, 1), dtype=np.float64)
    iters, skipped = C.c_int(0), C.c_int64(0)
    rc = lib().cvo_baum_welch(K, M, _p(a, C.c_double), _p(b, C.c_double), _p(pi, C.c_double), _p(obs, C.c_uint32),
                              _p(off, C.c_int64), len(off) - 1, int(n_iter), float(tol), _p(ll, C.c_double),
                              C.byref(iters), C.byref(skipped), int(nthreads))
    if rc:
        raise OracleError(rc)
    return dict(a=a, b=b, pi=pi, loglik=ll[: iters.value], iters=iters.value, skipped=skipped.value)
