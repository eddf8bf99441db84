"""ctypes binding of the forward-backward CPU oracle (oracle/libfb_oracle.so, fb_oracle.h).

TEST INFRASTRUCTURE ONLY: the checker of cv_loglik_batch / cv_posterior_batch in tests/, __graft_entry__.smoke() and
tools/fb_bench.py.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from .pyoracle import OracleError

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libfb_oracle.so")

_lib = None


def build(force: bool = False) -> str:
    """Compile the oracle with oracle/fb.mk (gcc -O2, no fast-math, no FMA contraction)."""
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(os.path.join(_HERE, "fb_oracle.c")):
        subprocess.check_call(["make", "-C", _HERE, "-f", "fb.mk", "-s", "-B"])
    return _SO


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        dp, u32p, i64p = C.POINTER(C.c_double), C.POINTER(C.c_uint32), C.POINTER(C.c_int64)
        L.cvo_forward_backward.argtypes = [C.c_int, C.c_int64, dp, dp, dp, u32p, i64p, C.c_int64, dp, dp, C.c_int]
        L.cvo_forward_backward.restype = C.c_int
        _lib = L
    return _lib


def _p(a, ty):
    return a.ctypes.data_as(C.POINTER(ty))


def forward_backward(logA, logB, logPi, obs_flat, seq_off, nthreads: int = 1, want_posteriors: bool = True):
    """Forward-backward with the semantics of cv_posterior_batch, in log space.  Returns dict(loglik f64[B] (log10,
    -inf for P(O) = 0), post f64[N, K] (rows of 0.0 for P(O) = 0) or None).  OracleError(code) on a bad input."""
    a = np.ascontiguousarray(logA, dtype=np.float64)
    b = np.ascontiguousarray(logB, dtype=np.float64)
    pi = np.ascontiguousarray(logPi, dtype=np.float64)
    K = a.shape[0]
    b = b.reshape(K, -1)
    M = b.shape[1]
    obs = np.ascontiguousarray(obs_flat, dtype=np.uint32)
    off = np.ascontiguousarray(seq_off, dtype=np.int64)
    B = len(off) - 1
    ll = np.zeros(B, dtype=np.float64)
    post = np.zeros((len(obs), K), dtype=np.float64) if want_posteriors else None
    rc = lib().cvo_forward_backward(K, M, _p(a, C.c_double), _p(b, C.c_double), _p(pi, C.c_double), _p(obs, C.c_uint32),
                                    _p(off, C.c_int64), B, _p(ll, C.c_double),
                                    _p(post, C.c_double) if post is not None else None, int(nthreads))
    if rc:
        raise OracleError(rc)
    return dict(loglik=ll, post=post)
