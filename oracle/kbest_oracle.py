"""ctypes binding of the k-best Viterbi CPU oracle (oracle/libkbest_oracle.so, kbest_oracle.h).

TEST INFRASTRUCTURE ONLY: the checker of cv_decode_batch_kbest in tests/, __graft_entry__.smoke() and
tools/kbest_bench.py.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from .pyoracle import OracleError

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libkbest_oracle.so")

_lib = None


def build(force: bool = False) -> str:
    """Compile the oracle with oracle/kbest.mk (gcc -O2, no fast-math, no FMA contraction)."""
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(os.path.join(_HERE, "kbest_oracle.c")):
        subprocess.check_call(["make", "-C", _HERE, "-f", "kbest.mk", "-s", "-B"])
    return _SO


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        dp, u32p, i64p = C.POINTER(C.c_double), C.POINTER(C.c_uint32), C.POINTER(C.c_int64)
        L.cvo_decode_batch_kbest.argtypes = [C.c_int, C.c_int64, dp, dp, u32p, i64p, C.c_int64, C.c_int, u32p, dp, C.c_int]
        L.cvo_decode_batch_kbest.restype = C.c_int
        _lib = L
    return _lib


def _p(a, ty):
    return a.ctypes.data_as(C.POINTER(ty))


def decode_batch_kbest(logA, logB, obs_flat, seq_off, k: int, nthreads: int = 1):
    """k-best Viterbi with the contract of cv_decode_batch_kbest.  Returns (paths u32[k, N], scores f64[k, B]);
    OracleError(code) on a bad input."""
    a = np.ascontiguousarray(logA, dtype=np.float64)
    K = a.shape[0]
    b = np.ascontiguousarray(logB, dtype=np.float64).reshape(K, -1)
    obs = np.ascontiguousarray(obs_flat, dtype=np.uint32)
    off = np.ascontiguousarray(seq_off, dtype=np.int64)
    B = len(off) - 1
    paths = np.zeros((max(int(k), 1), len(obs)), dtype=np.uint32)
    scores = np.zeros((max(int(k), 1), B), dtype=np.float64)
    rc = lib().cvo_decode_batch_kbest(K, b.shape[1], _p(a, C.c_double), _p(b, C.c_double), _p(obs, C.c_uint32),
                                      _p(off, C.c_int64), B, int(k), _p(paths, C.c_uint32), _p(scores, C.c_double),
                                      int(nthreads))
    if rc:
        raise OracleError(rc)
    return paths, scores
