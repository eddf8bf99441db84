"""Run one FP64 probe mode (cv_debug_probe_fp64: 0, 1 or 25) in a process of its own: python tools/probe_only.py MODE ITERS"""
import ctypes as C
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import consistent_viterbi_b200 as cv

L = cv._lib.lib()
mode, iters = int(sys.argv[1]), int(sys.argv[2])
ops, ms = C.c_double(), C.c_double()
cv._lib.check(L.cv_debug_probe_fp64(0, mode, iters, C.byref(ops), C.byref(ms)))
print(mode, f"{ops.value:.4e} fp64 ops/s {ms.value:.3f} ms")
