"""Scratch GPU probe: FP64 issue peak (cv_debug_probe_fp64 modes 0, 1, 25) and a quick POS-shape timing."""
import ctypes as C
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import consistent_viterbi_b200 as cv
from util import random_hmm

L = cv._lib.lib()
out = {}
for mode, iters in [(0, 20000), (1, 20000), (25, 20000)]:
    ops, ms = C.c_double(), C.c_double()
    cv._lib.check(L.cv_debug_probe_fp64(0, mode, iters, C.byref(ops), C.byref(ms)))
    out[f"probe_mode{mode}"] = {"fp64_ops_per_s": ops.value, "ms": ms.value}
    print(mode, f"{ops.value:.4e} fp64 ops/s  {ms.value:.3f} ms", flush=True)

rng = np.random.default_rng(3019)
K, M = 45, 20000
Bn = int(os.environ.get("POS_B", "200000"))
A, B, pi = random_hmm(rng, K, M, zero_frac=0.05, alpha=0.1)
lens = np.clip(np.rint(rng.gamma(2.5, 10.0, size=Bn)), 1, 200).astype(np.int64)
off = np.zeros(Bn + 1, dtype=np.int64); off[1:] = np.cumsum(lens)
obs = (rng.zipf(1.1, size=int(off[-1])) % M).astype(np.uint32)
cells = float(((lens - 1) * K * K).sum())
h = cv.HMM(A, B, pi)
L.cv_set_timing(1)
for it in range(3):
    t0 = time.perf_counter()
    paths, scores = cv.decode_batch(h, obs, off)
    t1 = time.perf_counter()
    kms = L.cv_last_kernel_ms(h.device_handle())
    bms = L.cv_last_backtrace_ms(h.device_handle())
print(f"POS B={Bn} cells={cells:.3e} e2e {1e3*(t1-t0):.2f} ms  fwd {kms:.3f} ms bt {bms:.3f} ms -> fwd {cells/kms/1e-3:.3e} total {cells/(kms+bms)/1e-3:.3e} cells/s", flush=True)
out["pos"] = {"B": Bn, "cells": cells, "kernel_ms": kms, "backtrace_ms": bms}
os.makedirs("gpurun_out", exist_ok=True)
json.dump(out, open("gpurun_out/probe.json", "w"), indent=1)
