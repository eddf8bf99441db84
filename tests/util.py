"""Shared generators for the parity tests (seeded, numpy only)."""
from __future__ import annotations

import os
import re

import numpy as np


def cp_path_bits():
    """{name: bit} of the CV_CP_PATH_* launch-path bits of include/cv_b200_debug.h (cv_debug_cp_last_paths)."""
    with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "cv_b200_debug.h")) as f:
        text = f.read()
    return {m.group(1): 1 << int(m.group(2)) for m in re.finditer(r"#define CV_CP_PATH_(\w+)\s+\(1u << (\d+)\)", text)}


def random_hmm(rng, K, M, zero_frac=0.2, alpha=0.5, ties=False):
    """log10 HMM in the reference's layout: logA[K,K] (from,to), logB[K,M], logPi[K].

    zero_frac of the probabilities are forced to 0 (-> -inf as hmm.rs:192-205 does).
    ties=True draws log-probs from a tiny set of dyadic values so that exact f64
    ties (and -0.0/+0.0) occur constantly and the lowest-index rule is exercised.
    """
    if ties:
        vals = np.array([-0.0, 0.0, -0.5, -1.0, -1.5, -2.0, -np.inf])
        A = rng.choice(vals, size=(K, K))
        B = rng.choice(vals, size=(K, M))
        pi = rng.choice(vals, size=K)
        return A, B, pi

    def rows(n, m):
        p = rng.dirichlet(np.full(m, alpha), size=n)
        p[rng.random((n, m)) < zero_frac] = 0.0
        with np.errstate(divide="ignore"):
            return np.log10(p)

    return rows(K, K), rows(K, M), rows(1, K)[0]


def random_batch(rng, B, M, tmin=1, tmax=12):
    lens = rng.integers(tmin, tmax + 1, size=B)
    off = np.zeros(B + 1, dtype=np.int64)
    off[1:] = np.cumsum(lens)
    obs = rng.integers(0, M, size=int(off[-1]), dtype=np.int64).astype(np.uint32)
    return obs, off


def random_superseq(rng, nseq, M, ncomp, p_active, tmin=1, tmax=8):
    """Super-sequence inputs of the CP solver: obs[N], is_seq_start[N], comp[N] (-1 = inactive).
    Component ids are compacted so every id < ncomp_eff has at least one element."""
    lens = rng.integers(tmin, tmax + 1, size=nseq)
    N = int(lens.sum())
    start = np.zeros(N, dtype=np.uint8)
    pos = 0
    for L in lens:
        start[pos] = 1
        pos += int(L)
    obs = rng.integers(0, M, size=N).astype(np.uint32)
    comp = np.full(N, -1, dtype=np.int32)
    if ncomp > 0:
        mask = rng.random(N) < p_active
        comp[mask] = rng.integers(0, ncomp, size=int(mask.sum()))
        used = sorted(set(int(c) for c in comp if c >= 0))
        remap = {c: i for i, c in enumerate(used)}
        comp = np.array([remap[int(c)] if c >= 0 else -1 for c in comp], dtype=np.int32)
        ncomp = len(used)
    return obs, start, comp, ncomp
