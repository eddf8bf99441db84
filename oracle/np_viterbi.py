"""Vectorized numpy restatement of viterbi::decode (src/viterbi_solver/viterbi.rs:5-32), generic in the float type.

TEST INFRASTRUCTURE ONLY (the product package never imports it).  With dtype=np.float64 it is the reference's
arithmetic and equals the C oracle (cv_oracle.c) bit for bit; with dtype=np.float32 it is the contract of the f32
decode mode (include/cv_b200.h, cv_decode_batch_f32):
  - the model is rounded to the float type once (astype: round to nearest even, as __double2float_rn);
  - candidates fl(delta[t-1][j] + a[j][i]), first maximum (np.argmax), then fl(best + b[i][o_t]);
  - an emission of -inf writes -inf and psi = 0 (viterbi.rs:12-21); delta[0] = 0 (pi and o_0 unused);
  - end state = first maximum of delta[T-1]; score = delta[T-1][end] widened to f64.
Sequences are processed longest first in sub-batches, all still-active sequences of a sub-batch as one
[b, K(to), K(from)] block per step: about 10 k sequences a second at K = 64.
"""
from __future__ import annotations

import numpy as np

_MAX_SEQS = 2048            # sequences per sub-batch
_MAX_PSI_CELLS = 1 << 26    # backpointers held per sub-batch (elements x K)


def decode_batch(logA, logB, obs_flat, seq_off, dtype=np.float64):
    """B independent viterbi::decode calls in `dtype` arithmetic. Returns (paths u32[N], scores f64[B]).

    ValueError where the reference panics: an empty sequence, an observation >= M, NaN in an argmax."""
    dtype = np.dtype(dtype).type
    aT = np.ascontiguousarray(np.asarray(logA, dtype=np.float64).astype(dtype).T)   # aT[to][from]
    b = np.asarray(logB, dtype=np.float64).astype(dtype)                              # b[state][obs]
    K, M = b.shape
    bT = np.ascontiguousarray(b.T)                                                    # bT[obs][state]
    obs = np.ascontiguousarray(obs_flat, dtype=np.int64)
    off = np.ascontiguousarray(seq_off, dtype=np.int64)
    B, N = off.shape[0] - 1, obs.shape[0]
    lens = np.diff(off)
    if B > 0 and (lens <= 0).any():
        raise ValueError("empty sequence")
    if N and (obs.min() < 0 or obs.max() >= M):
        raise ValueError("observation >= M")
    paths = np.zeros(N, dtype=np.uint32)
    scores = np.zeros(B, dtype=np.float64)
    order = np.argsort(-lens, kind="stable")                                          # longest first

    c0 = 0
    with np.errstate(over="ignore", invalid="ignore"):      # overflow to +-inf is part of the arithmetic restated
        while c0 < B:
            c0 = _sub_batch(aT, bT, obs, off, lens, order, c0, dtype, paths, scores)
    return paths, scores


def _sub_batch(aT, bT, obs, off, lens, order, c0, dtype, paths, scores):
    """Decode the sequences order[c0:c1] (one sub-batch) into paths / scores; returns c1."""
    K = aT.shape[0]
    neg = dtype(-np.inf)
    psi_t = np.uint8 if K <= 256 else np.uint32
    # at most _MAX_SEQS sequences and _MAX_PSI_CELLS backpointers, at least one sequence
    cells = np.cumsum(lens[order[c0:c0 + _MAX_SEQS]]) * K
    c1 = c0 + max(1, int(np.searchsorted(cells, _MAX_PSI_CELLS, side="right")))
    idx = order[c0:c1]
    L, start = lens[idx], off[idx]
    n, Tmax = idx.shape[0], int(L[0])
    active = np.searchsorted(-L, -np.arange(Tmax), side="left")                  # active[t] = #{L > t}
    delta = np.zeros((n, K), dtype=dtype)                                         # viterbi.rs:6
    psi = [None] * Tmax
    for t in range(1, Tmax):                                                      # viterbi.rs:9
        na = int(active[t])
        cand = delta[:na, None, :] + aT[None, :, :]                               # [na, to, from], viterbi.rs:15
        e = bT[obs[start[:na] + t]]                                               # [na, to], viterbi.rs:11
        dead = e == neg                                                           # viterbi.rs:12,19-21
        if np.isnan(cand).any(axis=2)[~dead].any():
            raise ValueError("NaN in an argmax (viterbi.rs:16)")
        j = cand.argmax(axis=2)                                                   # first maximum, viterbi.rs:16
        best = np.take_along_axis(cand, j[:, :, None], axis=2)[:, :, 0]
        new = best + e                                                            # viterbi.rs:17
        new[dead] = neg
        j[dead] = 0
        delta[:na] = new
        psi[t] = j.astype(psi_t)
    if np.isnan(delta).any():
        raise ValueError("NaN in an argmax (viterbi.rs:24)")
    cur = delta.argmax(axis=1)                                                    # viterbi.rs:24
    scores[idx] = delta[np.arange(n), cur].astype(np.float64)
    for t in range(Tmax - 1, -1, -1):                                             # viterbi.rs:26-30
        na = int(active[t])
        paths[start[:na] + t] = cur[:na]
        if t > 0:
            cur[:na] = psi[t][np.arange(na), cur[:na]]
    return c1
