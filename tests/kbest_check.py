"""Brute-force checks of a k-best Viterbi result (cv_decode_batch_kbest's contract) by enumerating every path."""
from __future__ import annotations

import itertools

import numpy as np

NO_PATH = 0xFFFFFFFF


def path_score(A, Bm, o, path):
    """the contract's score of one path: v_0 = 0, v_t = fl(fl(v_{t-1} + a[s_{t-1}][s_t]) + b[s_t][o_t])"""
    v = np.float64(0.0)
    for t in range(1, len(path)):
        v = (v + A[path[t - 1], path[t]]) + Bm[path[t], o[t]]
    return v


def all_scores(A, Bm, o):
    """scores of all K^T paths (numpy adds are binary64 adds in the contract's order)"""
    K, T = A.shape[0], len(o)
    paths = np.array(list(itertools.product(range(K), repeat=T)), dtype=np.int64).reshape(-1, T)
    v = np.zeros(len(paths))
    for t in range(1, T):
        v = (v + A[paths[:, t - 1], paths[:, t]]) + Bm[paths[:, t], o[t]]
    return v


def check_against_enumeration(A, Bm, obs, off, k, paths, scores, ref_path=None, ref_score=None):
    """paths u32[k, N], scores f64[k, B] of a k-best call on (A, Bm) against enumeration of every sequence's paths;
    ref_path / ref_score: the plain decode's outputs, which rank 0 must equal byte for byte."""
    Bm = Bm.reshape(A.shape[0], -1)
    K = A.shape[0]
    for b in range(len(off) - 1):
        o = obs[off[b]:off[b + 1]]
        T = len(o)
        npaths = min(k, K ** T)
        got = scores[:, b]
        assert (got[npaths:] == -np.inf).all() and (paths[npaths:, off[b]:off[b + 1]] == NO_PATH).all()
        assert (paths[:npaths, off[b]:off[b + 1]] < K).all()
        allv = np.sort(all_scores(A, Bm, o))[::-1][:npaths]
        assert (got[:npaths] == allv).all(), (b, got[:npaths], allv)            # top-k multiset (-0.0 == +0.0)
        assert (got[1:npaths] <= got[:npaths - 1]).all()
        seen = set()
        for r in range(npaths):
            p = paths[r, off[b]:off[b + 1]]
            assert np.float64(path_score(A, Bm, o, p)).tobytes() == np.float64(got[r]).tobytes(), (b, r)
            seen.add(p.tobytes())
        assert len(seen) == npaths
        if ref_path is not None:
            assert paths[0, off[b]:off[b + 1]].tobytes() == ref_path[off[b]:off[b + 1]].tobytes()
            assert np.float64(got[0]).tobytes() == np.float64(ref_score[b]).tobytes()
