"""cv_decode_batch_kbest (decode_batch_kbest / decode_kbest) against the k-best C oracle (cvo_decode_batch_kbest), byte
for byte: K = 1 .. 64 over every list capacity, random / tie-heavy / -inf-heavy / positive-entry / 2-D bdims models;
rank 0 against cv_decode_batch; brute-force enumeration on tiny shapes; lengths up to 5 000; 100 k POS-shape sentences;
independence of the batch, its order and the chunking; determinism; every status."""
import numpy as np
import pytest

import bench
import consistent_viterbi_b200 as cv
from kbest_check import NO_PATH, check_against_enumeration
from oracle import kbest_oracle as kbo
from util import random_batch, random_hmm

pytestmark = pytest.mark.gpu

KINDS = ["random", "ties", "neginf", "positive", "bdims"]


def _model(rng, K, M, kind):
    """(A, Bm, pi, bdims) of one model kind; "neginf" also makes the last symbol impossible in every state"""
    if kind == "ties":
        A, Bm, pi = random_hmm(rng, K, M, ties=True)
    else:
        A, Bm, pi = random_hmm(rng, K, M, zero_frac=0.4 if kind == "neginf" else 0.1)
    if kind == "neginf":
        Bm[:, M - 1] = -np.inf
    if kind == "positive":                          # any model cv_hmm_create accepts: positive entries too
        A = A + rng.uniform(0.0, 3.0, A.shape)
        Bm = Bm + rng.uniform(0.0, 3.0, Bm.shape)
    return A, Bm, pi, ((3, M // 3) if kind == "bdims" else None)


def _hmm(A, Bm, pi, bdims=None):
    K = A.shape[0]
    return cv.HMM(A.copy(), (Bm.reshape((K,) + tuple(bdims)) if bdims else Bm).copy(), pi.copy())


def _same(x, y):
    return x[0].tobytes() == y[0].tobytes() and x[1].tobytes() == y[1].tobytes()


@pytest.mark.parametrize("k", [1, 2, 5, 8, 16, 32])
@pytest.mark.parametrize("K", [1, 2, 3, 8, 13, 32, 33, 45, 64])
def test_matches_oracle(K, k):
    rng = np.random.default_rng(1000 * K + k)
    M = 12
    npos = max(300, int(6e6 // (K * K * k)))        # the oracle orders all K k candidates of every (t, i)
    for kind in KINDS:
        A, Bm, pi, bdims = _model(rng, K, M, kind)
        tmax = min(60, max(2, npos // 20))
        obs, off = random_batch(rng, max(4, npos // ((tmax + 1) // 2)), M, 1, tmax)
        if kind == "neginf":
            obs[off[1] + (off[2] - off[1]) // 2] = M - 1      # a fully impossible sequence
        h = _hmm(A, Bm, pi, bdims)
        got = cv.decode_batch_kbest(h, obs, off, k, device=0)
        ref = kbo.decode_batch_kbest(A, Bm, obs, off, k, nthreads=8)
        assert _same(got, ref), kind
        dp, ds = cv.decode_batch(h, obs, off, device=0)
        assert got[0][0].tobytes() == dp.tobytes() and got[1][0].tobytes() == ds.tobytes(), kind
        if kind == "neginf":
            assert got[1][0, 1] == -np.inf
        h.close()


def test_k1_is_the_plain_decode():
    rng = np.random.default_rng(5)
    for K in (4, 45, 64):
        A, Bm, pi = random_hmm(rng, K, 50, zero_frac=0.2)
        obs, off = random_batch(rng, 3000, 50, 1, 80)
        h = cv.HMM(A, Bm, pi)
        paths, scores = cv.decode_batch_kbest(h, obs, off, 1, device=0)
        dp, ds = cv.decode_batch(h, obs, off, device=0)
        assert paths.shape == (1, len(obs)) and paths[0].tobytes() == dp.tobytes() and scores[0].tobytes() == ds.tobytes()
        h.close()


@pytest.mark.parametrize("kind", ["random", "ties", "neginf"])
@pytest.mark.parametrize("K", [1, 2, 3, 4])
def test_enumeration_tiny(K, kind):
    rng = np.random.default_rng(77 * K + len(kind))
    M = 5
    A, Bm, pi, _ = _model(rng, K, M, kind)
    tmax = 6 if K == 4 else 7
    lens = np.concatenate([np.arange(1, tmax + 1), rng.integers(1, tmax + 1, size=6)])
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    obs = rng.integers(0, M, size=int(off[-1])).astype(np.uint32)
    h = cv.HMM(A, Bm, pi)
    dp, ds = cv.decode_batch(h, obs, off, device=0)
    for k in (1, 2, 3, 5, 8, 13, 16, 17, 31, 32):
        paths, scores = cv.decode_batch_kbest(h, obs, off, k, device=0)
        check_against_enumeration(A, Bm, obs, off, k, paths, scores, dp, ds)
    h.close()


def test_lengths_1_to_5000():
    rng = np.random.default_rng(9)
    K, M = 13, 40
    A, Bm, pi = random_hmm(rng, K, M, zero_frac=0.2)
    lens = np.array([1, 2, 3, 7, 33, 100, 1000, 5000, 2500, 1])
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    obs = rng.integers(0, M, size=int(off[-1])).astype(np.uint32)
    h = cv.HMM(A, Bm, pi)
    for k in (5, 8, 32):
        assert _same(cv.decode_batch_kbest(h, obs, off, k, device=0), kbo.decode_batch_kbest(A, Bm, obs, off, k, nthreads=8))
    h.close()


def test_pos_shape_100k_against_threaded_oracle():
    w = bench.workload_pos(0, 100_000)
    h = cv.HMM(w["A"], w["B"], w["pi"])
    got = cv.decode_batch_kbest(h, w["obs"], w["off"], 8, device=0)
    ref = kbo.decode_batch_kbest(w["A"], w["B"], w["obs"], w["off"], 8, nthreads=64)
    assert _same(got, ref)
    h.close()


def test_batch_order_and_chunking_do_not_matter():
    rng = np.random.default_rng(11)
    K, M, k = 45, 30, 8
    A, Bm, pi = random_hmm(rng, K, M, zero_frac=0.2)
    obs, off = random_batch(rng, 5000, M, 1, 60)
    h = cv.HMM(A, Bm, pi)
    L = cv._lib.lib()
    full = cv.decode_batch_kbest(h, obs, off, k, device=0)
    assert _same(full, cv.decode_batch_kbest(h, obs, off, k, device=0))            # two calls, same bytes
    lens = np.diff(off)
    for b in (0, 1234, 4999):                                                        # decoded alone
        alone = cv.decode_batch_kbest(h, obs[off[b]:off[b + 1]], np.array([0, lens[b]]), k, device=0)
        assert alone[0].tobytes() == full[0][:, off[b]:off[b + 1]].tobytes()
        assert alone[1][:, 0].tobytes() == full[1][:, b].tobytes()
    rev = np.arange(len(lens))[::-1]                                                 # reversed order
    obs_r = np.concatenate([obs[off[b]:off[b + 1]] for b in rev])
    off_r = np.concatenate([[0], np.cumsum(lens[rev])]).astype(np.int64)
    pr, sr = cv.decode_batch_kbest(h, obs_r, off_r, k, device=0)
    pos = np.concatenate([np.arange(off[b], off[b + 1]) for b in rev])
    assert pr.tobytes() == full[0][:, pos].tobytes() and sr.tobytes() == full[1][:, rev].tobytes()
    try:
        for n in (1, 7, 1000):                                                       # forced chunk sizes
            L.cv_debug_set_kbest_chunk_seqs(n)
            src = (obs[: off[600]], off[:601]) if n == 1 else (obs, off)
            got = cv.decode_batch_kbest(h, *src, k, device=0)
            want = (full[0][:, : src[1][-1]], full[1][:, : len(src[1]) - 1])
            assert got[0].tobytes() == np.ascontiguousarray(want[0]).tobytes()
            assert got[1].tobytes() == np.ascontiguousarray(want[1]).tobytes()
    finally:
        L.cv_debug_set_kbest_chunk_seqs(0)
    h.close()


def test_decode_kbest_single_sequence():
    rng = np.random.default_rng(12)
    A, Bm, pi = random_hmm(rng, 3, 6, zero_frac=0.0)
    h = cv.HMM(A, Bm.reshape(3, 2, 3), pi)
    seq = [[0, 1], [1, 2], [0, 0]]
    res = cv.decode_kbest(seq, h, 32, device=0)
    assert len(res) == 27                                                            # 3^3 paths, no "no path" rank
    obs = h.flatten_obs(seq)
    paths, scores = cv.decode_batch_kbest(h, obs, np.array([0, 3]), 32, device=0)
    for r, (p, s) in enumerate(res):
        assert p.dtype == np.uint64 and (p == paths[r]).all() and s == scores[r, 0]
    assert (res[0][0] == cv.decode(seq, h, device=0)).all()
    h.close()


def test_statuses():
    rng = np.random.default_rng(13)
    A, Bm, pi = random_hmm(rng, 5, 7)
    h = cv.HMM(A, Bm, pi)
    L = cv._lib.lib()
    hd = h.device_handle(0)
    obs, off = random_batch(rng, 4, 7, 1, 5)
    paths = np.zeros((4, len(obs)), dtype=np.uint32)
    scores = np.zeros((4, 4))

    def call(hh=hd, o=obs, so=off, B=4, k=4, p=paths, s=scores):
        ptr = lambda a: a.ctypes.data if isinstance(a, np.ndarray) else a
        return L.cv_decode_batch_kbest(hh, ptr(o), ptr(so), B, k, ptr(p), ptr(s))

    before = paths.copy()
    assert call(B=0) == 0 and (paths == before).all()
    assert call(hh=None) == 3 and call(o=None) == 3 and call(so=None) == 3 and call(p=None) == 3
    assert call(s=None) == 0
    assert call(so=off + 1) == 3
    assert call(k=0) == 3 and call(k=-1) == 3
    assert call(k=33) == 7
    bad = obs.copy()
    bad[-1] = 7
    assert call(o=bad) == 3
    empty = off.copy()
    empty[2] = empty[1]
    assert call(so=empty) == 1
    with pytest.raises(cv.CvError):
        cv.decode_batch_kbest(h, obs, off, 0, device=0)
    h.close()
    A, Bm, pi = random_hmm(rng, 65, 7)
    big = cv.HMM(A, Bm, pi)
    with pytest.raises(cv.CvError) as e:
        cv.decode_batch_kbest(big, obs, off, 2, device=0)
    assert e.value.code == 7
    big.close()
