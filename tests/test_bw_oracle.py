"""CPU tests of the Baum-Welch oracle (oracle/bw_oracle.c, the checker of cv_baum_welch): against
brute-force path enumeration, against the supervised MLE when every posterior is one-hot, monotone log-likelihood;
and the product's refusal to train without a device."""
import itertools

import numpy as np
import pytest

import consistent_viterbi_b200 as cv
from oracle import bw_oracle as bwo
from oracle import pyoracle as po
from util import random_hmm


def _p(x):
    with np.errstate(over="ignore"):
        return np.where(np.isneginf(x), 0.0, 10.0 ** np.asarray(x, dtype=np.float64))


def _brute(logA, logB, logPi, obs, off):
    """One EM iteration from explicit sums over all K^T paths."""
    A, Bm, pi = _p(logA), _p(logB), _p(logPi)
    K, M = Bm.shape
    xi, g_a, g_b, g0, em = np.zeros((K, K)), np.zeros(K), np.zeros(K), np.zeros(K), np.zeros((K, M))
    ll, skipped = 0.0, 0
    for i in range(len(off) - 1):
        o = obs[off[i]:off[i + 1]]
        T = len(o)
        paths, probs = list(itertools.product(range(K), repeat=T)), []
        for s in paths:
            pr = pi[s[0]] * Bm[s[0], o[0]]
            for t in range(1, T):
                pr *= A[s[t - 1], s[t]] * Bm[s[t], o[t]]
            probs.append(pr)
        P = sum(probs)
        if P == 0.0:
            skipped += 1
            continue
        ll += np.log10(P)
        for s, pr in zip(paths, probs):
            w = pr / P
            g0[s[0]] += w
            for t in range(T):
                g_b[s[t]] += w
                em[s[t], o[t]] += w
                if t < T - 1:
                    g_a[s[t]] += w
                if t >= 1:
                    xi[s[t - 1], s[t]] += w
    nc = len(off) - 1 - skipped
    with np.errstate(divide="ignore", invalid="ignore"):
        a = np.where(g_a[:, None] > 0, xi / g_a[:, None], 0.0)
        b = np.where(g_b[:, None] > 0, em / g_b[:, None], 0.0)
        p = g0 / nc if nc else np.zeros(K)
        return np.log10(a), np.log10(b), np.log10(p), ll, skipped


def _close(x, y, rtol):
    x, y = np.asarray(x), np.asarray(y)
    assert (np.isneginf(x) == np.isneginf(y)).all()
    f = ~np.isneginf(x)
    np.testing.assert_allclose(_p(x[f]), _p(y[f]), rtol=rtol, atol=0)


@pytest.mark.parametrize("K,seed", [(1, 0), (2, 1), (3, 2), (3, 3)])
def test_oracle_against_enumeration(K, seed):
    rng = np.random.default_rng(seed)
    M = 4
    A, Bm, pi = random_hmm(rng, K, M, zero_frac=0.25)
    Bm[:, 3] = -np.inf                                  # observation 3 impossible: its sequence has P(O) = 0
    lens = [1, 2, 6, 3, 1, 5, 4]
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    obs = rng.integers(0, 3, int(off[-1])).astype(np.uint32)
    obs[off[3] + 1] = 3
    ref = _brute(A, Bm, pi, obs, off)
    got = bwo.baum_welch(A, Bm, pi, obs, off, n_iter=1, nthreads=3)
    _close(got["a"], ref[0], 1e-12)
    _close(got["b"], ref[1], 1e-12)
    _close(got["pi"], ref[2], 1e-12)
    assert got["loglik"][0] == pytest.approx(ref[3], rel=1e-12)
    assert got["skipped"] == ref[4] >= 1
    assert np.isneginf(got["b"][:, 3]).all()


def test_one_hot_posteriors_equal_mle():
    """Every observation is emittable by exactly one state: posteriors are one-hot and one EM iteration is the
    supervised estimate of the tags that observation implies."""
    rng = np.random.default_rng(7)
    K, per = 4, 3
    M = K * per
    owner = np.repeat(np.arange(K), per)
    A, _, pi = random_hmm(rng, K, M, zero_frac=0.0)
    Bm = np.full((K, M), -np.inf)
    for m in range(M):
        Bm[owner[m], m] = np.log10(rng.uniform(0.05, 1.0))
    lens = rng.integers(1, 9, 40)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    obs = rng.integers(0, M, int(off[-1])).astype(np.uint32)
    tags = owner[obs].astype(np.int32)
    got = bwo.baum_welch(A, Bm, pi, obs, off, n_iter=1, nthreads=2)
    ref = po.mle(np.zeros((K, K)), np.zeros((K, M)), np.zeros(K), obs, tags, off)
    assert got["skipped"] == 0
    for g, r in zip((got["a"], got["b"], got["pi"]), ref):
        _close(g, r, 1e-13)


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_oracle_loglik_non_decreasing(seed):
    rng = np.random.default_rng(100 + seed)
    K, M = 4, 6
    A, Bm, pi = random_hmm(rng, K, M, zero_frac=0.1)
    lens = rng.integers(1, 15, 30)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    obs = rng.integers(0, M, int(off[-1])).astype(np.uint32)
    got = bwo.baum_welch(A, Bm, pi, obs, off, n_iter=20, nthreads=2)
    ll = got["loglik"]
    assert got["iters"] == 20
    assert (np.diff(ll) >= -1e-9 * np.abs(ll[:-1])).all()


def test_oracle_statuses():
    rng = np.random.default_rng(5)
    A, Bm, pi = random_hmm(rng, 3, 4)
    obs, off = np.array([0, 1, 2], np.uint32), np.array([0, 3], np.int64)
    with pytest.raises(po.OracleError) as e:
        bwo.baum_welch(A, Bm, pi, obs, np.array([0, 0, 3], np.int64))
    assert e.value.code == po.ERR_EMPTY
    with pytest.raises(po.OracleError) as e:
        bwo.baum_welch(A, Bm, pi, np.array([0, 4, 2], np.uint32), off)
    assert e.value.code == po.ERR_ARG
    with pytest.raises(po.OracleError) as e:
        bwo.baum_welch(A, Bm, pi, obs, off, n_iter=0)
    assert e.value.code == po.ERR_ARG
    A2 = A.copy(); A2[0, 0] = np.nan
    with pytest.raises(po.OracleError) as e:
        bwo.baum_welch(A2, Bm, pi, obs, off)
    assert e.value.code == po.ERR_NAN


def test_train_without_device_raises():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    rng = np.random.default_rng(0)
    A, Bm, pi = random_hmm(rng, 3, 5)
    h = cv.HMM(A, Bm, pi)
    with pytest.raises(cv.CvError) as e:
        h.train([[0, 1, 2], [3]], n_iter=1)
    assert e.value.code == cv._lib.ERR_CUDA
