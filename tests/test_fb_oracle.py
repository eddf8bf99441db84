"""CPU tests of the forward-backward oracle (oracle/fb_oracle.c cvo_forward_backward, the checker of cv_loglik_batch /
cv_posterior_batch): against brute-force path enumeration, against the log-likelihood of cvo_baum_welch, posterior
rows that sum to 1; and the product's refusal to run without a device."""
import itertools

import numpy as np
import pytest

import consistent_viterbi_b200 as cv
from oracle import bw_oracle as bwo
from oracle import fb_oracle as fbo
from oracle import pyoracle as po
from util import random_batch, random_hmm


def _p(x):
    return np.where(np.isneginf(x), 0.0, 10.0 ** np.where(np.isneginf(x), 0.0, x))


def _brute(logA, logB, logPi, obs, off):
    """P(O) and gamma_t(i) of every sequence from explicit sums over all K^T paths."""
    A, Bm, pi = _p(logA), _p(logB), _p(logPi)
    K = A.shape[0]
    P, post = [], np.zeros((len(obs), K))
    for i in range(len(off) - 1):
        o = obs[off[i]:off[i + 1]]
        T = len(o)
        tot, g = 0.0, np.zeros((T, K))
        for s in itertools.product(range(K), repeat=T):
            pr = pi[s[0]] * Bm[s[0], o[0]]
            for t in range(1, T):
                pr *= A[s[t - 1], s[t]] * Bm[s[t], o[t]]
            tot += pr
            for t in range(T):
                g[t, s[t]] += pr
        P.append(tot)
        if tot > 0.0:
            post[off[i]:off[i + 1]] = g / tot
    return np.array(P), post


@pytest.mark.parametrize("K,seed", [(1, 0), (2, 1), (3, 2), (4, 3), (4, 4)])
def test_oracle_against_enumeration(K, seed):
    rng = np.random.default_rng(seed)
    M = 4
    A, Bm, pi = random_hmm(rng, K, M, zero_frac=0.25)
    Bm[:, 3] = -np.inf                                  # observation 3 impossible: its sequence has P(O) = 0
    lens = [1, 2, 6, 3, 1, 5, 4, 6]
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    obs = rng.integers(0, 3, int(off[-1])).astype(np.uint32)
    obs[off[3] + 1] = 3
    P, post = _brute(A, Bm, pi, obs, off)
    got = fbo.forward_backward(A, Bm, pi, obs, off, nthreads=3)
    zero = P == 0.0
    assert zero[3] and np.isneginf(got["loglik"][zero]).all() and np.isfinite(got["loglik"][~zero]).all()
    np.testing.assert_allclose(10.0 ** got["loglik"][~zero], P[~zero], rtol=1e-13, atol=0)
    np.testing.assert_allclose(got["post"], post, rtol=0, atol=1e-13)
    assert (got["post"][off[3]:off[4]] == 0.0).all()


def test_loglik_sum_equals_baum_welch():
    rng = np.random.default_rng(21)
    K, M = 6, 12
    A, Bm, pi = random_hmm(rng, K, M, zero_frac=0.2)
    Bm[:, 11] = -np.inf
    obs, off = random_batch(rng, 300, M, 1, 40)
    got = fbo.forward_backward(A, Bm, pi, obs, off, nthreads=4)
    bw = bwo.baum_welch(A, Bm, pi, obs, off, n_iter=1, nthreads=2)
    ll = got["loglik"]
    assert int(np.isneginf(ll).sum()) == bw["skipped"] >= 1
    assert ll[np.isfinite(ll)].sum() == pytest.approx(bw["loglik"][0], rel=1e-12)


def test_posterior_rows_sum_to_one():
    rng = np.random.default_rng(22)
    K, M = 13, 40
    A, Bm, pi = random_hmm(rng, K, M, zero_frac=0.15)
    obs, off = random_batch(rng, 200, M, 1, 80)
    got = fbo.forward_backward(A, Bm, pi, obs, off, nthreads=4)
    ok = np.repeat(np.isfinite(got["loglik"]), np.diff(off))
    assert ok.any()
    np.testing.assert_allclose(got["post"][ok].sum(axis=1), 1.0, rtol=0, atol=1e-13)
    assert (got["post"][~ok] == 0.0).all()
    # the thread count does not change a byte: every sequence is computed on its own
    one = fbo.forward_backward(A, Bm, pi, obs, off, nthreads=1)
    assert one["loglik"].tobytes() == got["loglik"].tobytes() and one["post"].tobytes() == got["post"].tobytes()


def test_oracle_statuses():
    rng = np.random.default_rng(5)
    A, Bm, pi = random_hmm(rng, 3, 4)
    with pytest.raises(po.OracleError) as e:
        fbo.forward_backward(A, Bm, pi, np.array([0, 1, 2], np.uint32), np.array([0, 0, 3], np.int64))
    assert e.value.code == po.ERR_EMPTY
    with pytest.raises(po.OracleError) as e:
        fbo.forward_backward(A, Bm, pi, np.array([0, 4, 2], np.uint32), np.array([0, 3], np.int64))
    assert e.value.code == po.ERR_ARG


def test_inference_without_device_raises():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    rng = np.random.default_rng(0)
    A, Bm, pi = random_hmm(rng, 3, 5)
    h = cv.HMM(A, Bm, pi)
    obs, off = np.array([0, 1, 2], np.uint32), np.array([0, 3], np.int64)
    for fn in (lambda: cv.loglik_batch(h, obs, off), lambda: cv.posterior_batch(h, obs, off),
               lambda: cv.score(h, [[0, 1, 2], [3]])):
        with pytest.raises(cv.CvError) as e:
            fn()
        assert e.value.code == cv._lib.ERR_CUDA
