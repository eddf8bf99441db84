"""cv_baum_welch (HMM.train / train_arrays) against the log-space C oracle: one iteration from the same start must
agree to 1e-9 relative on every probability >= 1e-250, -inf exactly where the oracle has -inf, the log-likelihood to
1e-12 relative, and the skipped count exactly."""
import numpy as np
import pytest

import consistent_viterbi_b200 as cv
from oracle import bw_oracle as bwo
from oracle import pyoracle as po
from util import random_batch, random_hmm

pytestmark = pytest.mark.gpu


def _p(x):
    return np.where(np.isneginf(x), 0.0, 10.0 ** np.where(np.isneginf(x), 0.0, x))


def _agree(got, ref):
    got, ref = np.asarray(got), np.asarray(ref)
    assert (np.isneginf(got) == np.isneginf(ref)).all(), "-inf pattern differs"
    f = ~np.isneginf(ref) & (ref >= -250)
    np.testing.assert_allclose(_p(got[f]), _p(ref[f]), rtol=1e-9, atol=0)


def _hmm(A, Bm, pi):
    """A model of its own: HMM keeps contiguous f64 arrays without copying, and training updates them in place."""
    return cv.HMM(A.copy(), Bm.copy(), pi.copy())


def _one(A, Bm, pi, obs, off, bdims=None):
    K = A.shape[0]
    h = _hmm(A, Bm.reshape((K,) + tuple(bdims)) if bdims else Bm, pi)
    res = h.train_arrays(obs, off, n_iter=1, device=0)
    ref = bwo.baum_welch(A, Bm, pi, obs, off, n_iter=1, nthreads=8)
    _agree(h.a, ref["a"])
    _agree(h.b.reshape(K, -1), ref["b"])
    _agree(h.pi, ref["pi"])
    assert res["iters"] == 1 and res["skipped"] == ref["skipped"]
    assert res["loglik"][0] == pytest.approx(ref["loglik"][0], rel=1e-12)
    return h, res, ref


@pytest.mark.parametrize("K", [1, 3, 8, 13, 45, 64])
def test_one_iteration_matches_oracle(K):
    rng = np.random.default_rng(1000 + K)
    M = 30
    A, Bm, pi = random_hmm(rng, K, M, zero_frac=0.15)
    Bm[:, :] = np.where(np.isneginf(Bm).all(axis=0, keepdims=True), np.log10(1.0 / M), Bm)   # every symbol emittable
    obs, off = random_batch(rng, 150, M, 1, 200)
    _one(A, Bm, pi, obs, off, bdims=(5, 6))


def test_long_sequence_underflow_scaled():
    """T = 10 000 with emissions near 1e-5: unscaled probabilities underflow after ~60 steps."""
    rng = np.random.default_rng(11)
    K, M = 6, 100000
    A, _, pi = random_hmm(rng, K, K, zero_frac=0.0)
    Bm = np.log10(rng.uniform(0.5, 1.5, (K, M)) / M)
    obs, off = random_batch(rng, 3, M, 10000, 10000)
    _, res, _ = _one(A, Bm, pi, obs, off)
    assert np.isfinite(res["loglik"][0]) and res["loglik"][0] < -40000


def test_structural_zeros_and_skipped():
    rng = np.random.default_rng(12)
    K, M = 5, 9
    A, Bm, pi = random_hmm(rng, K, M, zero_frac=0.3)
    Bm[:, 8] = -np.inf                                     # symbol 8 is impossible
    obs, off = random_batch(rng, 200, M - 1, 1, 40)
    obs[off[5]] = 8; obs[off[17] + 0] = 8; obs[off[100]] = 8
    h, res, _ = _one(A, Bm, pi, obs, off)
    assert res["skipped"] == 3
    assert np.isneginf(h.a[np.isneginf(A)]).all() and np.isneginf(h.b[np.isneginf(Bm)]).all()
    assert np.isneginf(h.pi[np.isneginf(pi)]).all()


def test_multi_iteration_and_tol():
    rng = np.random.default_rng(13)
    K, M = 8, 20
    A, Bm, pi = random_hmm(rng, K, M, zero_frac=0.1)
    obs, off = random_batch(rng, 300, M, 1, 50)
    h = _hmm(A, Bm, pi)
    lls = []
    for _ in range(10):
        a0, b0, p0 = h.a.copy(), h.b.copy(), h.pi.copy()
        res = h.train_arrays(obs, off, n_iter=1, device=0)
        ref = bwo.baum_welch(a0, b0, p0, obs, off, n_iter=1, nthreads=8)
        _agree(h.a, ref["a"]); _agree(h.b, ref["b"]); _agree(h.pi, ref["pi"])
        assert res["loglik"][0] == pytest.approx(ref["loglik"][0], rel=1e-12)
        lls.append(res["loglik"][0])
    assert (np.diff(lls) >= -1e-9 * np.abs(lls[:-1])).all()
    h2 = _hmm(A, Bm, pi)
    full = h2.train_arrays(obs, off, n_iter=10, device=0)
    np.testing.assert_allclose(full["loglik"], lls, rtol=1e-12)
    ll = full["loglik"]
    assert full["iters"] == 10
    rel = (ll[1:] - ll[:-1]) / np.abs(ll[:-1])        # rel[k - 1]: improvement of iteration k over k - 1
    tol = float(rel[2]) * 1.0001
    k = int(np.argmax(rel < tol)) + 1                  # first iteration that meets the stopping rule (<= 3)
    h3 = _hmm(A, Bm, pi)
    early = h3.train_arrays(obs, off, n_iter=10, tol=tol, device=0)
    assert early["iters"] == k + 1 <= 4
    np.testing.assert_allclose(early["loglik"], ll[: k + 1], rtol=1e-12)


def test_deterministic_bytes():
    rng = np.random.default_rng(14)
    A, Bm, pi = random_hmm(rng, 45, 500, zero_frac=0.1)
    obs, off = random_batch(rng, 3000, 500, 1, 60)
    out = []
    for _ in range(2):
        h = _hmm(A, Bm, pi)
        res = h.train_arrays(obs, off, n_iter=2, device=0)
        out.append((h.a.tobytes(), h.b.tobytes(), h.pi.tobytes(), res["loglik"].tobytes()))
    assert out[0] == out[1]


def test_statuses():
    rng = np.random.default_rng(15)
    A, Bm, pi = random_hmm(rng, 4, 6)
    obs, off = np.array([0, 1, 2], np.uint32), np.array([0, 3], np.int64)

    def code(fn):
        with pytest.raises(cv.CvError) as e:
            fn()
        return e.value.code

    assert code(lambda: _hmm(A, Bm, pi).train_arrays(obs, np.array([0, 0, 3], np.int64), 1, device=0)) == cv._lib.ERR_EMPTY
    assert code(lambda: _hmm(A, Bm, pi).train_arrays(np.array([0, 6, 1], np.uint32), off, 1, device=0)) == cv._lib.ERR_ARG
    assert code(lambda: _hmm(A, Bm, pi).train_arrays(obs, off, 0, device=0)) == cv._lib.ERR_ARG
    A2 = A.copy(); A2[1, 2] = np.inf
    assert code(lambda: _hmm(A2, Bm, pi).train_arrays(obs, off, 1, device=0)) == cv._lib.ERR_NAN
    A3, B3, p3 = random_hmm(rng, 65, 6)
    assert code(lambda: _hmm(A3, B3, p3).train_arrays(obs, off, 1, device=0)) == cv._lib.ERR_UNSUPPORTED


def test_trained_model_decodes():
    rng = np.random.default_rng(16)
    K, M = 12, 40
    A, Bm, pi = random_hmm(rng, K, M, zero_frac=0.1)
    obs, off = random_batch(rng, 500, M, 1, 30)
    h = _hmm(A, Bm, pi)
    h.train([obs[off[i]:off[i + 1]] for i in range(len(off) - 1)], n_iter=3, device=0)
    paths, scores = cv.decode_batch(h, obs, off, device=0)
    rp, rs = po.decode_batch(h.a, h.b, obs, off)
    assert (paths == rp).all() and scores.tobytes() == rs.tobytes()
