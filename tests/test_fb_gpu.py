"""cv_loglik_batch / cv_posterior_batch (loglik_batch, posterior_batch, score) against the log-space C oracle
(cvo_forward_backward): log-likelihood to 1e-12 relative, posteriors to 1e-12 absolute, forbidden states exactly 0.0,
path and pmax taken from the returned rows bit for bit; the edge cases of the scaling, batch independence and
determinism, the ties to Baum-Welch and decoding, and every status of the two entry points."""
import itertools

import numpy as np
import pytest

import consistent_viterbi_b200 as cv
from oracle import fb_oracle as fbo
from oracle import pyoracle as po
from util import random_batch, random_hmm

pytestmark = pytest.mark.gpu


def _hmm(A, Bm, pi, bdims=None):
    K = A.shape[0]
    return cv.HMM(A.copy(), (Bm.reshape((K,) + tuple(bdims)) if bdims else Bm).copy(), pi.copy())


def _first_argmax(post):
    """lowest index of the maximum of every row, and the maximum"""
    return post.argmax(axis=1).astype(np.uint32), post.max(axis=1)


def _check(res, ref, Bm, obs):
    """res: posterior_batch(want_posteriors=True); ref: fbo.forward_backward"""
    ll, rl = res["loglik"], ref["loglik"]
    assert (np.isneginf(ll) == np.isneginf(rl)).all(), "P(O) = 0 pattern differs"
    f = np.isfinite(rl)
    assert (np.abs(ll[f] - rl[f]) <= 1e-12 * np.maximum(1.0, np.abs(rl[f]))).all(), np.max(np.abs(ll[f] - rl[f]))
    post, rp = res["post"], ref["post"]
    err = np.max(np.abs(post - rp)) if post.size else 0.0
    assert err <= 1e-12, err
    forbidden = np.isneginf(Bm.reshape(Bm.shape[0], -1)[:, obs].T)        # [N, K]: emission -inf at that position
    assert (post[forbidden] == 0.0).all()
    path, pmax = _first_argmax(post)
    assert res["path"].tobytes() == path.tobytes() and res["pmax"].tobytes() == pmax.tobytes()
    if rp.shape[1] > 1:
        top2 = np.sort(rp, axis=1)[:, -2:]
        clear = top2[:, 1] - top2[:, 0] > 1e-9
        assert (res["path"][clear] == rp.argmax(axis=1)[clear]).all()


def _run(A, Bm, pi, obs, off, bdims=None):
    h = _hmm(A, Bm, pi, bdims)
    res = cv.posterior_batch(h, obs, off, device=0, want_posteriors=True)
    ref = fbo.forward_backward(A, Bm, pi, obs, off, nthreads=8)
    _check(res, ref, Bm, obs)
    return h, res, ref


@pytest.mark.parametrize("K", [1, 3, 8, 13, 45, 64])
def test_matches_oracle(K):
    rng = np.random.default_rng(2000 + K)
    M = 30
    A, Bm, pi = random_hmm(rng, K, M, zero_frac=0.15)
    Bm[:, :] = np.where(np.isneginf(Bm).all(axis=0, keepdims=True), np.log10(1.0 / M), Bm)   # every symbol emittable
    obs, off = random_batch(rng, 150, M, 1, 200)
    h, res, ref = _run(A, Bm, pi, obs, off, bdims=(5, 6))
    assert np.isfinite(res["loglik"]).any()
    ll = cv.loglik_batch(h, obs, off, device=0)
    assert ll.tobytes() == res["loglik"].tobytes()


def test_long_sequence_underflow_scaled():
    """T = 10 000 with emissions near 1e-5: unscaled probabilities underflow after ~60 steps."""
    rng = np.random.default_rng(31)
    K, M = 6, 100000
    A, _, pi = random_hmm(rng, K, K, zero_frac=0.0)
    Bm = np.log10(rng.uniform(0.5, 1.5, (K, M)) / M)
    obs, off = random_batch(rng, 3, M, 10000, 10000)
    _, res, _ = _run(A, Bm, pi, obs, off)
    assert np.isfinite(res["loglik"]).all() and (res["loglik"] < -40000).all()


def test_emissions_near_1e_300():
    """One-step sequences whose normaliser Z = sum_i pi_i b_i(o) is subnormal (pi ~ 1e-9, b ~ 1e-300): 1/Z would
    overflow, the posteriors must not.  Longer sequences over the same emissions underflow the scaled forward sum
    (products of two emissions), which the contract treats as P(O) = 0."""
    rng = np.random.default_rng(32)
    K, M = 4, 10
    A, _, _ = random_hmm(rng, K, K, zero_frac=0.0)
    Bm = np.log10(rng.uniform(0.5, 1.5, (K, M))) - 300.0
    pi = np.log10(rng.uniform(0.5, 1.5, K)) - 9.0
    obs, off = random_batch(rng, 200, M, 1, 1)
    _, res, ref = _run(A, Bm, pi, obs, off)
    assert np.isfinite(res["loglik"]).all() and (res["loglik"] < -308).any()
    assert np.isfinite(res["post"]).all() and np.allclose(res["post"].sum(axis=1), 1.0, rtol=0, atol=1e-12)
    obs2, off2 = random_batch(rng, 20, M, 2, 6)
    r2 = cv.posterior_batch(_hmm(A, Bm, pi), obs2, off2, device=0, want_posteriors=True)
    assert np.isneginf(r2["loglik"]).all()
    assert (r2["post"] == 0.0).all() and (r2["path"] == 0).all() and (r2["pmax"] == 0.0).all()


def test_impossible_sequences_leave_neighbours_unchanged():
    rng = np.random.default_rng(33)
    K, M = 5, 9
    A, Bm, pi = random_hmm(rng, K, M, zero_frac=0.3)
    Bm[:, 8] = -np.inf                                     # symbol 8 is impossible
    obs, off = random_batch(rng, 200, M - 1, 1, 40)
    bad = [5, 17, 100]
    for b in bad:
        obs[off[b] + (off[b + 1] - off[b]) // 2] = 8
    h, res, ref = _run(A, Bm, pi, obs, off)
    assert np.isneginf(res["loglik"][bad]).all()
    for b in bad:
        s = slice(off[b], off[b + 1])
        assert (res["post"][s] == 0.0).all() and (res["path"][s] == 0).all() and (res["pmax"][s] == 0.0).all()
    # the same batch without the impossible sequences: every other sequence gets the same bytes
    keep = [b for b in range(len(off) - 1) if b not in bad]
    o2 = np.concatenate([obs[off[b]:off[b + 1]] for b in keep])
    off2 = np.concatenate([[0], np.cumsum(np.diff(off)[keep])]).astype(np.int64)
    r2 = cv.posterior_batch(h, o2, off2, device=0, want_posteriors=True)
    pos = np.concatenate([np.arange(off[b], off[b + 1]) for b in keep])
    assert r2["loglik"].tobytes() == res["loglik"][keep].tobytes()
    assert r2["post"].tobytes() == res["post"][pos].tobytes()
    assert r2["path"].tobytes() == res["path"][pos].tobytes() and r2["pmax"].tobytes() == res["pmax"][pos].tobytes()


def test_single_step_sequences():
    rng = np.random.default_rng(34)
    K, M = 45, 50
    A, Bm, pi = random_hmm(rng, K, M, zero_frac=0.1)
    obs, off = random_batch(rng, 500, M, 1, 1)
    _run(A, Bm, pi, obs, off)


def _pos_batch(seed, B=3000):
    rng = np.random.default_rng(seed)
    A, Bm, pi = random_hmm(rng, 45, 500, zero_frac=0.1)
    obs, off = random_batch(rng, B, 500, 1, 60)
    return A, Bm, pi, obs, off


def _subset(obs, off, idx):
    o = np.concatenate([obs[off[b]:off[b + 1]] for b in idx]).astype(np.uint32)
    return o, np.concatenate([[0], np.cumsum(np.diff(off)[idx])]).astype(np.int64)


def _rows(res, off, b, K):
    s = slice(off[b], off[b + 1])
    return (res["loglik"][b].tobytes(), res["path"][s].tobytes(), res["pmax"][s].tobytes(), res["post"][s].tobytes())


def test_batch_independence_and_chunks():
    A, Bm, pi, obs, off = _pos_batch(41)
    K, B = 45, len(off) - 1
    h = _hmm(A, Bm, pi)
    full = cv.posterior_batch(h, obs, off, device=0, want_posteriors=True)
    rev = list(range(B))[::-1]
    o_r, off_r = _subset(obs, off, rev)
    rres = cv.posterior_batch(h, o_r, off_r, device=0, want_posteriors=True)
    L = cv._lib.lib()
    chunked = []
    try:
        for n in (1, 7, 1000):
            L.cv_debug_set_fb_chunk_seqs(n)
            chunked.append(cv.posterior_batch(h, obs, off, device=0, want_posteriors=True))
    finally:
        L.cv_debug_set_fb_chunk_seqs(0)
    for c in chunked:
        for k in ("loglik", "path", "pmax", "post"):
            assert c[k].tobytes() == full[k].tobytes()
    for b in (0, 1, 63, 64, 1234, 2998, 2999):
        alone = cv.posterior_batch(h, *_subset(obs, off, [b]), device=0, want_posteriors=True)
        want = _rows(full, off, b, K)
        assert _rows(alone, np.array([0, off[b + 1] - off[b]]), 0, K) == want
        assert _rows(rres, off_r, B - 1 - b, K) == want
    ll = cv.loglik_batch(h, obs, off, device=0)
    assert ll.tobytes() == full["loglik"].tobytes()
    try:
        L.cv_debug_set_fb_chunk_seqs(7)
        assert cv.loglik_batch(h, obs, off, device=0).tobytes() == ll.tobytes()
    finally:
        L.cv_debug_set_fb_chunk_seqs(0)


def test_two_calls_same_bytes():
    A, Bm, pi, obs, off = _pos_batch(42)
    out = []
    for _ in range(2):
        h = _hmm(A, Bm, pi)
        r = cv.posterior_batch(h, obs, off, device=0, want_posteriors=True)
        out.append(tuple(r[k].tobytes() for k in ("loglik", "path", "pmax", "post")) + (cv.loglik_batch(h, obs, off, 0).tobytes(),))
    assert out[0] == out[1]
    assert out[0][0] == out[0][4]


def test_null_output_combinations():
    A, Bm, pi, obs, off = _pos_batch(43, B=400)
    K, B, N = 45, len(off) - 1, len(obs)
    h = _hmm(A, Bm, pi)
    full = cv.posterior_batch(h, obs, off, device=0, want_posteriors=True)
    L = cv._lib.lib()
    for mask in itertools.product((0, 1), repeat=4):
        bufs = [np.full(N, 7, np.uint32), np.full(N, -1.0), np.full((N, K), -1.0), np.full(B, 5.0)]
        ptrs = [b.ctypes.data if m else None for b, m in zip(bufs, mask)]
        cv._lib.check(L.cv_posterior_batch(h.device_handle(0), obs.ctypes.data, off.ctypes.data, B, *ptrs))
        for m, b, k in zip(mask, bufs, ("path", "pmax", "post", "loglik")):
            if m:
                assert b.tobytes() == full[k].tobytes(), (mask, k)


def test_ties_to_training_and_decoding():
    rng = np.random.default_rng(44)
    K, M = 12, 40
    A, Bm, pi = random_hmm(rng, K, M, zero_frac=0.1)
    Bm[:, 39] = -np.inf
    obs, off = random_batch(rng, 500, M, 1, 30)
    obs[off[9]] = 39
    h = _hmm(A, Bm, pi)
    res = cv.posterior_batch(h, obs, off, device=0, want_posteriors=True)
    # the decoder on the same handle still equals the oracle bit for bit
    paths, scores = cv.decode_batch(h, obs, off, device=0)
    rp, rs = po.decode_batch(A, Bm, obs, off)
    assert (paths == rp).all() and scores.tobytes() == rs.tobytes()
    t = _hmm(A, Bm, pi)
    tr = t.train_arrays(obs, off, n_iter=1, device=0)
    ll = res["loglik"]
    assert np.isneginf(ll[9]) and int(np.isneginf(ll).sum()) == tr["skipped"]
    assert ll[np.isfinite(ll)].sum() == pytest.approx(tr["loglik"][0], rel=1e-12)
    first = res["post"][off[:-1]][np.isfinite(ll)]
    np.testing.assert_allclose(first.mean(axis=0), 10.0 ** t.pi, rtol=1e-9, atol=0)
    seqs = [obs[off[b]:off[b + 1]] for b in range(len(off) - 1) if np.isfinite(ll[b])]
    assert cv.score(h, seqs, device=0) == pytest.approx(ll[np.isfinite(ll)].sum(), rel=1e-14)


def test_statuses():
    rng = np.random.default_rng(45)
    A, Bm, pi = random_hmm(rng, 4, 6)
    obs, off = np.array([0, 1, 2], np.uint32), np.array([0, 3], np.int64)
    L = cv._lib.lib()
    h = _hmm(A, Bm, pi)
    hd = h.device_handle(0)

    def code(fn):
        with pytest.raises(cv.CvError) as e:
            fn()
        return e.value.code

    # B = 0: CV_OK, nothing written
    ll = np.full(2, 3.0)
    path = np.full(2, 9, np.uint32)
    assert L.cv_loglik_batch(hd, obs.ctypes.data, off.ctypes.data, 0, ll.ctypes.data) == cv._lib.OK
    assert L.cv_posterior_batch(hd, obs.ctypes.data, off.ctypes.data, 0, path.ctypes.data, None, None, ll.ctypes.data) == cv._lib.OK
    assert (ll == 3.0).all() and (path == 9).all()
    for fn in (cv.loglik_batch, cv.posterior_batch):
        assert code(lambda: fn(h, obs, np.array([0, 0, 3], np.int64), device=0)) == cv._lib.ERR_EMPTY
        assert code(lambda: fn(h, np.array([0, 6, 1], np.uint32), off, device=0)) == cv._lib.ERR_ARG
    assert L.cv_loglik_batch(None, obs.ctypes.data, off.ctypes.data, 1, ll.ctypes.data) == cv._lib.ERR_ARG
    assert L.cv_posterior_batch(None, obs.ctypes.data, off.ctypes.data, 1, None, None, None, None) == cv._lib.ERR_ARG
    assert L.cv_loglik_batch(hd, None, off.ctypes.data, 1, ll.ctypes.data) == cv._lib.ERR_ARG
    assert L.cv_loglik_batch(hd, obs.ctypes.data, None, 1, ll.ctypes.data) == cv._lib.ERR_ARG
    assert L.cv_loglik_batch(hd, obs.ctypes.data, off.ctypes.data, 1, None) == cv._lib.ERR_ARG
    assert L.cv_posterior_batch(hd, None, off.ctypes.data, 1, None, None, None, ll.ctypes.data) == cv._lib.ERR_ARG
    assert L.cv_posterior_batch(hd, obs.ctypes.data, None, 1, None, None, None, ll.ctypes.data) == cv._lib.ERR_ARG
    A3, B3, p3 = random_hmm(rng, 65, 6)
    h3 = _hmm(A3, B3, p3)
    assert code(lambda: cv.loglik_batch(h3, obs, off, device=0)) == cv._lib.ERR_UNSUPPORTED
    assert code(lambda: cv.posterior_batch(h3, obs, off, device=0)) == cv._lib.ERR_UNSUPPORTED
    h3.close()
    # the positive-entry bound at its exact edge: 64 is accepted (and right), the next double is refused
    for where in ("a", "b", "pi"):
        m = {"a": A.copy(), "b": Bm.copy(), "pi": pi.copy()}
        m[where].flat[1] = 64.0
        he = _hmm(m["a"], m["b"], m["pi"])
        res = cv.posterior_batch(he, obs, off, device=0, want_posteriors=True)
        ref = fbo.forward_backward(m["a"], m["b"], m["pi"], obs, off)
        _check(res, ref, m["b"], obs)
        m[where].flat[1] = np.nextafter(64.0, np.inf)
        hx = _hmm(m["a"], m["b"], m["pi"])
        assert code(lambda: cv.loglik_batch(hx, obs, off, device=0)) == cv._lib.ERR_UNSUPPORTED
        assert code(lambda: cv.posterior_batch(hx, obs, off, device=0)) == cv._lib.ERR_UNSUPPORTED
        he.close(); hx.close()
    h.close()
