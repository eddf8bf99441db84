"""CPU tests of oracle/np_viterbi.py, the vectorized numpy restatement of viterbi::decode that is generic in the
float type.  In f64 it must equal the C oracle bit for bit -- that pins its logic to the reference; the f32 runs differ
from it only in the dtype and are the reference of the f32 decode mode (tests/test_f32_mode_gpu.py).  The last test
measures how far the f32 recurrence drifts from the f64 one with the sequence length: the bound stated in
include/cv_b200.h and viterbi.decode_batch_f32."""
import numpy as np
import pytest

from oracle import np_viterbi as nv
from oracle import pyoracle as po
from util import random_batch, random_hmm


def _assert_f64_equals_oracle(A, B, obs, off):
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=4)
    p, s = nv.decode_batch(A, B, obs, off, np.float64)
    bad = np.flatnonzero(p != rp)
    assert bad.size == 0, f"{bad.size} path mismatches, first at {bad[:5]}"
    assert s.tobytes() == rs.tobytes(), "score bytes differ"


def _batch(lens, M, rng):
    off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    return rng.integers(0, M, size=int(off[-1])).astype(np.uint32), off


@pytest.mark.parametrize("K", [1, 2, 3, 8, 9, 17, 45, 64, 70])
def test_f64_equals_oracle_random(K):
    rng = np.random.default_rng(900 + K)
    M = int(rng.integers(1, 30))
    A, B, _ = random_hmm(rng, K, M, zero_frac=0.2)
    obs, off = random_batch(rng, 600, M, 1, 40)
    _assert_f64_equals_oracle(A, B, obs, off)


@pytest.mark.parametrize("K", [2, 5, 16, 45])
def test_f64_equals_oracle_ties_zeros_and_neg_inf(K):
    """Dyadic values with +-0.0 and -inf: exact ties everywhere, the first-maximum rule decides."""
    rng = np.random.default_rng(910 + K)
    A, B, _ = random_hmm(rng, K, 6, ties=True)
    obs, off = random_batch(rng, 800, 6, 1, 30)
    _assert_f64_equals_oracle(A, B, obs, off)


def test_f64_equals_oracle_all_neg_inf_emission_columns_and_sparse_models():
    rng = np.random.default_rng(920)
    for K in (3, 17, 33):
        A, B, _ = random_hmm(rng, K, 8, zero_frac=0.5)
        B[:, 0] = -np.inf                                            # observation 0 is impossible in every state
        B[:, 5] = -np.inf
        obs, off = random_batch(rng, 500, 8, 1, 12)
        _assert_f64_equals_oracle(A, B, obs, off)


def test_f64_equals_oracle_positive_log_scores_subnormals_and_large_magnitudes():
    rng = np.random.default_rng(930)
    K, M = 12, 10
    A, B, _ = random_hmm(rng, K, M, zero_frac=0.1)
    A[3, 5], B[7, 2], A[0, 0] = 0.75, 1.5, 3.0                      # positive log-scores
    obs, off = random_batch(rng, 400, M, 1, 30)
    _assert_f64_equals_oracle(A, B, obs, off)
    # f64 subnormal entries: sums of subnormals are exact, ties and signs of zero decide the paths
    vals = np.array([1e-310, -1e-310, 2e-310, -3e-310, 0.0, -0.0, -np.inf])
    As, Bs = rng.choice(vals, size=(K, K)), rng.choice(vals, size=(K, M))
    _assert_f64_equals_oracle(As, Bs, obs, off)
    # entries at the model magnitude bound of cv_hmm_create (|x| <= 2^900) and around 2^899
    big = np.array([2.0 ** 900, -2.0 ** 900, 2.0 ** 899, -2.0 ** 899, -1.5 * 2.0 ** 899, 1.0, -np.inf])
    Ab, Bb = rng.choice(big, size=(K, K)), rng.choice(big, size=(K, M))
    lens = rng.integers(1, 120, size=300)
    obs2, off2 = _batch(lens, M, rng)
    _assert_f64_equals_oracle(Ab, Bb, obs2, off2)


def test_f64_overflow_to_neg_inf_keeps_the_reference_backpointer():
    """A finite best candidate plus a finite emission that rounds to -inf: the reference still stores the argmax as psi
    (path [1, 0]), it does not treat the -inf as an impossible emission."""
    A = np.array([[-1e308, -1e308], [-5e307, -5e307]])
    B = np.array([[0.0, -1.5e308], [0.0, -1.5e308]])
    obs, off = np.array([0, 1], np.uint32), np.array([0, 2], np.int64)
    p, s = nv.decode_batch(A, B, obs, off, np.float64)
    assert p.tolist() == [1, 0] and s[0] == -np.inf
    _assert_f64_equals_oracle(A, B, obs, off)


def test_f64_long_and_single_step_sequences_in_one_batch():
    """Sub-batches are cut by count and by backpointer cells: many length-1 sequences next to long ones."""
    rng = np.random.default_rng(940)
    K, M = 9, 7
    A, B, _ = random_hmm(rng, K, M, zero_frac=0.2)
    lens = rng.integers(1, 4, size=5000)
    lens[rng.choice(5000, size=5, replace=False)] = rng.integers(1000, 3000, size=5)
    obs, off = _batch(lens, M, rng)
    _assert_f64_equals_oracle(A, B, obs, off)


def test_f32_picks_the_first_maximum_of_candidates_that_tie_after_rounding():
    """-1.0 and -1.0 + 2^-30 are distinct in f64 (predecessor 1 wins) and equal after rounding to f32 (predecessor 0)."""
    A = np.array([[-1.0, -1.0], [-1.0 + 2.0 ** -30, -1.0 + 2.0 ** -30]])
    B = np.zeros((2, 1))
    obs, off = np.zeros(2, np.uint32), np.array([0, 2], np.int64)
    p64, s64 = nv.decode_batch(A, B, obs, off, np.float64)
    p32, s32 = nv.decode_batch(A, B, obs, off, np.float32)
    assert p64.tolist() == [1, 0] and s64[0] == -1.0 + 2.0 ** -30
    assert p32.tolist() == [0, 0] and s32[0] == -1.0
    _assert_f64_equals_oracle(A, B, obs, off)


@pytest.mark.parametrize("tiny", [1e-40, 1e-45])
def test_f32_subnormal_sums_are_not_flushed(tiny):
    """Entries in the f32 subnormal range: +-tiny decide the argmax (flushed to zero they would tie and pick 0) and
    their sums are exact multiples of the smallest subnormal."""
    t32 = float(np.float32(tiny))
    assert 0.0 < t32 < float(np.finfo(np.float32).tiny)
    A = np.array([[-tiny, -tiny], [tiny, tiny]])
    B = np.array([[tiny], [tiny]])
    T = 5
    obs, off = np.zeros(T, np.uint32), np.array([0, T], np.int64)
    p, s = nv.decode_batch(A, B, obs, off, np.float32)
    assert p.tolist() == [1, 1, 1, 1, 0]                  # predecessor 1 (+tiny) wins every step, end state = first max
    assert s[0] == 2 * (T - 1) * t32                      # (T-1) x (a + b), exact in the subnormal range


def test_f32_length_one_and_two_sequences():
    """Length 1: path [0], score 0 (pi and the first observation are unused).  Length 2: delta[1][i] =
    max_j fl32(0 + a[j][i]) + b[i][o_1], computed by hand in f32."""
    rng = np.random.default_rng(950)
    K, M = 5, 4
    A, B, _ = random_hmm(rng, K, M, zero_frac=0.2)
    obs = np.array([3, 2, 1, 0, 1], np.uint32)
    off = np.array([0, 1, 3, 4, 5], np.int64)                 # lengths 1, 2, 1, 1
    p, s = nv.decode_batch(A, B, obs, off, np.float32)
    a32, b32 = A.astype(np.float32), B.astype(np.float32)
    for b in (0, 2, 3):
        assert p[off[b]] == 0 and s[b] == 0.0
    o1 = obs[off[1] + 1]
    j = a32.argmax(axis=0)                                    # best predecessor of every state (first maximum)
    d1 = np.where(b32[:, o1] == -np.inf, np.float32(-np.inf), a32[j, np.arange(K)] + b32[:, o1])
    end = int(d1.argmax())
    psi = 0 if b32[end, o1] == -np.inf else int(j[end])
    assert p[1:3].tolist() == [psi, end] and s[1] == np.float64(d1[end])


def test_f32_score_deviation_grows_with_the_sequence_length():
    """The f32 recurrence against the f64 oracle on log-probability models (K = 45, 20 sequences per length): the
    relative score deviation grows with T (measured: 4.8e-7 at T = 80, 1.9e-6 at 2000, 9.5e-6 at 20 000) and stays
    below the bound 2 T 2^-24 stated in include/cv_b200.h -- a fixed 1e-5 is not a bound for long sequences."""
    K, M, nseq = 45, 50, 20
    dev = {}
    for T in (80, 2000, 20000):
        rng = np.random.default_rng(960 + T)
        A, B, _ = random_hmm(rng, K, M, zero_frac=0.05)
        obs, off = _batch(np.full(nseq, T), M, rng)
        _, rs = po.decode_batch(A, B, obs, off, nthreads=8)
        _, s32 = nv.decode_batch(A, B, obs, off, np.float32)
        assert np.isfinite(rs).all() and np.isfinite(s32).all()
        dev[T] = float(np.max(np.abs(s32 - rs) / np.abs(rs)))
        assert dev[T] <= 2 * T * 2.0 ** -24, (T, dev[T])
    assert dev[80] < dev[2000] < dev[20000], dev
