"""Model magnitudes (include/cv_b200.h, cv_hmm_create): finite entries beyond 2^900 are refused, so that no sum the
kernels form can overflow and every -inf a kernel sees means "impossible", as the lazy backpointer rule of the
backtraces assumes; the f32 mode refuses entries beyond 2^64.  At the accepted extremes -- entries around +-2^899, f64
subnormals -- every decode path and the constrained solver still equal the C oracle bit for bit."""
import numpy as np
import pytest

import consistent_viterbi_b200 as cv
from oracle import np_viterbi as nv
from oracle import pyoracle as po
from test_cp_gpu import _check as _check_cp
from util import random_hmm, random_superseq

pytestmark = pytest.mark.gpu

BOUND, BOUND32 = 2.0 ** 900, 2.0 ** 64


def _rejected(A, B, pi):
    with pytest.raises(cv.CvError) as e:
        cv.HMM(A, B, pi).device_handle()
    assert e.value.code == cv._lib.ERR_UNSUPPORTED


def test_finite_overflow_models_are_rejected():
    """Models on which a finite candidate plus a finite emission overflows.  Negative overflow: the reference stores the
    argmax as backpointer (path [1, 0], score -inf) while the lazy backtraces would take -inf for an impossible emission
    and return [0, 0].  Positive overflow: +inf + -inf would be NaN in the forward epilogue.  Embedded in K = 65 and 130
    as well (the large-K kernel)."""
    A = np.array([[-1e308, -1e308], [-5e307, -5e307]])
    B = np.array([[0.0, -1.5e308], [0.0, -1.5e308]])
    p, s = po.decode_batch(A, B, np.array([0, 1], np.uint32), np.array([0, 2], np.int64))
    assert p.tolist() == [1, 0] and s[0] == -np.inf
    Ap = np.full((2, 2), 1e308)
    Bp = np.array([[1e308, -np.inf], [1e308, 1e308]])
    for A2, B2 in ((A, B), (Ap, Bp)):
        for K in (2, 65, 130):
            Ak = np.full((K, K), -np.inf); Ak[:2, :2] = A2
            Bk = np.full((K, 2), -np.inf); Bk[:2] = B2
            _rejected(Ak, Bk, np.zeros(K))


@pytest.mark.parametrize("where", ["A", "B", "pi"])
def test_magnitude_bound_is_inclusive(where):
    """+-2^900 is accepted, the next double beyond it refused, in logA, logB and logPi alike; -inf stays accepted."""
    rng = np.random.default_rng(40)
    K, M = 5, 4
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.2)
    for x, ok in ((BOUND, True), (-BOUND, True), (np.nextafter(BOUND, np.inf), False),
                  (-np.nextafter(BOUND, np.inf), False), (-np.inf, True)):
        m = {"A": A.copy(), "B": B.copy(), "pi": pi.copy()}
        m[where].flat[3] = x
        if ok:
            h = cv.HMM(m["A"], m["B"], m["pi"])
            h.device_handle()
            h.close()
        else:
            _rejected(m["A"], m["B"], m["pi"])


def test_f32_mode_magnitude_bound():
    """The f32 mode accepts |x| <= 2^64 (f32 parity at the bound) and refuses a model with a larger finite entry, which
    the exact mode still decodes."""
    rng = np.random.default_rng(41)
    K, M, Bn = 20, 10, 9000
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.2)
    A[rng.random((K, K)) < 0.1] = BOUND32
    A[rng.random((K, K)) < 0.1] = -BOUND32
    B[rng.random((K, M)) < 0.1] = -BOUND32
    lens = rng.integers(1, 40, size=Bn)
    off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    obs = rng.integers(0, M, size=int(off[-1])).astype(np.uint32)
    rp, rs = nv.decode_batch(A, B, obs, off, np.float32)
    h = cv.HMM(A, B, pi)
    p, s = cv.decode_batch_f32(h, obs, off)
    assert (p == rp).all() and (np.isneginf(s) == np.isneginf(rs)).all() and (s == rs).all()
    h.close()
    for x in (np.nextafter(BOUND32, np.inf), -np.nextafter(BOUND32, np.inf)):
        A2 = A.copy(); A2[1, 2] = x
        h = cv.HMM(A2, B, pi)
        with pytest.raises(cv.CvError) as e:
            cv.decode_batch_f32(h, obs, off)
        assert e.value.code == cv._lib.ERR_UNSUPPORTED
        rc = cv._lib.lib().cv_decode_batch_dev_f32(h.device_handle(), None, None, 1, 1, 1, None, None, None, 1)
        assert rc == cv._lib.ERR_UNSUPPORTED                         # refused before any buffer is looked at
        rp64, rs64 = po.decode_batch(A2, B, obs, off, nthreads=8)
        p64, s64 = cv.decode_batch(h, obs, off)
        assert (p64 == rp64).all() and s64.tobytes() == rs64.tobytes()
        h.close()


def _extreme_model(rng, K, M, kind):
    if kind == "large":        # entries around +-2^899 next to ordinary ones: sums in the 2^906 range, cancellations
        vals = np.array([2.0 ** 899, -2.0 ** 899, -1.5 * 2.0 ** 899, -2.0 ** 898, BOUND, -BOUND, 0.5, -1.0, -np.inf])
        prob = [0.12, 0.2, 0.12, 0.12, 0.04, 0.04, 0.12, 0.12, 0.12]
    else:                      # f64 subnormals: exact sums, ties, signed zeros
        vals = np.array([1e-310, -1e-310, 2.5e-310, -4e-310, 5e-324, -5e-324, 0.0, -0.0, -np.inf])
        prob = [0.12, 0.12, 0.12, 0.12, 0.1, 0.1, 0.1, 0.1, 0.12]
    A, B = rng.choice(vals, size=(K, K), p=prob), rng.choice(vals, size=(K, M), p=prob)
    return A, B


def _check_decode(h, A, B, obs, off, what):
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    p, s = cv.decode_batch(h, obs, off)
    bad = np.flatnonzero(p != rp)
    assert bad.size == 0, f"{what}: {bad.size} path mismatches, first at {bad[:5]}"
    assert s.tobytes() == rs.tobytes(), f"{what}: score bytes differ"


@pytest.mark.parametrize("kind", ["large", "subnormal"])
@pytest.mark.parametrize("K", [3, 17, 45, 64])
def test_small_k_paths_equal_oracle_at_extreme_magnitudes(K, kind):
    """Warp-per-sequence kernel, tile kernel (chain_max 0) with the one-thread and the four-lane backtrace, on ~100-step
    sequences."""
    rng = np.random.default_rng(4100 + K + (1000 if kind == "large" else 0))
    M = 9
    A, B = _extreme_model(rng, K, M, kind)
    lens = rng.integers(60, 140, size=3000)
    lens[:200] = rng.integers(1, 4, size=200)
    off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    obs = rng.integers(0, M, size=int(off[-1])).astype(np.uint32)
    h = cv.HMM(A, B, np.zeros(K))
    L = cv._lib.lib()
    try:
        for chain_max, split in ((-1, 1), (0, 0), (0, 2)):
            L.cv_debug_set_chain_max_batch(chain_max)
            L.cv_debug_set_bt_split(split)
            _check_decode(h, A, B, obs, off, f"chain_max={chain_max} bt_split={split}")
    finally:
        L.cv_debug_set_chain_max_batch(-1)
        L.cv_debug_set_bt_split(1)
    h.close()


@pytest.mark.parametrize("kind", ["large", "subnormal"])
@pytest.mark.parametrize("K", [65, 130])
def test_large_k_path_equals_oracle_at_extreme_magnitudes(K, kind):
    rng = np.random.default_rng(4300 + K + (1000 if kind == "large" else 0))
    M = 7
    A, B = _extreme_model(rng, K, M, kind)
    lens = rng.integers(80, 120, size=150)
    off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    obs = rng.integers(0, M, size=int(off[-1])).astype(np.uint32)
    h = cv.HMM(A, B, np.zeros(K))
    _check_decode(h, A, B, obs, off, f"K={K} {kind}")
    h.close()


@pytest.mark.parametrize("kind", ["large", "subnormal"])
@pytest.mark.parametrize("K", [4, 12, 45, 70])
def test_cp_solve_equals_oracle_at_extreme_magnitudes(K, kind):
    """cv_cp_solve: solution, objective bits, explored nodes, upper bounds and the final state (test_cp_gpu._check)."""
    rng = np.random.default_rng(4500 + K + (1000 if kind == "large" else 0))
    M = 6
    A, B = _extreme_model(rng, K, M, kind)
    pi = _extreme_model(rng, K, 1, kind)[1][:, 0]
    for _ in range(3):
        obs, start, comp, ncomp = random_superseq(rng, 8, M, 3, 0.15, 20, 100)
        _check_cp(A, B, pi, obs, start, comp, ncomp, max_nodes=200)
