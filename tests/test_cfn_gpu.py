"""cv_cfn_tables (write_cfn's numeric part, cfn.rs:82-167) against the literal C restatement: cost tables, unary
costs and lower bound bit for bit, including -inf models, sequence starts inside segments, a last boundary at the
very end and the reference's `== 0.0 => assign` accumulation rule."""
import numpy as np
import pytest

import consistent_viterbi_b200 as cv
from oracle import pyoracle as po
from util import random_hmm, random_superseq

pytestmark = pytest.mark.gpu


def _same(x, y):
    return np.ascontiguousarray(x).tobytes() == np.ascontiguousarray(y).tobytes()


@pytest.mark.parametrize("seed", range(12))
def test_cfn_tables_match_oracle(seed):
    rng = np.random.default_rng(8800 + seed)
    K = int(rng.choice([2, 5, 12, 16, 31, 33, 45, 64]))
    M = int(rng.integers(3, 30))
    A, B, pi = random_hmm(rng, K, M, zero_frac=float(rng.choice([0.0, 0.15])), ties=(seed % 4 == 0))
    obs, start, comp, k = random_superseq(rng, int(rng.integers(3, 40)), M, int(rng.integers(1, 5)), float(rng.choice([0.05, 0.3])), 1, 25)
    if k == 0:
        comp[len(comp) // 2] = 0
        k = 1
    if seed % 3 == 0:
        comp[-1] = k - 1                                          # last boundary may sit on the last element
    h = cv.HMM(A, B, pi)
    got = cv.cfn_tables(h, obs, start, comp, k)
    ref = po.cfn_tables(A, B, pi, obs, start, comp, k)
    assert got["nboundaries"] == ref["nboundaries"]
    assert _same(got["tables"], ref["tables"]), "cost tables differ"
    assert _same(got["unary"], ref["unary"]), "unary costs differ"
    assert _same(np.float64(got["lower_bound"]), np.float64(ref["lower_bound"]))
    h.close()


def test_cfn_larger_and_errors():
    rng = np.random.default_rng(5)
    K, M = 16, 64
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.0)
    obs, start, comp, k = random_superseq(rng, 300, M, 4, 0.2, 20, 60)
    h = cv.HMM(A, B, pi)
    got = cv.cfn_tables(h, obs, start, comp, k)
    ref = po.cfn_tables(A, B, pi, obs, start, comp, k)
    assert _same(got["tables"], ref["tables"]) and _same(got["unary"], ref["unary"]) and got["lower_bound"] == ref["lower_bound"]
    t = got["tables"]
    assert _same(t, np.transpose(t, (1, 0, 3, 2)))                # the two mirrored entries always move together
    with pytest.raises(cv.CvError) as e:                          # no constrained element: .last().unwrap() panics
        cv.cfn_tables(h, obs, start, np.full_like(comp, -1), 2)
    assert e.value.code == cv._lib.ERR_EMPTY
    h.close()
    A, B, pi = random_hmm(rng, 65, M, zero_frac=0.0)              # the warp-per-chain step covers K <= 64
    h = cv.HMM(A, B, pi)
    with pytest.raises(cv.CvError) as e:
        cv.cfn_tables(h, obs, start, comp, k)
    assert e.value.code == cv._lib.ERR_UNSUPPORTED
    h.close()


def _check_cfn(A, B, pi, obs, start, comp, k):
    h = cv.HMM(A, B, pi)
    try:
        got = cv.cfn_tables(h, obs, start, comp, k)
    finally:
        h.close()
    ref = po.cfn_tables(A, B, pi, obs, start, comp, k)
    assert got["nboundaries"] == ref["nboundaries"]
    assert _same(got["tables"], ref["tables"]), "cost tables differ"
    assert _same(got["unary"], ref["unary"]), "unary costs differ"
    assert _same(np.float64(got["lower_bound"]), np.float64(ref["lower_bound"]))
    return got


@pytest.mark.parametrize("K", [1, 32, 64])
@pytest.mark.parametrize("k", [1, 3])
def test_cfn_edge_shapes(K, k):
    """K = 1, K = 32 (the last shape with one state per lane) and K = 64 (no padded lanes), with one component (no
    boundary pair, no table) and with three; tied and -inf model entries."""
    rng = np.random.default_rng(8900 + 10 * K + k)
    M = 9
    for ties in (True, False):
        A, B, pi = random_hmm(rng, K, M, zero_frac=0.15, ties=ties)
        obs, start, comp, kk = random_superseq(rng, 30, M, k, 0.15, 1, 20)
        assert kk == k
        _check_cfn(A, B, pi, obs, start, comp, k)


def test_cfn_many_chains_and_long_pair_lists():
    """More chains than one wave of the grid-stride loop (148 SMs * 8 CTAs * 4 warps = 4736) and, with two
    components, every boundary pair in the one table: far more than one 16-pair round of the accumulation."""
    rng = np.random.default_rng(8950)
    K, M = 16, 12
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.1)
    obs, start, comp, k = random_superseq(rng, 200, M, 2, 0.3, 5, 30)
    assert k == 2
    got = _check_cfn(A, B, pi, obs, start, comp, k)
    npairs = got["nboundaries"] - 1
    assert npairs * K > 4736 and npairs > 3 * 16, npairs
