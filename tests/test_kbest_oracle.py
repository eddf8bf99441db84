"""The k-best Viterbi oracle (cvo_decode_batch_kbest) against exhaustive enumeration of every path: K = 1..4,
T <= 7, every k <= 32, random, tie-heavy and -inf-heavy models.  The score multiset is the top k of all paths, every
path rescores to its score bit for bit, the paths are distinct, "no path" ranks appear exactly where K^T < k, and
rank 0 is the plain decode's oracle (cvo_decode_batch)."""
import numpy as np
import pytest

from kbest_check import NO_PATH, check_against_enumeration
from oracle import kbest_oracle as kbo
from oracle import pyoracle as po
from util import random_hmm


def _model(rng, K, M, kind):
    if kind == "ties":
        A, Bm, _ = random_hmm(rng, K, M, ties=True)
    else:
        A, Bm, _ = random_hmm(rng, K, M, zero_frac=0.5 if kind == "neginf" else 0.0)
    if kind == "neginf":
        Bm[:, M - 1] = -np.inf                      # a symbol no state can emit: every path of its sequences is -inf
    return A, Bm


@pytest.mark.parametrize("kind", ["random", "ties", "neginf"])
@pytest.mark.parametrize("K", [1, 2, 3, 4])
def test_oracle_matches_enumeration(K, kind):
    rng = np.random.default_rng(100 * K + len(kind))
    M = 5
    A, Bm = _model(rng, K, M, kind)
    tmax = {1: 7, 2: 7, 3: 7, 4: 6}[K]
    lens = np.concatenate([np.arange(1, tmax + 1), rng.integers(1, tmax + 1, size=6)])
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    obs = rng.integers(0, M, size=int(off[-1])).astype(np.uint32)
    rp, rs = po.decode_batch(A, Bm, obs, off)
    for k in range(1, 33):
        paths, scores = kbo.decode_batch_kbest(A, Bm, obs, off, k, nthreads=4)
        check_against_enumeration(A, Bm, obs, off, k, paths, scores, rp, rs)


def test_oracle_threads_and_statuses():
    rng = np.random.default_rng(7)
    A, Bm = _model(rng, 3, 4, "random")
    off = np.array([0, 3, 4, 9], dtype=np.int64)
    obs = rng.integers(0, 4, size=9).astype(np.uint32)
    one = kbo.decode_batch_kbest(A, Bm, obs, off, 5, nthreads=1)
    many = kbo.decode_batch_kbest(A, Bm, obs, off, 5, nthreads=8)
    assert one[0].tobytes() == many[0].tobytes() and one[1].tobytes() == many[1].tobytes()
    assert (one[0][3:, 3] == NO_PATH).all() and (one[1][3:, 1] == -np.inf).all()   # one element, K = 3: three paths
    for args, code in (((obs, np.array([0, 3, 3, 9]), 5), 1), ((obs, off, 0), 3),
                       ((np.where(obs == 0, 4, obs).astype(np.uint32), off, 5), 3)):
        with pytest.raises(po.OracleError) as e:
            kbo.decode_batch_kbest(A, Bm, *args)
        assert e.value.code == code
