"""The f32 decode mode (cv_decode_batch_f32 / cv_decode_batch_dev_f32) against its contract in include/cv_b200.h: the
model rounded to f32 once, every add one IEEE binary32 add, first-maximum backpointers.  The reference is the numpy
restatement oracle/np_viterbi.py run in float32 (pinned to the C oracle in f64 by tests/test_np_viterbi.py).  Paths
must be equal and scores equal as values: -inf where the reference has -inf, and zeros compare by value (the sign of a
zero f32 score is unspecified, it cannot change a path).

Batches have more than 8192 sequences: smaller calls are decoded by the exact f64 kernel by contract."""
import numpy as np
import pytest

import consistent_viterbi_b200 as cv
from oracle import np_viterbi as nv
from oracle import pyoracle as po
from util import random_hmm

pytestmark = pytest.mark.gpu

EXACT_MAX_B = 8192                  # f32 calls of at most this many sequences take the f64 warp-per-sequence kernel


def _assert_f32_equal(p, s, rp, rs, what):
    bad = np.flatnonzero(p != rp)
    assert bad.size == 0, f"{what}: {bad.size} path elements differ from the f32 reference, first at {bad[:5]}"
    assert not np.isnan(s).any(), f"{what}: NaN score"
    assert (np.isneginf(s) == np.isneginf(rs)).all(), f"{what}: -inf pattern differs"
    bad = np.flatnonzero(s != rs)
    assert bad.size == 0, f"{what}: {bad.size} scores differ, first {bad[:3]}: {s[bad[:3]]} vs {rs[bad[:3]]}"


def _model(kind, K, M, rng):
    """logA [K,K], logB [K,M] of one of the model families the f32 kernels must get exactly right."""
    if kind == "ties":                     # dyadic values, +-0.0 and -inf: exact ties, the first maximum decides
        vals = np.array([-0.0, 0.0, -0.5, -1.0, -1.5, -2.0, -np.inf])
        prob = [0.03, 0.03, 0.22, 0.22, 0.22, 0.18, 0.10]     # few zeros: an all-zero path would make every score 0
        A, B = rng.choice(vals, size=(K, K), p=prob), rng.choice(vals, size=(K, M), p=prob)
    elif kind == "round_ties":             # distinct in f64, equal after rounding to f32 (|perturbation| < half an ulp)
        base = np.array([-0.5, -0.75, -1.0, -1.5, -2.0, -3.0])
        eps = np.array([0.0, 2.0 ** -30, -2.0 ** -30, 2.0 ** -27, -2.0 ** -28])
        A = rng.choice(base, size=(K, K)) + rng.choice(eps, size=(K, K))
        B = rng.choice(base, size=(K, M)) + rng.choice(eps, size=(K, M))
    elif kind == "subnormal":              # f32 subnormal range: must neither flush to zero nor lose a tie break
        vals = np.array([1e-40, -1e-40, 1e-45, -1e-45, -3e-39, 2e-39, 0.0, -0.0, -np.inf])
        A, B = rng.choice(vals, size=(K, K)), rng.choice(vals, size=(K, M))
    elif kind == "sparse":                 # half of the probabilities zero (-inf)
        A, B, _ = random_hmm(rng, K, M, zero_frac=0.5)
    elif kind == "positive":               # log-scores, not log-probabilities: some entries > 0
        A, B, _ = random_hmm(rng, K, M, zero_frac=0.1)
        A[rng.random((K, K)) < 0.05] = rng.uniform(0.0, 2.0)
        B[rng.random((K, M)) < 0.05] = rng.uniform(0.0, 3.0)
    elif kind == "dead_columns":           # observations that are impossible in every state
        A, B, _ = random_hmm(rng, K, M, zero_frac=0.2)
        B[:, 0] = -np.inf
        B[:, 3] = -np.inf
    else:
        raise ValueError(kind)
    return A, B


def _ragged_batch(rng, Bn, M, tmax=30, nlong=3):
    """Bn sequences: a third of length 1, the rest 2..tmax, and `nlong` of 1000-3000 steps (they stay in the tiles: the
    long-sequence split is off in f32 mode)."""
    lens = rng.integers(2, tmax + 1, size=Bn)
    lens[rng.random(Bn) < 1 / 3] = 1
    lens[rng.choice(Bn, size=nlong, replace=False)] = rng.integers(1000, 3001, size=nlong)
    off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    obs = rng.integers(0, M, size=int(off[-1])).astype(np.uint32)
    return obs, off


KINDS = ["ties", "round_ties", "subnormal", "sparse", "positive", "dead_columns"]
KS = [1, 2, 3, 7, 8, 9, 15, 16, 17, 24, 31, 33, 45, 47, 48, 57, 61, 63, 64]
# every K with two model families, every family at six or seven K: the balanced slot split on (K % 8 != 0 and
# K / ceil(K/8) >= 5) and off, odd K (the pair loop's tail), one state group (K <= 8), a partial last backtrace chunk
CASES = [(K, KINDS[i % 6]) for i, K in enumerate(KS)] + [(K, KINDS[(i + 3) % 6]) for i, K in enumerate(KS)]


@pytest.mark.parametrize("K,kind", CASES)
def test_f32_mode_equals_f32_reference(K, kind):
    rng = np.random.default_rng(10_000 + 100 * K + KINDS.index(kind))
    M = 12
    A, B = _model(kind, K, M, rng)
    Bn = 8193 if K % 2 else 8193 + 64 * int(rng.integers(1, 20)) + int(rng.integers(1, 63))
    obs, off = _ragged_batch(rng, Bn, M)
    rp, rs = nv.decode_batch(A, B, obs, off, np.float32)
    h = cv.HMM(A, B, np.zeros(K))
    p, s = cv.decode_batch_f32(h, obs, off)
    _assert_f32_equal(p, s, rp, rs, f"K={K} {kind} B={Bn}")
    if kind == "round_ties" and K > 1:
        # the case is only a test if f32 and f64 disagree somewhere
        p64, _ = po.decode_batch(A, B, obs, off, nthreads=8)
        assert (p64 != rp).any(), "f32 and f64 agree everywhere: the model does not separate them"
    h.close()


def test_f32_mode_host_pipelines_and_chunks():
    """Every host path (streamed copies past one launch / one launch per chunk, backtrace next to or after the forward
    kernel) with forced chunk counts.  16 chunks of a 30 000-sequence call are below 8192 sequences each: the f32
    routing is decided once per call, so they must still be decoded in f32."""
    rng = np.random.default_rng(77)
    K, M, Bn = 45, 40, 30000
    A, B = _model("round_ties", K, M, rng)
    obs, off = _ragged_batch(rng, Bn, M, tmax=25, nlong=4)
    rp, rs = nv.decode_batch(A, B, obs, off, np.float32)
    h = cv.HMM(A, B, np.zeros(K))
    L = cv._lib.lib()
    try:
        for conc, streamed in ((1, 1), (1, 0), (0, 0)):
            L.cv_debug_set_pipeline(conc, streamed)
            for chunks in (-1, 2, 5, 16):
                L.cv_debug_set_chunks(chunks)
                for rep in range(2):                            # second call reuses flags / counters / buffers
                    p, s = cv.decode_batch_f32(h, obs, off)
                    _assert_f32_equal(p, s, rp, rs, f"conc={conc} streamed={streamed} chunks={chunks} rep={rep}")
    finally:
        L.cv_debug_set_pipeline(1, 1)
        L.cv_debug_set_chunks(-1)
    h.close()


def test_f32_mode_routing_is_decided_per_call():
    """A call of EXACT_MAX_B sequences returns the exact f64 result (score bytes of the C oracle), one more sequence
    the f32 result, whatever the chunk count and the chain-kernel override say."""
    rng = np.random.default_rng(78)
    K, M = 33, 20
    A, B = _model("round_ties", K, M, rng)
    obs, off = _ragged_batch(rng, EXACT_MAX_B + 1, M, tmax=20, nlong=1)
    r32p, r32s = nv.decode_batch(A, B, obs, off, np.float32)
    sm_obs, sm_off = obs[:off[EXACT_MAX_B]], off[:EXACT_MAX_B + 1]
    r64p, r64s = po.decode_batch(A, B, sm_obs, sm_off, nthreads=8)
    assert (r32p[:off[EXACT_MAX_B]] != r64p).any()            # the two results are distinguishable
    h = cv.HMM(A, B, np.zeros(K))
    L = cv._lib.lib()
    try:
        for chain_max in (-1, 0, 1 << 20):
            L.cv_debug_set_chain_max_batch(chain_max)
            for chunks in (-1, 1, 3, 16):
                L.cv_debug_set_chunks(chunks)
                p, s = cv.decode_batch_f32(h, sm_obs, sm_off)
                assert (p == r64p).all() and s.tobytes() == r64s.tobytes(), ("exact", chain_max, chunks)
                p, s = cv.decode_batch_f32(h, obs, off)
                _assert_f32_equal(p, s, r32p, r32s, f"f32 chain_max={chain_max} chunks={chunks}")
    finally:
        L.cv_debug_set_chain_max_batch(-1)
        L.cv_debug_set_chunks(-1)
    h.close()


def test_f32_device_entry_on_a_user_stream():
    """cv_decode_batch_dev_f32 on a user stream with max_len exact, larger than needed and <= 0 (not known), and with
    forced chunks; two calls return identical bytes."""
    import torch
    rng = np.random.default_rng(79)
    K, M, Bn = 47, 30, 20000
    A, B = _model("ties", K, M, rng)
    obs, off = _ragged_batch(rng, Bn, M, tmax=40, nlong=2)
    rp, rs = nv.decode_batch(A, B, obs, off, np.float32)
    h = cv.HMM(A, B, np.zeros(K))
    L = cv._lib.lib()
    hd = h.device_handle(torch.cuda.current_device())
    N = len(obs)
    d_obs = torch.from_numpy(obs.view(np.int32)).cuda()
    d_off = torch.from_numpy(off).cuda()
    true_max = int(np.diff(off).max())
    st = torch.cuda.Stream()
    try:
        for chunks, max_lens in ((-1, (true_max, 3 * true_max + 5, 0, -1)), (3, (true_max, 2 * true_max))):
            L.cv_debug_set_chunks(chunks)
            for ml in max_lens:
                got = []
                for _ in range(2):
                    d_path = torch.full((N,), -1, dtype=torch.int32, device="cuda")
                    d_score = torch.full((Bn,), np.nan, dtype=torch.float64, device="cuda")
                    torch.cuda.synchronize()
                    with torch.cuda.stream(st):
                        cv._lib.check(L.cv_decode_batch_dev_f32(hd, d_obs.data_ptr(), d_off.data_ptr(), Bn, N, ml,
                                                                d_path.data_ptr(), d_score.data_ptr(), st.cuda_stream, 1))
                    st.synchronize()
                    got.append((d_path.cpu().numpy().view(np.uint32), d_score.cpu().numpy()))
                _assert_f32_equal(got[0][0], got[0][1], rp, rs, f"chunks={chunks} max_len={ml}")
                assert got[0][0].tobytes() == got[1][0].tobytes() and got[0][1].tobytes() == got[1][1].tobytes(), ml
    finally:
        L.cv_debug_set_chunks(-1)
    h.close()
