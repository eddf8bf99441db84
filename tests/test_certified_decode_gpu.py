"""The certified exact decode (K <= 64, models of log-probabilities): f32 forward pass, a backtrace that certifies every
backpointer against an error bound of the f64 recurrence (decode_small.cuh), f64 re-decode of the sequences it cannot
certify.  Its results must be the f64 results bit for bit: the same bytes as the forced f64 path and as the C oracle.

Batches have more than 8192 sequences: smaller ones go to the warp-per-sequence f64 kernel and are never certified."""
import ctypes as C

import numpy as np
import pytest

import consistent_viterbi_b200 as cv
from oracle import pyoracle as po
from util import random_hmm

pytestmark = pytest.mark.gpu

BN = 9000


def _batch(rng, M, Bn=BN, tmax=12, nlong=0):
    """Bn sequences, a third of length 1, the rest 2..tmax, plus `nlong` of 300-600 steps (the long-sequence split)."""
    lens = rng.integers(2, tmax + 1, size=Bn)
    lens[rng.random(Bn) < 1 / 3] = 1
    if nlong:
        lens[rng.choice(Bn, size=nlong, replace=False)] = rng.integers(300, 601, size=nlong)
    off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    return rng.integers(0, M, size=int(off[-1])).astype(np.uint32), off


def _dev(h, obs, off, u8=False, scores=True):
    """cv_decode_batch_dev(_u8) on the current stream; returns (paths u32, scores or None, flagged count)."""
    import torch
    L = cv._lib.lib()
    hd = h.device_handle(torch.cuda.current_device())
    Bn, N = len(off) - 1, len(obs)
    d_obs = torch.from_numpy(obs.view(np.int32)).cuda()
    d_off = torch.from_numpy(off).cuda()
    d_path = torch.full((N,), 0xAB, dtype=torch.uint8, device="cuda") if u8 else torch.full((N,), -1, dtype=torch.int32, device="cuda")
    d_score = torch.full((Bn,), np.nan, dtype=torch.float64, device="cuda") if scores else None
    fn = L.cv_decode_batch_dev_u8 if u8 else L.cv_decode_batch_dev
    cv._lib.check(fn(hd, d_obs.data_ptr(), d_off.data_ptr(), Bn, N, int(np.diff(off).max()), d_path.data_ptr(),
                     d_score.data_ptr() if scores else None, torch.cuda.current_stream().cuda_stream, 1))
    torch.cuda.synchronize()
    p = d_path.cpu().numpy().astype(np.uint32) if u8 else d_path.cpu().numpy().view(np.uint32)
    return p, (d_score.cpu().numpy() if scores else None), int(L.cv_debug_last_flagged(hd))


def _f64(h, obs, off):
    L = cv._lib.lib()
    L.cv_debug_set_certified(0)
    try:
        p, s, n = _dev(h, obs, off)
    finally:
        L.cv_debug_set_certified(1)
    assert n == -1
    return p, s


def _same(p, s, rp, rs, what):
    bad = np.flatnonzero(p != rp)
    assert bad.size == 0, f"{what}: {bad.size} path elements differ, first at {bad[:5]}"
    if s is not None:
        assert s.tobytes() == rs.tobytes(), f"{what}: score bytes differ at {np.flatnonzero(s.view(np.uint64) != rs.view(np.uint64))[:5]}"


@pytest.mark.parametrize("K", list(range(1, 65)))
def test_certified_equals_f64_and_oracle(K):
    """Every K: device entry (u32 and u8 paths, with and without scores) and the one-piece host path against the forced
    f64 path and the oracle.  Every third K has half its probabilities zero (-inf-heavy); every fourth adds long
    sequences that the long-sequence split hands to the f64 warp kernel."""
    rng = np.random.default_rng(50_000 + K)
    M = 23
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.6 if K % 3 == 0 else 0.1)
    obs, off = _batch(rng, M, nlong=3 if K % 4 == 0 else 0)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    h = cv.HMM(A, B, pi)
    fp, fs = _f64(h, obs, off)
    _same(fp, fs, rp, rs, f"K={K} forced f64")
    p, s, n = _dev(h, obs, off)
    assert n >= 0, "an eligible model must take the certified path"
    _same(p, s, rp, rs, f"K={K} certified ({n} flagged)")
    p, _, n = _dev(h, obs, off, u8=True, scores=False)
    assert n >= 0
    _same(p, None, rp, None, f"K={K} certified u8, no scores")
    p, s = cv.decode_batch(h, obs, off)
    _same(p, s, rp, rs, f"K={K} host path")
    h.close()


def _near_tie_model(rng, K, M):
    """Dyadic log-probabilities moved by a few f64 ulps or by ~1e-7 relative: distinct in f64, most of them tied or
    misordered after rounding to f32."""
    base = np.array([-0.5, -1.0, -1.5, -2.0])

    def draw(shape):
        x = rng.choice(base, size=shape)
        ulps = rng.integers(-4, 5, size=shape).astype(np.float64)
        x = x + ulps * np.spacing(x)
        rel = rng.random(shape) < 0.3
        x[rel] *= 1.0 + rng.uniform(-2e-7, 2e-7, size=int(rel.sum()))
        return np.minimum(x, 0.0)
    return draw((K, K)), draw((K, M))


def test_near_ties_need_the_bound():
    """With the bound scaled to 0 the f32 path is taken as it is and differs from the f64 path (the test can see the
    error); with the default bound the result is exact and some sequences went to the fallback."""
    rng = np.random.default_rng(51)
    K, M = 45, 17
    A, B = _near_tie_model(rng, K, M)
    obs, off = _batch(rng, M, tmax=30)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    h = cv.HMM(A, B, np.zeros(K))
    L = cv._lib.lib()
    try:
        L.cv_debug_set_cert_tolerance(0.0)
        p, s, n = _dev(h, obs, off)
        assert n == 0
        assert (p != rp).any() or s.tobytes() != rs.tobytes(), "the near-tie model does not separate f32 from f64"
    finally:
        L.cv_debug_set_cert_tolerance(1.0)
    p, s, n = _dev(h, obs, off)
    assert n > 0
    _same(p, s, rp, rs, f"near ties, default bound ({n} flagged)")
    h.close()


@pytest.mark.parametrize("scale", [1.0, float("inf")])
def test_everything_to_the_fallback(scale):
    """A uniform model ties every decision (and the infinite bound certifies none): every sequence is re-decoded by
    the f64 tile path, the result is exact."""
    rng = np.random.default_rng(52)
    K, M = 33, 11
    if scale == 1.0:
        A, B = np.full((K, K), np.log10(1.0 / K)), np.full((K, M), np.log10(1.0 / M))
    else:
        A, B, _ = random_hmm(rng, K, M, zero_frac=0.2)
    obs, off = _batch(rng, M)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    h = cv.HMM(A, B, np.zeros(K))
    L = cv._lib.lib()
    try:
        L.cv_debug_set_cert_tolerance(scale)
        p, s, n = _dev(h, obs, off)
    finally:
        L.cv_debug_set_cert_tolerance(1.0)
    assert n == BN
    _same(p, s, rp, rs, f"all flagged, scale {scale}")
    h.close()


@pytest.mark.parametrize("kind", ["positive", "beyond_2_64", "k_above_64"])
def test_ineligible_models_take_the_f64_path(kind):
    rng = np.random.default_rng(53)
    K, M = (70 if kind == "k_above_64" else 20), 13
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.1)
    if kind == "positive":
        A[0, 1] = 0.25
    elif kind == "beyond_2_64":
        B[2, 3] = -2.0 ** 65
    obs, off = _batch(rng, M, tmax=6)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    h = cv.HMM(A, B, pi)
    p, s, n = _dev(h, obs, off)
    assert n == -1
    _same(p, s, rp, rs, kind)
    h.close()
