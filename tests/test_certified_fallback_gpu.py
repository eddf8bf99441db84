"""Routes of the certified decode's f64 re-decode (certified_fallback, cv_api.cu): every flagged sequence on the tile path,
every one on the warp-per-sequence kernel, or the longest of them on the warp-per-sequence kernel beside the tile path.
Each route must give the forced f64 path's bytes and the C oracle's, and the route a call took is asserted from
cv_debug_last_fallback_chain.

Batches have more than 8192 sequences (smaller ones are never certified) with lengths up to 500 steps, so that the
flagged sequences span many tiles and their longest ones are far longer than the rest.  The main pass hands 4096 of the
longest to its own warp-per-sequence kernel (long-sequence split), so they are never flagged.  On the near-tie model about
12 000 others are flagged (the automatic route splits them); on the uniform model the bound is scaled to infinity, so
that about 20 000 are flagged: more than two tiles per SM, where the automatic route keeps them all on the tile path."""
import numpy as np
import pytest

import consistent_viterbi_b200 as cv
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu


def _batch(rng, M, BN):
    """BN sequences: 40 % of 1-20 steps, 40 % of 21-120, 20 % of 121-500."""
    u = rng.random(BN)
    lens = np.where(u < 0.4, rng.integers(1, 21, BN), np.where(u < 0.8, rng.integers(21, 121, BN), rng.integers(121, 501, BN)))
    off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    return rng.integers(0, M, size=int(off[-1])).astype(np.uint32), off


def _near_tie_model(rng, K, M):
    """Dyadic log-probabilities moved by a few f64 ulps or by ~1e-7 relative: most decisions tied or misordered in f32."""
    base = np.array([-0.5, -1.0, -1.5, -2.0])

    def draw(shape):
        x = rng.choice(base, size=shape)
        x = x + rng.integers(-4, 5, size=shape).astype(np.float64) * np.spacing(x)
        rel = rng.random(shape) < 0.3
        x[rel] *= 1.0 + rng.uniform(-2e-7, 2e-7, size=int(rel.sum()))
        return np.minimum(x, 0.0)
    return draw((K, K)), draw((K, M))


_CASES = {}


def _case(name):
    """(model handle, obs, off, oracle paths, oracle scores) of one workload, built once per module."""
    if name not in _CASES:
        if name == "near_tie":                 # K = 45: the warp kernel reads logA from shared memory
            rng = np.random.default_rng(61)
            K, M = 45, 17
            A, B = _near_tie_model(rng, K, M)
            obs, off = _batch(rng, M, 16000)
        else:                                  # uniform, K = 20: the warp kernel keeps its logA column in registers
            rng = np.random.default_rng(62)
            K, M = 20, 11
            A, B = np.full((K, K), np.log10(1.0 / K)), np.full((K, M), np.log10(1.0 / M))
            obs, off = _batch(rng, M, 24000)
        rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
        _CASES[name] = (cv.HMM(A, B, np.zeros(K)), obs, off, rp, rs)
    return _CASES[name]


def _dev(h, obs, off, u8, scores, tol=1.0):
    """cv_decode_batch_dev(_u8) on the current stream with the certified bound scaled by tol: (paths u32, scores or
    None, flagged, flagged on the warp kernel)."""
    import torch
    L = cv._lib.lib()
    hd = h.device_handle(torch.cuda.current_device())
    Bn, N = len(off) - 1, len(obs)
    d_obs = torch.from_numpy(obs.view(np.int32)).cuda()
    d_off = torch.from_numpy(off).cuda()
    d_path = torch.full((N,), 0xAB, dtype=torch.uint8, device="cuda") if u8 else torch.full((N,), -1, dtype=torch.int32, device="cuda")
    d_score = torch.full((Bn,), np.nan, dtype=torch.float64, device="cuda") if scores else None
    fn = L.cv_decode_batch_dev_u8 if u8 else L.cv_decode_batch_dev
    L.cv_debug_set_cert_tolerance(tol)
    try:
        cv._lib.check(fn(hd, d_obs.data_ptr(), d_off.data_ptr(), Bn, N, int(np.diff(off).max()), d_path.data_ptr(),
                         d_score.data_ptr() if scores else None, torch.cuda.current_stream().cuda_stream, 1))
    finally:
        L.cv_debug_set_cert_tolerance(1.0)
    torch.cuda.synchronize()
    p = d_path.cpu().numpy().astype(np.uint32) if u8 else d_path.cpu().numpy().view(np.uint32)
    return p, (d_score.cpu().numpy() if scores else None), int(L.cv_debug_last_flagged(hd)), int(L.cv_debug_last_fallback_chain(hd))


def _same(p, s, rp, rs, what):
    bad = np.flatnonzero(p != rp)
    assert bad.size == 0, f"{what}: {bad.size} path elements differ, first at {bad[:5]}"
    if s is not None:
        assert s.tobytes() == rs.tobytes(), f"{what}: score bytes differ at {np.flatnonzero(s.view(np.uint64) != rs.view(np.uint64))[:5]}"


def test_forced_f64_equals_oracle():
    L = cv._lib.lib()
    for name in ("near_tie", "uniform"):
        h, obs, off, rp, rs = _case(name)
        L.cv_debug_set_certified(0)
        try:
            p, s, n, _ = _dev(h, obs, off, False, True)
        finally:
            L.cv_debug_set_certified(1)
        assert n == -1
        _same(p, s, rp, rs, f"{name}: forced f64")


# route: (cv_debug_set_fallback route, n_chain); "n-1" / "n+7" / "half" are relative to the flagged count
ROUTES = {
    "auto": (0, 0), "tile": (1, 0), "chain": (2, 0), "split0": (3, 0), "split1": (3, 1), "split64": (3, 64),
    "split65": (3, 65), "split_half": (3, "half"), "split_n-1": (3, "n-1"), "split_n+7": (3, "n+7"),
}


@pytest.mark.parametrize("route", list(ROUTES))
@pytest.mark.parametrize("name", ["near_tie", "uniform"])
def test_fallback_route(name, route):
    import torch
    L = cv._lib.lib()
    h, obs, off, rp, rs = _case(name)
    tol = float("inf") if name == "uniform" else 1.0
    _, _, n, _ = _dev(h, obs, off, False, False, tol)       # the flagged count (automatic route)
    assert n > 8192
    r, k = ROUTES[route]
    k = {"half": n // 2, "n-1": n - 1, "n+7": n + 7}.get(k, k)
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    auto = n if n <= 8192 else 0 if n > 2 * 64 * sms else min(n, 2 * sms)
    want = {0: auto, 1: 0, 2: n, 3: min(max(k, 0), n)}[r]
    L.cv_debug_set_fallback(r, k)
    try:
        for u8, scores in ((False, True), (True, False), (True, True), (False, False)):
            p, s, nf, nc = _dev(h, obs, off, u8, scores, tol)
            assert nf == n
            assert nc == want, f"{name} {route}: {nc} flagged sequences on the warp kernel, expected {want}"
            _same(p, s, rp, rs if scores else None, f"{name} {route} u8={u8} scores={scores}")
    finally:
        L.cv_debug_set_fallback(0, 0)
