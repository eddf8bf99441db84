"""The f32 forward kernel of long batches (decode_f32_fwd_kernel<4>: 64 registers, so that the concurrent backtrace fits
beside it; launch_decode_small runs it above 1300 sequences per SM and the 78-register build below).  Every state-group
count G = ceil(K / 8) changes the forward CTA's size and the residency budget of the concurrent launch.

- certified exact decode: the same bytes as the forced f64 path;
- f32 mode: the same bytes as the same call decoded in chunks short enough for the 78-register build."""
import numpy as np
import pytest

import consistent_viterbi_b200 as cv
from util import random_hmm

pytestmark = pytest.mark.gpu


def _batch(rng, M, Bn):
    lens = rng.integers(1, 13, size=Bn)
    off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    return rng.integers(0, M, size=int(off[-1])).astype(np.uint32), off


def _dev(h, fn, obs, off):
    import torch
    hd = h.device_handle(torch.cuda.current_device())
    Bn, N = len(off) - 1, len(obs)
    d_obs = torch.from_numpy(obs.view(np.int32)).cuda()
    d_off = torch.from_numpy(off).cuda()
    d_path = torch.full((N,), -1, dtype=torch.int32, device="cuda")
    d_score = torch.full((Bn,), np.nan, dtype=torch.float64, device="cuda")
    cv._lib.check(fn(hd, d_obs.data_ptr(), d_off.data_ptr(), Bn, N, int(np.diff(off).max()), d_path.data_ptr(),
                     d_score.data_ptr(), torch.cuda.current_stream().cuda_stream, 1))
    torch.cuda.synchronize()
    return d_path.cpu().numpy(), d_score.cpu().numpy()


def _same(a, b, what):
    assert a[0].tobytes() == b[0].tobytes(), f"{what}: paths differ"
    assert a[1].tobytes() == b[1].tobytes(), f"{what}: score bytes differ"


@pytest.mark.parametrize("K", [1, 8, 9, 33, 45, 57, 64])
def test_long_batch_certified_and_f32(K):
    import torch
    L = cv._lib.lib()
    Bn = 1400 * torch.cuda.get_device_properties(0).multi_processor_count
    rng = np.random.default_rng(60_000 + K)
    M = 37
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.3)
    obs, off = _batch(rng, M, Bn)
    h = cv.HMM(A, B, pi)
    L.cv_debug_set_certified(0)
    try:
        ref = _dev(h, L.cv_decode_batch_dev, obs, off)
    finally:
        L.cv_debug_set_certified(1)
    _same(_dev(h, L.cv_decode_batch_dev, obs, off), ref, f"K={K} certified")
    assert L.cv_debug_last_flagged(h.device_handle(torch.cuda.current_device())) >= 0, "the certified path must run"
    f32 = _dev(h, L.cv_decode_batch_dev_f32, obs, off)
    L.cv_debug_set_chunks(4)
    try:
        _same(_dev(h, L.cv_decode_batch_dev_f32, obs, off), f32, f"K={K} f32 in four chunks")
    finally:
        L.cv_debug_set_chunks(-1)
    h.close()
