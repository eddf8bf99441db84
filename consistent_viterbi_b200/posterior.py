"""Forward-backward inference on the GPU (cv_loglik_batch / cv_posterior_batch, include/cv_b200.h): per-sequence
log10 P(O), posterior marginals gamma_t(i) = P(s_t = i | O) and posterior (maximum posterior marginal) decoding.

The model is the HMM's log10 entries read as probabilities; unlike `decode`, pi and the first observation count, as in
`HMM.train`.  A sequence with P(O) = 0 gets loglik -inf, posterior rows of 0.0, path 0 and pmax 0.0.  K <= 64."""
from __future__ import annotations

import numpy as np

from . import _lib
from .hmm import HMM


def _arrays(obs_flat, seq_off):
    obs_flat = np.ascontiguousarray(obs_flat, dtype=np.uint32)
    seq_off = np.ascontiguousarray(seq_off, dtype=np.int64)
    B = seq_off.shape[0] - 1
    if B > 0 and int(seq_off[-1]) != obs_flat.shape[0]:
        raise ValueError("seq_off[-1] != len(obs_flat)")
    return obs_flat, seq_off, max(B, 0)


def loglik_batch(hmm: HMM, obs_flat, seq_off, device: int = -1) -> np.ndarray:
    """log10 P(O) of every sequence, f64[B] (-inf where P(O) = 0).  obs_flat u32[N], seq_off i64[B+1]."""
    obs_flat, seq_off, B = _arrays(obs_flat, seq_off)
    ll = np.zeros(B, dtype=np.float64)
    rc = _lib.lib().cv_loglik_batch(hmm.device_handle(device), obs_flat.ctypes.data, seq_off.ctypes.data, B,
                                    ll.ctypes.data)
    _lib.check(rc)
    return ll


def posterior_batch(hmm: HMM, obs_flat, seq_off, device: int = -1, want_posteriors: bool = False) -> dict:
    """Posterior decoding of every sequence.  Returns dict(path u32[N] = lowest argmax of each posterior row,
    pmax f64[N] = that maximum, loglik f64[B], post f64[N, K] = gamma_t(i) of every position, or None unless
    want_posteriors)."""
    obs_flat, seq_off, B = _arrays(obs_flat, seq_off)
    N, K = obs_flat.shape[0], hmm.nstates()
    path = np.zeros(N, dtype=np.uint32)
    pmax = np.zeros(N, dtype=np.float64)
    ll = np.zeros(B, dtype=np.float64)
    post = np.zeros((N, K), dtype=np.float64) if want_posteriors else None
    rc = _lib.lib().cv_posterior_batch(hmm.device_handle(device), obs_flat.ctypes.data, seq_off.ctypes.data, B,
                                       path.ctypes.data, pmax.ctypes.data,
                                       post.ctypes.data if post is not None else None, ll.ctypes.data)
    _lib.check(rc)
    return dict(path=path, pmax=pmax, loglik=ll, post=post)


def score(hmm: HMM, sequences, device: int = -1) -> float:
    """Summed log10 P(O) of a list of [T, D] observation sequences (flattened with hmm.flatten_obs): the held-out
    score by which to compare models.  -inf if any sequence is impossible under the model."""
    obs = [hmm.flatten_obs(sq) for sq in sequences]
    off = np.zeros(len(obs) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(o) for o in obs])
    obs_flat = np.concatenate(obs) if obs else np.zeros(0, dtype=np.uint32)
    return float(loglik_batch(hmm, obs_flat, off, device).sum())
