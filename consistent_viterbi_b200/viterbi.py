"""Plain Viterbi, mirror of `viterbi::decode` (src/viterbi_solver/viterbi.rs:5-32).

`decode(sequence, hmm)` keeps the reference's signature and return value (state
path, one entry per element); `decode_batch` is the batched form the GPU path is
built for.  Both run on the GPU through the C ABI -- there is no CPU path."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .hmm import HMM


def decode_batch(hmm: HMM, obs_flat, seq_off, device: int = -1, want_scores: bool = True):
    """B independent viterbi::decode calls.

    obs_flat u32[N] flattened observations, seq_off i64[B+1].  Returns
    (paths u32[N], scores f64[B]) with scores[b] = delta[T-1][end] of sequence b."""
    obs_flat = np.ascontiguousarray(obs_flat, dtype=np.uint32)
    seq_off = np.ascontiguousarray(seq_off, dtype=np.int64)
    B = seq_off.shape[0] - 1
    N = obs_flat.shape[0]
    if B > 0 and int(seq_off[-1]) != N:
        raise ValueError("seq_off[-1] != len(obs_flat)")
    paths = np.zeros(N, dtype=np.uint32)
    scores = np.zeros(max(B, 0), dtype=np.float64)
    h = hmm.device_handle(device)
    rc = _lib.lib().cv_decode_batch(h, obs_flat.ctypes.data, seq_off.ctypes.data, B, paths.ctypes.data,
                                    scores.ctypes.data if want_scores else None)
    _lib.check(rc)
    return paths, scores


def decode_batch_f32(hmm: HMM, obs_flat, seq_off, device: int = -1):
    """OPTIONAL f32 mode (cv_decode_batch_f32): the recurrence in IEEE binary32, paths = the optimum of the f32
    recurrence (may differ from the f64 path at near-ties).  For models with every entry <= 0 a score is within about
    2 T 2^-24 relative of the exact mode for a sequence of T steps (measured: 4.8e-7 at T = 80, 9.5e-6 at T = 20 000).
    Not the parity path."""
    obs_flat = np.ascontiguousarray(obs_flat, dtype=np.uint32)
    seq_off = np.ascontiguousarray(seq_off, dtype=np.int64)
    B, N = seq_off.shape[0] - 1, obs_flat.shape[0]
    paths = np.zeros(N, dtype=np.uint32)
    scores = np.zeros(max(B, 0), dtype=np.float64)
    rc = _lib.lib().cv_decode_batch_f32(hmm.device_handle(device), obs_flat.ctypes.data, seq_off.ctypes.data, B,
                                        paths.ctypes.data, scores.ctypes.data)
    _lib.check(rc)
    return paths, scores


def decode_batch_narrow(hmm: HMM, obs_flat, seq_off, device: int = -1):
    """decode_batch with narrow host formats (cv_decode_batch_u16u8): observations cross PCIe as u16 (M <= 65536),
    states come back as u8 (K <= 64 here).  Same results; returns (paths u8[N], scores f64[B])."""
    obs16 = np.ascontiguousarray(obs_flat, dtype=np.uint16)
    if (np.asarray(obs_flat) != obs16).any():
        raise ValueError("observation does not fit u16")
    seq_off = np.ascontiguousarray(seq_off, dtype=np.int64)
    B, N = seq_off.shape[0] - 1, obs16.shape[0]
    if B > 0 and int(seq_off[-1]) != N:
        raise ValueError("seq_off[-1] != len(obs_flat)")
    paths = np.zeros(N, dtype=np.uint8)
    scores = np.zeros(max(B, 0), dtype=np.float64)
    rc = _lib.lib().cv_decode_batch_u16u8(hmm.device_handle(device), obs16.ctypes.data, seq_off.ctypes.data, B,
                                          paths.ctypes.data, scores.ctypes.data)
    _lib.check(rc)
    return paths, scores


def decode_batch_kbest(hmm: HMM, obs_flat, seq_off, k: int, device: int = -1):
    """The k highest-scoring state paths of every sequence (cv_decode_batch_kbest, contract in include/cv_b200.h).

    obs_flat u32[N], seq_off i64[B+1].  Returns (paths u32[k, N], scores f64[k, B]): row r holds rank r laid out as
    decode_batch's outputs, and row 0 is decode_batch's result byte for byte.  A sequence of T elements has
    min(k, K^T) paths; a rank beyond that is "no path": score -inf, every path element 0xFFFFFFFF.  K <= 64, k <= 32."""
    obs_flat = np.ascontiguousarray(obs_flat, dtype=np.uint32)
    seq_off = np.ascontiguousarray(seq_off, dtype=np.int64)
    B, N = seq_off.shape[0] - 1, obs_flat.shape[0]
    if B > 0 and int(seq_off[-1]) != N:
        raise ValueError("seq_off[-1] != len(obs_flat)")
    kk = max(int(k), 0)
    paths = np.zeros((kk, N), dtype=np.uint32)
    scores = np.zeros((kk, max(B, 0)), dtype=np.float64)
    rc = _lib.lib().cv_decode_batch_kbest(hmm.device_handle(device), obs_flat.ctypes.data, seq_off.ctypes.data, B,
                                          int(k), paths.ctypes.data, scores.ctypes.data)
    _lib.check(rc)
    return paths, scores


def decode_kbest(sequence, hmm: HMM, k: int, device: int = -1) -> list:
    """The k best state paths of one sequence as a list of (path u64[T], score), best first; fewer than k when the
    sequence has fewer than k paths."""
    obs = hmm.flatten_obs(sequence) if len(sequence) else np.zeros(0, dtype=np.uint32)
    off = np.array([0, len(obs)], dtype=np.int64)
    paths, scores = decode_batch_kbest(hmm, obs, off, k, device=device)
    return [(paths[r].astype(np.uint64), float(scores[r, 0])) for r in range(paths.shape[0]) if paths[r, 0] != 0xFFFFFFFF]


def decode(sequence, hmm: HMM, device: int = -1) -> np.ndarray:
    """viterbi::decode(sequence, hmm) -> Array1<usize> (viterbi.rs:5). `sequence` is a
    list of D-dimensional observations (Vec<[usize; D]>)."""
    obs = hmm.flatten_obs(sequence) if len(sequence) else np.zeros(0, dtype=np.uint32)
    off = np.array([0, len(obs)], dtype=np.int64)
    paths, _ = decode_batch(hmm, obs, off, device=device, want_scores=False)
    return paths.astype(np.uint64)
