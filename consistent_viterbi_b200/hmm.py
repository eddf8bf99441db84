"""HMM container mirroring the reference's `struct HMM<D>{a,b,pi}` (src/hmm/hmm.rs:10-18)
and its accessors (hmm.rs:207-234).  All values are log10 probabilities, zero
probability is -inf (hmm.rs:192-205).  `device_handle()` uploads the model through
the C ABI (cv_hmm_create); nothing here computes Viterbi on the CPU."""
from __future__ import annotations

import ctypes as C
import json
import math

import numpy as np

from . import _lib


class HMM:
    def __init__(self, a, b, pi):
        """a[K,K] (from,to); b[K, *bdims]; pi[K] -- hmm.rs:11-17."""
        self.a = np.ascontiguousarray(a, dtype=np.float64)
        self.b = np.ascontiguousarray(b, dtype=np.float64)
        self.pi = np.ascontiguousarray(pi, dtype=np.float64)
        K = self.a.shape[0]
        if self.a.shape != (K, K) or self.b.shape[0] != K or self.pi.shape != (K,):
            raise ValueError("inconsistent HMM shapes")
        if self.b.ndim < 2:
            raise ValueError("b must be [K, *bdims]")
        self.bdims = tuple(int(x) for x in self.b.shape[1:])
        self._handles = {}

    # ---- construction / supervised training (hmm.rs:22-62) ----
    @classmethod
    def new(cls, nstates: int, bdims, rng=None):
        """HMM::new (hmm.rs:22-28): a random row-normalised model.  The reference draws from `thread_rng()` (not
        reproducible by construction); pass a numpy Generator, or rng=None for the all-zero model that turns
        maximum_likelihood_estimation into the plain count-based estimate."""
        bdims = tuple(int(x) for x in bdims)
        if rng is None:
            return cls(np.zeros((nstates, nstates)), np.zeros((nstates,) + bdims), np.zeros(nstates))
        a = rng.random((nstates, nstates))
        b = rng.random((nstates,) + bdims)
        pi = rng.random(nstates)
        a /= a.sum(axis=1, keepdims=True)
        b /= b.reshape(nstates, -1).sum(axis=1).reshape((nstates,) + (1,) * len(bdims))
        return cls(a, b, pi / pi.sum())

    def maximum_likelihood_estimation(self, sequences, tags, device: int = -1):
        """HMM::maximum_likelihood_estimation + log (hmm.rs:30-62,192-205) through cv_mle: events are counted on
        the GPU and added on top of this model's current (probability) values exactly as the reference's
        `+= 1.0` loop would; afterwards a, b, pi hold ln(x)/ln(10) (-inf for 0).
        sequences: list of [T, D] observation arrays, tags: list of tag lists (None / -1 = missing -> error)."""
        self.close()                                                     # device copies become stale
        obs = [self.flatten_obs(sq) for sq in sequences]
        off = np.zeros(len(obs) + 1, dtype=np.int64)
        off[1:] = np.cumsum([len(o) for o in obs])
        obs_flat = np.concatenate(obs) if obs else np.zeros(0, dtype=np.uint32)
        tg = np.array([(-1 if t is None else int(t)) for tl in tags for t in tl], dtype=np.int32)
        if len(tg) != len(obs_flat):
            raise ValueError("sequences and tags differ in length")
        return self.mle_arrays(obs_flat, tg, off, device)

    def mle_arrays(self, obs_flat, tags_flat, seq_off, device: int = -1):
        """cv_mle on flat arrays; returns the device time (ms) of the counting kernels."""
        obs_flat = np.ascontiguousarray(obs_flat, dtype=np.uint32)
        tags_flat = np.ascontiguousarray(tags_flat, dtype=np.int32)
        seq_off = np.ascontiguousarray(seq_off, dtype=np.int64)
        K = self.nstates()
        bd = (C.c_uint64 * len(self.bdims))(*self.bdims)
        ms = C.c_double(0.0)
        rc = _lib.lib().cv_mle(K, len(self.bdims), bd, self.a.ctypes.data, self.b.ctypes.data, self.pi.ctypes.data,
                               obs_flat.ctypes.data, tags_flat.ctypes.data, seq_off.ctypes.data, len(seq_off) - 1,
                               int(device), C.byref(ms))
        _lib.check(rc)
        return ms.value

    # ---- unsupervised training: Baum-Welch (cv_baum_welch) ----
    def train(self, sequences, n_iter: int = 10, tol: float = 0.0, device: int = -1):
        """HMM::train's role (hmm.rs:69-190) with the semantics of cv_baum_welch (include/cv_b200.h), which this
        library defines and does not restate from hmm.rs: Baum-Welch EM from the current model on the GPU.  Unlike
        decoding, pi and the first observation of every sequence count.  sequences: list of [T, D] observation arrays.
        Updates a, b, pi in place; returns what train_arrays returns."""
        obs = [self.flatten_obs(sq) for sq in sequences]
        off = np.zeros(len(obs) + 1, dtype=np.int64)
        off[1:] = np.cumsum([len(o) for o in obs])
        obs_flat = np.concatenate(obs) if obs else np.zeros(0, dtype=np.uint32)
        return self.train_arrays(obs_flat, off, n_iter, tol, device)

    def train_arrays(self, obs_flat, seq_off, n_iter: int = 10, tol: float = 0.0, device: int = -1):
        """cv_baum_welch on flat arrays.  Returns dict(loglik = log10 P(O) before each iteration's update, summed over
        the contributing sequences; iters = iterations run; skipped = sequences with P(O) = 0 in the last iteration;
        device_ms)."""
        self.close()                                                     # device copies become stale
        obs_flat = np.ascontiguousarray(obs_flat, dtype=np.uint32)
        seq_off = np.ascontiguousarray(seq_off, dtype=np.int64)
        K = self.nstates()
        b2 = np.ascontiguousarray(self.b.reshape(K, -1))
        bd = (C.c_uint64 * len(self.bdims))(*self.bdims)
        ll = np.zeros(max(int(n_iter), 1), dtype=np.float64)
        iters, skipped, ms = C.c_int(0), C.c_int64(0), C.c_double(0.0)
        rc = _lib.lib().cv_baum_welch(K, len(self.bdims), bd, self.a.ctypes.data, b2.ctypes.data, self.pi.ctypes.data,
                                      obs_flat.ctypes.data, seq_off.ctypes.data, len(seq_off) - 1, int(n_iter),
                                      float(tol), int(device), ll.ctypes.data_as(C.POINTER(C.c_double)),
                                      C.byref(iters), C.byref(skipped), C.byref(ms))
        _lib.check(rc)
        self.b = b2.reshape(self.b.shape)
        return dict(loglik=ll[: iters.value].copy(), iters=iters.value, skipped=skipped.value, device_ms=ms.value)

    # ---- reference accessors (host-side, used by SuperSequence.reorder and tests) ----
    def nstates(self) -> int:                       # hmm.rs:207-209
        return self.a.shape[0]

    def nobs(self) -> int:
        return int(np.prod(self.bdims))

    def flatten_obs(self, values) -> np.ndarray:
        """Row-major flattening of D-dimensional observations over bdims (b[state][&obs[..]])."""
        v = np.asarray(values, dtype=np.int64)
        if v.ndim == 1 and len(self.bdims) == 1:
            v = v[:, None]
        v = v.reshape(-1, v.shape[-1])
        D = len(self.bdims)
        if v.shape[1] < D:  # load_sequences leaves missing features at 0 (src/utils.rs:25-28)
            v = np.concatenate([v, np.zeros((v.shape[0], D - v.shape[1]), dtype=np.int64)], axis=1)
        flat = np.zeros(v.shape[0], dtype=np.int64)
        for d in range(D):
            if v.shape[0] and (v[:, d].min() < 0 or v[:, d].max() >= self.bdims[d]):
                raise IndexError("observation out of bounds (reference: ndarray index panic)")
            flat = flat * self.bdims[d] + v[:, d]
        return flat.astype(np.uint32)

    def emit_prob(self, state, obs_flat):           # hmm.rs:228-230
        return self.b.reshape(self.nstates(), -1)[state, obs_flat]

    def init_prob(self, state, obs_flat):           # hmm.rs:211-213
        return self.pi[state] + self.emit_prob(state, obs_flat)

    def transition_prob(self, f, t, obs_flat):      # hmm.rs:220-222
        return self.a[f, t] + self.emit_prob(t, obs_flat)

    # ---- hmm.json (ndarray-serde layout, hmm.rs:236-264) ----
    @staticmethod
    def _arr(x):
        def enc(v):
            return None if v == -math.inf else float(v)
        return {"v": 1, "dim": list(x.shape), "data": [enc(v) for v in x.reshape(-1)]}

    def write(self, path):
        """HMM::write (hmm.rs:236-240): field order a, b, pi; -inf serialises as null."""
        K = self.nstates()
        doc = {
            "a": self._arr(self.a),
            "b": {"v": 1, "dim": [K], "data": [self._arr(self.b[s]) for s in range(K)]},
            "pi": self._arr(self.pi),
        }
        with open(path, "w") as f:
            json.dump(doc, f, separators=(",", ":"))

    @classmethod
    def from_json(cls, path):
        """HMM::from_json (hmm.rs:242-264): null -> -inf."""
        with open(path) as f:
            doc = json.load(f)

        def dec(o):
            data = np.array([(-math.inf if v is None else v) for v in o["data"]], dtype=np.float64)
            return data.reshape(o["dim"])

        a = dec(doc["a"])
        b = np.stack([dec(o) for o in doc["b"]["data"]])
        return cls(a, b, dec(doc["pi"]))

    # ---- device ----
    def device_handle(self, device: int = -1):
        key = int(device)
        if key not in self._handles:
            L = _lib.lib()
            out = C.c_void_p()
            bd = (C.c_uint64 * len(self.bdims))(*self.bdims)
            K = self.nstates()
            b2 = np.ascontiguousarray(self.b.reshape(K, -1))
            rc = L.cv_hmm_create(K, len(self.bdims), bd,
                                 self.a.ctypes.data_as(C.POINTER(C.c_double)),
                                 b2.ctypes.data_as(C.POINTER(C.c_double)),
                                 self.pi.ctypes.data_as(C.POINTER(C.c_double)), key, C.byref(out))
            _lib.check(rc)
            self._handles[key] = out
        return self._handles[key]

    def close(self):
        for h in self._handles.values():
            _lib.lib().cv_hmm_destroy(h)
        self._handles.clear()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
