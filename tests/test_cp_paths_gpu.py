"""cv_cp_solve on every launch path its host code can choose, against the C oracle bit for bit: solution, objective
bits, explored nodes, sweep steps, every node's upper bound and (where it is small) the final delta / psi state.

Every case also asserts the path bits of cv_debug_cp_last_paths, so a case that a changed selection rule moves off
the path it names fails instead of silently covering something else.  Paths that only the environment selects
(CV_CP_SUM, CV_CP_HOSTPOLL, CV_CP_FULLWARP are read once, when the library loads) run in a subprocess."""
import os
import subprocess
import sys

import numpy as np
import pytest

import consistent_viterbi_b200 as cv
from oracle import pyoracle as po
from util import cp_path_bits, random_hmm, random_superseq

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TESTS = os.path.join(ROOT, "tests")


P = cp_path_bits()


def _names(bits):
    return sorted(n for n, b in P.items() if bits & b)


def _expect(paths, on=(), off=()):
    for n in on:
        assert paths & P[n], f"path {n} not taken; taken: {_names(paths)}"
    for n in off:
        assert not paths & P[n], f"path {n} taken; taken: {_names(paths)}"


def _check(A, B, pi, obs, start, comp, ncomp, max_nodes=0, state=True, leaf=1):
    """Solve on the GPU and with the oracle, compare everything; returns (path bits, GPU result)."""
    ref = po.cp_solve(A, B, pi, obs, start, comp, ncomp, max_nodes=max_nodes, trace_nodes=1 << 16, want_state=state)
    L = cv._lib.lib()
    h = cv.HMM(A, B, pi)
    L.cv_debug_set_cp_leaf_batch(leaf)
    try:
        got = cv.cp_solve_arrays(h, obs, start, comp, ncomp, max_nodes=max_nodes, want_state=state, want_ub=1 << 16)
        paths = L.cv_debug_cp_last_paths(h.device_handle())
    finally:
        L.cv_debug_set_cp_leaf_batch(1)
        h.close()
    assert got["explored"] == ref["explored"]
    assert got["steps"] == ref["steps"]
    n = min(len(got["ub"]), int(ref["explored"]))
    assert got["ub"][:n].tobytes() == ref["ub"][:n].tobytes(), "per-node upper bounds differ"
    assert np.float64(got["obj"]).tobytes() == np.float64(ref["obj"]).tobytes()
    bad = np.nonzero(got["sol"] != ref["sol"])[0]
    assert bad.size == 0, f"{bad.size} solution mismatches, first at {bad[:5]}"
    if state:
        assert got["delta"].tobytes() == ref["delta"].tobytes(), "final delta state differs"
        assert (got["psi"] == ref["psi"]).all(), "final psi state differs"
    return paths, got


def _compact(comp):
    """Renumber the components that occur to 0 .. ncomp-1 in order of first id."""
    used = np.unique(comp[comp >= 0])
    remap = np.full(int(comp.max()) + 2 if comp.size else 1, -1, dtype=np.int32)
    remap[used] = np.arange(used.size, dtype=np.int32)
    out = np.where(comp >= 0, remap[np.maximum(comp, 0)], -1).astype(np.int32)
    return out, int(used.size)


def _superseq_n(rng, N, M, tmin, tmax):
    """obs / is_seq_start of exactly N elements (sequence lengths tmin..tmax, the last one cut), nothing clamped."""
    lens = rng.integers(tmin, tmax + 1, size=N // tmin + 1)
    starts = np.cumsum(lens) - lens
    start = np.zeros(N, dtype=np.uint8)
    start[starts[starts < N]] = 1
    obs = rng.integers(0, M, size=N).astype(np.uint32)
    return obs, start, np.full(N, -1, dtype=np.int32)


def _clamp(rng, comp, ncomp, p_active):
    """Put a random p_active share of the rows into ncomp components; returns the compacted ids."""
    idx = np.nonzero(rng.random(comp.size) < p_active)[0]
    comp = comp.copy()
    comp[idx] = rng.integers(0, ncomp, size=idx.size)
    return _compact(comp)


# ---- sweep shapes ---------------------------------------------------------------------------------------------------
SWEEP = {7: "SWEEP_1_2_16", 8: "SWEEP_1_2_16", 15: "SWEEP_1_4_16", 16: "SWEEP_1_4_16", 25: "SWEEP_1_8",
         28: "SWEEP_1_8", 32: "SWEEP_1_8", 34: "SWEEP_2_0", 57: "SWEEP_2_0", 63: "SWEEP_2_0", 64: "SWEEP_2_0"}


@pytest.mark.parametrize("K", sorted(SWEEP))
def test_sweep_shapes_ties_odd_segments(K):
    """Every component has an odd number of positions, so every depth has an odd number of sweeps: with two
    segments per warp (K <= 16) the second half of the last warp has none.  Tied and -inf model entries, sequence
    starts inside the segments, leaf batch and node by node."""
    rng = np.random.default_rng(7100 + K)
    M = 10
    for ties in (True, False):
        A, B, pi = random_hmm(rng, K, M, zero_frac=0.15, ties=ties)
        obs, start, comp, ncomp = random_superseq(rng, 40, M, 3, 0.12, 1, 12)
        for c in range(ncomp):
            pos = np.nonzero(comp == c)[0]
            if pos.size % 2 == 0:
                comp[pos[-1]] = -1
        assert all(np.count_nonzero(comp == c) % 2 == 1 for c in range(ncomp))
        for leaf in (1, 0):
            paths, _ = _check(A, B, pi, obs, start, comp, ncomp, max_nodes=90, leaf=leaf)
            _expect(paths, on=[SWEEP[K], "BT_IN_SMEM"], off=[s for s in set(SWEEP.values()) if s != SWEEP[K]])


# ---- emissions from shared or global memory -----------------------------------------------------------------------
@pytest.mark.parametrize("M", [192, 193])
def test_emissions_smem_edge_k64(M):
    """K = 64: logB^T of M = 192 symbols is exactly 96 KB and is staged; one symbol more and the sweep reads it from
    global memory with L1 prefetch."""
    rng = np.random.default_rng(7300 + M)
    A, B, pi = random_hmm(rng, 64, M, zero_frac=0.0)
    obs, start, comp, ncomp = random_superseq(rng, 30, M, 2, 0.1, 2, 30)
    obs[::7] = M - 1                                              # the last row of logB^T is read
    paths, _ = _check(A, B, pi, obs, start, comp, ncomp, max_nodes=100)
    _expect(paths, on=["SWEEP_2_0", "LEAF_BATCH"] + (["BT_IN_SMEM"] if M == 192 else []),
            off=[] if M == 192 else ["BT_IN_SMEM"])


@pytest.mark.parametrize("leaf", [1, 0])
def test_pos_vocabulary_emissions_from_global(leaf):
    """A constrained POS-tagging shape: K = 45 with a 20 000-word vocabulary, logB^T far beyond shared memory."""
    rng = np.random.default_rng(7400)
    K, M = 45, 20000
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.0)
    obs, start, comp, ncomp = random_superseq(rng, 60, M, 2, 0.06, 5, 40)
    paths, _ = _check(A, B, pi, obs, start, comp, ncomp, max_nodes=120, leaf=leaf)
    _expect(paths, on=["SWEEP_2_0"] + (["LEAF_BATCH"] if leaf else []),
            off=["BT_IN_SMEM"] + ([] if leaf else ["LEAF_BATCH"]))


# ---- backtrack ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [399, 400])
def test_backtrack_rows_smem_edge(K):
    """256 psi rows of K = 399 states fit the backtrack's shared memory; from K = 400 on the maps and the fill walk
    psi in global memory."""
    rng = np.random.default_rng(7500 + K)
    M = 6
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.0)
    obs, start, comp = _superseq_n(rng, 300, M, 3, 20)
    comp[[255, 280]] = 0
    comp[[270, 295]] = 1
    paths, got = _check(A, B, pi, obs, start, comp, 2, max_nodes=5)
    assert got["obj"] > -np.inf                                  # a backtrack ran
    _expect(paths, on=["SWEEP_GENERIC"] + (["BTR_ROWS_GMEM"] if K >= 400 else []),
            off=["BTR_CHAIN_GMEM"] + ([] if K >= 400 else ["BTR_ROWS_GMEM"]))


@pytest.mark.parametrize("N", [256, 257, 258])
def test_backtrack_chunk_boundary(N):
    """N - 1 walked rows = 255, 256 (one chunk of CP_BT_CHUNK = 256 rows, full) and 257 (a second chunk of one row)."""
    rng = np.random.default_rng(7600 + N)
    K, M = 12, 7
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.0)
    obs, start, comp = _superseq_n(rng, N, M, 1, 30)
    comp, ncomp = _clamp(rng, comp, 2, 0.05)
    assert ncomp == 2
    paths, got = _check(A, B, pi, obs, start, comp, ncomp, max_nodes=60)
    assert got["obj"] > -np.inf
    _expect(paths, on=["SWEEP_1_4_16"], off=["BTR_ROWS_GMEM", "BTR_CHAIN_GMEM"])


# ---- generic sweep limit --------------------------------------------------------------------------------------------
def test_generic_sweep_limit():
    """K = 3200 is the largest model the generic sweep's shared memory holds (Kl = 3200); K = 3201 is refused."""
    rng = np.random.default_rng(7800)
    M = 4
    A, B, pi = random_hmm(rng, 3200, M, zero_frac=0.0)
    obs, start, comp = _superseq_n(rng, 24, M, 3, 10)
    comp[[17, 20]] = 0
    paths, got = _check(A, B, pi, obs, start, comp, 1, max_nodes=3)
    assert got["obj"] > -np.inf
    _expect(paths, on=["SWEEP_GENERIC", "BTR_ROWS_GMEM"])
    A, B, pi = random_hmm(rng, 3201, M, zero_frac=0.0)
    h = cv.HMM(A, B, pi)
    try:
        with pytest.raises(cv.CvError) as e:
            cv.cp_solve_arrays(h, obs, start, comp, 1, max_nodes=3)
        assert e.value.code == cv._lib.ERR_UNSUPPORTED
    finally:
        h.close()


# ---- bound sums inside a solve --------------------------------------------------------------------------------------
def test_leaf_batch_block_sum():
    """More than 4096 bound terms at K = 40: the leaf batch runs the block-structured sum with one list per sibling."""
    rng = np.random.default_rng(7900)
    K, M = 40, 16
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.0)
    obs, start, comp = _superseq_n(rng, 16000, M, 3, 30)
    comp, ncomp = _clamp(rng, comp, 2, 0.3)
    assert np.count_nonzero(comp >= 0) > 4096 and ncomp == 2
    paths, _ = _check(A, B, pi, obs, start, comp, ncomp, max_nodes=1 + K)
    _expect(paths, on=["SWEEP_2_0", "LEAF_BATCH", "SUM_BLOCKS", "SUM_LOOP"], off=["SUM_PREFIX", "SUM_ONE_CTA"])


@pytest.mark.parametrize("leaf", [1, 0])
def test_prefix_block_sum(leaf):
    """More than 262 144 bound terms (2048 blocks): the block prefixes come from their own kernel, for the leaf
    batch's three lists and for a single list."""
    rng = np.random.default_rng(8000 + leaf)
    K, M = 3, 5
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.0)
    obs, start, comp = _superseq_n(rng, 1_400_000, M, 2, 40)
    comp, ncomp = _clamp(rng, comp, 1, 0.2)
    assert np.count_nonzero(comp >= 0) >= 262144
    paths, _ = _check(A, B, pi, obs, start, comp, ncomp, leaf=leaf)
    _expect(paths, on=["SWEEP_1_2_16", "SUM_PREFIX"] + (["LEAF_BATCH"] if leaf else []),
            off=["SUM_BLOCKS", "SUM_ONE_CTA", "SUM_LOOP"] + ([] if leaf else ["LEAF_BATCH"]))


# ---- paths only the environment selects (read once at load: run in a fresh process) -----------------------------
def _env_case(name):
    rng = np.random.default_rng(8100)
    if name == "sum_one_cta":
        A, B, pi = random_hmm(rng, 12, 8, zero_frac=0.0)
        obs, start, comp, ncomp = random_superseq(rng, 40, 8, 2, 0.1, 2, 20)
        paths, _ = _check(A, B, pi, obs, start, comp, ncomp, max_nodes=40)
        _expect(paths, on=["LEAF_BATCH", "SUM_ONE_CTA"], off=["SUM_LOOP", "SUM_BLOCKS", "SUM_PREFIX"])
    elif name == "sum_loop":
        A, B, pi = random_hmm(rng, 5, 8, zero_frac=0.0)
        obs, start, comp = _superseq_n(rng, 24000, 8, 2, 30)
        comp, ncomp = _clamp(rng, comp, 2, 0.25)
        assert np.count_nonzero(comp >= 0) > 4096
        paths, _ = _check(A, B, pi, obs, start, comp, ncomp, max_nodes=12)
        _expect(paths, on=["LEAF_BATCH", "SUM_LOOP"], off=["SUM_BLOCKS", "SUM_PREFIX", "SUM_ONE_CTA"])
    elif name == "bound_copy":
        A, B, pi = random_hmm(rng, 12, 8, zero_frac=0.1)
        obs, start, comp, ncomp = random_superseq(rng, 40, 8, 3, 0.1, 2, 20)
        for leaf in (1, 0):
            paths, _ = _check(A, B, pi, obs, start, comp, ncomp, max_nodes=60, leaf=leaf)
            _expect(paths, on=["BOUND_COPY"])
    elif name in ("fullwarp_8", "fullwarp_16"):
        K = int(name.split("_")[1])
        for ties in (True, False):
            A, B, pi = random_hmm(rng, K, 8, zero_frac=0.15, ties=ties)
            obs, start, comp, ncomp = random_superseq(rng, 40, 8, 3, 0.12, 1, 14)
            for leaf in (1, 0):
                paths, _ = _check(A, B, pi, obs, start, comp, ncomp, max_nodes=60, leaf=leaf)
                fw, half = ("SWEEP_FW_1_2", "SWEEP_1_2_16") if K == 8 else ("SWEEP_FW_1_4", "SWEEP_1_4_16")
                _expect(paths, on=[fw], off=[half])
    else:
        raise ValueError(name)


@pytest.mark.parametrize("name,env", [
    ("sum_one_cta", {"CV_CP_SUM": "2"}),
    ("sum_loop", {"CV_CP_SUM": "0"}),
    ("bound_copy", {"CV_CP_HOSTPOLL": "0"}),
    ("fullwarp_8", {"CV_CP_FULLWARP": "1"}),
    ("fullwarp_16", {"CV_CP_FULLWARP": "1"}),
])
def test_environment_paths(name, env):
    flags = ["-I"] if sys.flags.isolated else (["-s"] if sys.flags.no_user_site else [])
    code = f"import sys; sys.path[:0] = {[ROOT, TESTS]!r}; import test_cp_paths_gpu as t; t._env_case({name!r})"
    r = subprocess.run([sys.executable, *flags, "-c", code], env={**os.environ, **env}, cwd=ROOT,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
