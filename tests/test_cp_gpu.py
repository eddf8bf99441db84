"""GPU parity tests (mode R2): cv_cp_solve through the C ABI against the C oracle -- solution, objective
bits, explored nodes, sweep steps, every node's upper bound and the full final delta/psi state."""
import numpy as np
import pytest

import consistent_viterbi_b200 as cv
from oracle import pyoracle as po
from util import cp_path_bits, random_hmm, random_superseq

pytestmark = pytest.mark.gpu


def _check(A, B, pi, obs, start, comp, ncomp, max_nodes=0):
    """Returns the solve's launch path bits (cv_debug_cp_last_paths), 0 when both sides raised."""
    h = cv.HMM(A, B, pi)
    try:
        ref = po.cp_solve(A, B, pi, obs, start, comp, ncomp, max_nodes=max_nodes, trace_nodes=1 << 16, want_state=True)
        ref_err = None
    except po.OracleError as e:
        ref_err = e.code
    try:
        got = cv.cp_solve_arrays(h, obs, start, comp, ncomp, max_nodes=max_nodes, want_state=True, want_ub=1 << 16)
        got_err = None
    except cv.CvError as e:
        got_err = e.code
    assert ref_err == got_err, (ref_err, got_err)
    if ref_err is not None:
        h.close()
        return 0
    assert got["explored"] == ref["explored"]
    assert got["steps"] == ref["steps"]
    n = min(len(got["ub"]), int(ref["explored"]))
    assert got["ub"][:n].tobytes() == ref["ub"][:n].tobytes(), "per-node upper bounds differ"
    assert np.float64(got["obj"]).tobytes() == np.float64(ref["obj"]).tobytes()
    assert (got["sol"] == ref["sol"]).all()
    assert got["delta"].tobytes() == ref["delta"].tobytes(), "final delta state differs"
    assert (got["psi"] == ref["psi"]).all(), "final psi state differs"
    paths = cv._lib.lib().cv_debug_cp_last_paths(h.device_handle())
    h.close()
    return paths


@pytest.mark.parametrize("seed", range(8))
def test_cp_random_small(seed):
    rng = np.random.default_rng(500 + seed)
    for it in range(12):
        K = int(rng.integers(1, 7)); M = int(rng.integers(1, 6))
        A, B, pi = random_hmm(rng, K, M, ties=(it % 3 == 0), zero_frac=0.15)
        obs, start, comp, ncomp = random_superseq(rng, int(rng.integers(1, 7)), M, int(rng.integers(0, 4)), 0.3, 1, 12)
        _check(A, B, pi, obs, start, comp, ncomp)


@pytest.mark.parametrize("K", [8, 9, 12, 16, 24, 25, 28, 32, 34, 45, 57, 63, 64])
def test_cp_mid_k(K):
    """Every warp-per-segment sweep shape: its path bit (include/cv_b200_debug.h) must be the one K selects."""
    rng = np.random.default_rng(600 + K)
    M = 12
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.1)
    obs, start, comp, ncomp = random_superseq(rng, 30, M, 3, 0.08, 5, 60)
    paths = _check(A, B, pi, obs, start, comp, ncomp, max_nodes=60)
    P = cp_path_bits()
    want = ["SWEEP_1_2_16", "SWEEP_1_4_16", "SWEEP_1_6", "SWEEP_1_8"][(K + 7) // 8 - 1] if K <= 32 else "SWEEP_2_0"
    sweeps = P["SWEEP_1_2_16"] | P["SWEEP_1_4_16"] | P["SWEEP_1_6"] | P["SWEEP_1_8"] | P["SWEEP_2_0"]
    assert paths & sweeps == P[want], hex(paths)


@pytest.mark.parametrize("K", [65, 100, 130, 300])
def test_cp_large_k_generic_path(K):
    """K > 64: generic sweep kernel (states looped per lane, logA from L2), u16 backpointers."""
    rng = np.random.default_rng(650 + K)
    M = 9
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.1)
    obs, start, comp, ncomp = random_superseq(rng, 8, M, 2, 0.1, 3, 25)
    _check(A, B, pi, obs, start, comp, ncomp, max_nodes=12)


def test_cp_no_constraints_and_prefix():
    rng = np.random.default_rng(77)
    A, B, pi = random_hmm(rng, 5, 4, zero_frac=0.0)
    obs, start, comp, ncomp = random_superseq(rng, 6, 4, 0, 0.0, 2, 30)
    _check(A, B, pi, obs, start, comp, 0)
    # constraints only at the very end: long init_viterbi prefix
    obs, start, comp, _ = random_superseq(rng, 5, 4, 0, 0.0, 10, 40)
    comp[-1] = 0
    _check(A, B, pi, obs, start, comp, 1)
    # first element clamped: empty prefix, t == 0 bound term
    comp2 = np.full(len(obs), -1, dtype=np.int32); comp2[0] = 0; comp2[3] = 0; comp2[4] = 1
    _check(A, B, pi, obs, start, comp2, 2)


def test_cp_trucks_like():
    """BASELINE configs[0] stand-in (real datasets/trucks absent): D=2 bdims [16,8], K=12, control tags on ~10 %
    of the positions over 4 tag values, prop = 1; node budget so the oracle finishes quickly."""
    rng = np.random.default_rng(3019)
    K, M = 12, 128
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.2, alpha=0.5)
    obs, start, comp, ncomp = random_superseq(rng, 40, M, 4, 0.10, 50, 200)
    _check(A, B, pi, obs, start, comp, ncomp, max_nodes=150)


def test_cp_solver_interface_and_superseq(tmp_path):
    """Solver trait mirror + SuperSequence assembly (from_tags, reorder, parse_solution) on a tiny corpus."""
    rng = np.random.default_rng(12)
    K, bd = 4, (3, 2)
    A, B, pi = random_hmm(rng, K, 6, zero_frac=0.1)
    hmm = cv.HMM(A, B.reshape(K, *bd), pi)
    seqs = [[[int(rng.integers(0, 3)), int(rng.integers(0, 2))] for _ in range(int(rng.integers(2, 9)))] for _ in range(7)]
    tags = [[(int(rng.integers(0, 2)) if rng.random() < 0.3 else None) for _ in s] for s in seqs]
    # file round trip (src/utils.rs formats)
    with open(tmp_path / "sequences", "w") as f:
        for i, s in enumerate(seqs):
            for v in s:
                f.write(f"{i} {v[0]} {v[1]}\n")
    with open(tmp_path / "test_tags", "w") as f:
        for i, tg in enumerate(tags):
            for t in tg:
                f.write(f"{i} {-1 if t is None else t}\n")
    assert cv.load_sequences(tmp_path / "sequences") == seqs
    assert cv.load_tags(tmp_path / "test_tags") == tags
    cons = cv.Constraints.from_tags(tags)
    ss = cv.SuperSequence(seqs, cons, hmm)
    ss.recompute_constraints(1.0)
    solver = cv.CPSolver(hmm, ss)
    assert solver.get_name() == "cp"
    solver.solve()
    obs, start, comp, ncomp = ss.solver_inputs()
    ref = po.cp_solve(A, B, pi, obs, start, comp, ncomp)
    assert (solver.get_solution() == ref["sol"]).all()
    assert np.float64(solver.get_objective()).tobytes() == np.float64(ref["obj"]).tobytes()
    assert solver.get_explored_nodes() == ref["explored"]
    per_seq = ss.parse_solution(solver.get_solution())
    assert [len(x) for x in per_seq] == [len(s) for s in seqs]
    # all members of an active component share one state in the solution
    sol = solver.get_solution()
    if ref["obj"] > -np.inf:
        for c in range(ncomp):
            assert len(set(int(x) for x in sol[comp == c])) == 1


def test_cp_dense_deep_search():
    """Dense model (no zero probabilities): bounds stay finite, so the search goes several components deep and
    prunes by value; 400 nodes of it against the oracle, with every bound and the final state."""
    import bench
    w = bench.workload_cp("trucks")
    _check(w["A"], w["B"], w["pi"], w["obs"], w["start"], w["comp"], w["ncomp"], max_nodes=400)


@pytest.mark.parametrize("seed", range(6))
def test_cp_leaf_batch_equals_node_by_node(seed):
    """The K sibling leaves of the last component evaluated as one batch (cp_leaf_group) against the node-by-node
    loop and the oracle: complete delta / psi state, every bound, counters -- with node budgets that stop inside a
    leaf group, adjacent clamped positions, ties and -inf entries, 1 to 4 components."""
    rng = np.random.default_rng(9100 + seed)
    L = cv._lib.lib()
    try:
        for it in range(10):
            K = int(rng.integers(2, 10)); M = int(rng.integers(2, 7))
            A, B, pi = random_hmm(rng, K, M, ties=(it % 4 == 0), zero_frac=0.15)
            obs, start, comp, ncomp = random_superseq(rng, int(rng.integers(2, 10)), M, int(rng.integers(1, 5)),
                                                      float(rng.choice([0.1, 0.3, 0.6])), 1, 14)
            budget = int(rng.choice([0, 0, 7, 23, 61]))
            for on in (1, 0):
                L.cv_debug_set_cp_leaf_batch(on)
                _check(A, B, pi, obs, start, comp, ncomp, max_nodes=budget)
    finally:
        L.cv_debug_set_cp_leaf_batch(1)


def test_cp_leaf_batch_mid_size():
    rng = np.random.default_rng(77)
    L = cv._lib.lib()
    try:
        for K in (12, 16, 33):
            A, B, pi = random_hmm(rng, K, 20, zero_frac=0.05)
            obs, start, comp, ncomp = random_superseq(rng, 40, 20, 3, 0.15, 20, 120)
            for on in (1, 0):
                L.cv_debug_set_cp_leaf_batch(on)
                _check(A, B, pi, obs, start, comp, ncomp, max_nodes=150)
    finally:
        L.cv_debug_set_cp_leaf_batch(1)
