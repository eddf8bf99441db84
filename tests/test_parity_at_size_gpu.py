"""GPU parity at BASELINE.json's own sizes (VERDICT r01 "weak #1"): the complete configs[2] batch, a configs[3]
slice at the full T = 4096, configs[4] at N = 640 k and the complete trucks-like search -- all through the C ABI,
all compared with the C oracle (the literal restatement of viterbi.rs:5-32 / cp.rs:20-152) bit for bit.

Plus the two launch-shape hazards ADVICE r01 found: delta-history sizing when tiles straddle chunks of the streamed
host path, and the warp-per-sequence kernel on a multi-chunk call."""
import os

import numpy as np
import pytest

import consistent_viterbi_b200 as cv
from oracle import pyoracle as po
from test_cp_paths_gpu import _check, _expect, _superseq_n
from util import random_hmm

pytestmark = pytest.mark.gpu

NT = os.cpu_count() or 1


def test_pos_full_batch_equals_oracle():
    """configs[2], all 1 000 000 sentences (5.1e10 cells): every path element and every score bit against the
    oracle (viterbi.rs:5-32), through the host-buffer entry point (streamed copies) AND the device-resident one."""
    import torch

    import bench
    wl = bench.workload_pos(0, 1_000_000)
    rp, rs = po.decode_batch(wl["A"], wl["B"], wl["obs"], wl["off"], nthreads=NT)
    h = cv.HMM(wl["A"], wl["B"], wl["pi"])
    p, s = cv.decode_batch(h, wl["obs"], wl["off"])                     # cv_decode_batch
    assert int((p != rp).sum()) == 0
    assert s.tobytes() == rs.tobytes()
    # cv_decode_batch_dev on torch's stream: the bench's `value` leg
    L = cv._lib.lib()
    hd = h.device_handle(torch.cuda.current_device())
    N, B = len(wl["obs"]), len(wl["off"]) - 1
    d_obs = torch.from_numpy(wl["obs"].view(np.int32)).cuda()
    d_off = torch.from_numpy(wl["off"]).cuda()
    d_path = torch.empty(N, dtype=torch.int32, device="cuda")
    d_score = torch.empty(B, dtype=torch.float64, device="cuda")
    cv._lib.check(L.cv_decode_batch_dev(hd, d_obs.data_ptr(), d_off.data_ptr(), B, N, int(np.diff(wl["off"]).max()),
                                        d_path.data_ptr(), d_score.data_ptr(), torch.cuda.current_stream().cuda_stream, 1))
    torch.cuda.synchronize()
    assert int((d_path.cpu().numpy().view(np.uint32) != rp).sum()) == 0
    assert d_score.cpu().numpy().tobytes() == rs.tobytes()
    h.close()


def test_large_state_T4096_slice_equals_oracle():
    """configs[3] at its full length: K = 1024, M = 4096, T = 4096 (the 4096-step history indexing, size_t slab
    arithmetic).  B = 128 sequences on the GPU, once as one group of row blocks and once forced into groups of one
    row block (the path the full 137 GB history takes); 16 of them against the oracle (7e10 cells)."""
    import bench
    wl = bench.workload_large(0, 128, 4096)
    h = cv.HMM(wl["A"], wl["B"], wl["pi"])
    L = cv._lib.lib()
    p1, s1 = cv.decode_batch(h, wl["obs"], wl["off"])
    try:
        L.cv_debug_set_large_group_rb(1)
        p2, s2 = cv.decode_batch(h, wl["obs"], wl["off"])
    finally:
        L.cv_debug_set_large_group_rb(0)
    assert (p1 == p2).all() and s1.tobytes() == s2.tobytes()
    off = wl["off"]
    sel = list(range(0, 128, 8))[:16]
    sub_obs = np.concatenate([wl["obs"][off[b]:off[b + 1]] for b in sel])
    sub_off = np.arange(len(sel) + 1, dtype=np.int64) * 4096
    rp, rs = po.decode_batch(wl["A"], wl["B"], sub_obs, sub_off, nthreads=NT)
    assert (np.concatenate([p1[off[b]:off[b + 1]] for b in sel]) == rp).all()
    assert s1[sel].tobytes() == rs.tobytes()
    h.close()


def _cp_check(w, max_nodes, want_state):
    h = cv.HMM(w["A"], w["B"], w["pi"])
    args = (w["obs"], w["start"], w["comp"], w["ncomp"])
    ref = po.cp_solve(w["A"], w["B"], w["pi"], *args, max_nodes=max_nodes, trace_nodes=1 << 16, want_state=want_state)
    got = cv.cp_solve_arrays(h, *args, max_nodes=max_nodes, want_state=want_state, want_ub=1 << 16)
    assert got["explored"] == ref["explored"] and got["steps"] == ref["steps"]
    n = min(len(got["ub"]), int(ref["explored"]))
    assert n > 0 and got["ub"][:n].tobytes() == ref["ub"][:n].tobytes(), "per-node upper bounds differ"
    assert np.float64(got["obj"]).tobytes() == np.float64(ref["obj"]).tobytes()
    assert (got["sol"] == ref["sol"]).all()
    if want_state:
        assert got["delta"].tobytes() == ref["delta"].tobytes(), "final delta state differs"
        assert (got["psi"] == ref["psi"]).all(), "final psi state differs"
    h.close()
    return ref


def test_cp_heavy_640k_equals_oracle():
    """configs[4] (K = 16, 64 sequences x T = 10 000, N = 640 000, ~20 % clamped) with a 40-node budget: the bound of
    every node, the final delta / psi state of all 640 000 rows, solution, objective, node and step counts
    (cp.rs:95-126).  The budget reaches the last component, so the batched leaf level is covered."""
    import bench
    w = bench.workload_cp("heavy")
    assert w["N"] == 640000
    ref = _cp_check(w, max_nodes=40, want_state=True)
    assert ref["explored"] == 40


def test_cp_trucks_complete_search_equals_oracle():
    """configs[0] stand-in (trucks-like, K = 12, N = 46 k): the COMPLETE branch and bound -- every node's bound,
    objective bits, solution, explored nodes and sweep steps."""
    import bench
    w = bench.workload_cp("trucks")
    ref = _cp_check(w, max_nodes=0, want_state=True)
    assert ref["explored"] > 5000


def test_streamed_history_with_tiles_straddling_chunks():
    """ADVICE r01 (high): tiles are ordered by (chunk, length) and may straddle chunks; a batch of length-1 sequences
    with a few very long ones placed at the chunk boundaries needs up to 2*nch-1 staircase terms of history."""
    rng = np.random.default_rng(77)
    K, M = 45, 50
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.1)
    Bn, nch = 480252, 4
    lens = np.ones(Bn, dtype=np.int64)
    for c in range(nch):                                  # long sequences at the start and the end of every chunk
        b0, b1 = Bn * c // nch, Bn * (c + 1) // nch
        lens[[b0, b0 + 1, b1 - 1]] = rng.integers(1500, 2001, size=3)
    lens[rng.integers(0, Bn, size=40)] = rng.integers(2, 60, size=40)
    off = np.zeros(Bn + 1, dtype=np.int64)
    off[1:] = np.cumsum(lens)
    obs = rng.integers(0, M, size=int(off[-1])).astype(np.uint32)
    h = cv.HMM(A, B, pi)
    L = cv._lib.lib()
    try:
        L.cv_debug_set_chunks(nch)
        p, s = cv.decode_batch(h, obs, off)
    finally:
        L.cv_debug_set_chunks(-1)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=NT)
    assert (p == rp).all() and s.tobytes() == rs.tobytes()
    h.close()


@pytest.mark.parametrize("K", [7, 24, 45])
def test_chain_kernel_on_a_multi_chunk_call(K):
    """ADVICE r01 (medium): three chunks with the default warp-per-sequence threshold -- chunks 1 and 2 index the
    chunk-local backpointer buffer with absolute offsets unless the kernel subtracts the chunk's first offset."""
    rng = np.random.default_rng(900 + K)
    M = 30
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.15)
    lens = rng.integers(1, 300, size=900)
    off = np.zeros(len(lens) + 1, dtype=np.int64)
    off[1:] = np.cumsum(lens)
    obs = rng.integers(0, M, size=int(off[-1])).astype(np.uint32)
    h = cv.HMM(A, B, pi)
    L = cv._lib.lib()
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=NT)
    try:
        for streamed in (1, 0):
            L.cv_debug_set_chunks(3)
            L.cv_debug_set_pipeline(-1, streamed)
            p, s = cv.decode_batch(h, obs, off)
            assert (p == rp).all() and s.tobytes() == rs.tobytes()
    finally:
        L.cv_debug_set_chunks(-1)
        L.cv_debug_set_pipeline(1, 1)
    h.close()


@pytest.mark.parametrize("N", [402945, 402946])
def test_backtrack_chain_smem_edge(N):
    """K = 64: the chunk maps of N - 1 = 402 944 rows (1574 chunks) fit the entry chain's shared memory, one row more
    (1575 chunks) and one thread walks them in global memory.  The only component sits in the last rows, so the
    oracle's cost is the unconstrained prefix, N K^2 = 1.7e9 cell updates, once (about a minute per case)."""
    rng = np.random.default_rng(7700 + N)
    K, M = 64, 20
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.0)
    obs, start, comp = _superseq_n(rng, N, M, 5, 40)
    comp[[N - 180, N - 120, N - 61, N - 1]] = 0
    paths, got = _check(A, B, pi, obs, start, comp, 1, state=False)
    assert got["obj"] > -np.inf
    _expect(paths, on=["SWEEP_2_0", "LEAF_BATCH"] + (["BTR_CHAIN_GMEM"] if N > 402945 else []),
            off=["BTR_ROWS_GMEM"] + ([] if N > 402945 else ["BTR_CHAIN_GMEM"]))
