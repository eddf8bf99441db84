"""GPU parity tests (mode R1): cv_decode_batch through the C ABI against the C
oracle, bit-exact on paths (u32) and scores (f64 bit patterns)."""
import numpy as np
import pytest

import consistent_viterbi_b200 as cv
from oracle import pyoracle as po
from util import random_batch, random_hmm

pytestmark = pytest.mark.gpu


def _check(A, B, pi, obs, off):
    """Both K <= 64 kernels are exercised: the warp-per-sequence kernel (default for small batches) and the
    lock-step tile kernel (forced with cv_debug_set_chain_max_batch(0))."""
    h = cv.HMM(A, B, pi)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    L = cv._lib.lib()
    try:
        for chain_max in (-1, 0):
            L.cv_debug_set_chain_max_batch(chain_max)
            paths, scores = cv.decode_batch(h, obs, off)
            bad = np.nonzero(paths != rp)[0]
            assert bad.size == 0, f"chain_max={chain_max}: {bad.size} path mismatches, first at {bad[:5]}"
            assert scores.tobytes() == rs.tobytes(), f"chain_max={chain_max}: scores differ"
    finally:
        L.cv_debug_set_chain_max_batch(-1)
    h.close()


@pytest.mark.parametrize("K", [1, 2, 3, 7, 8, 9, 12, 16, 18, 24, 31, 33, 45, 48, 57, 64])
def test_small_k_random(K):
    rng = np.random.default_rng(1000 + K)
    M = int(rng.integers(1, 40))
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.2)
    obs, off = random_batch(rng, 700, M, 1, 40)
    _check(A, B, pi, obs, off)


@pytest.mark.parametrize("K,Bn,tmax", [(65, 300, 20), (100, 130, 30), (128, 64, 40), (129, 200, 12), (200, 70, 25),
                                       (256, 65, 10), (257, 40, 10), (300, 100, 8)])
def test_large_k_random(K, Bn, tmax):
    """K > 64: tiled logA kernel (work items (t, row block, column block), TMA ring)."""
    rng = np.random.default_rng(3000 + K)
    M = int(rng.integers(2, 30))
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.3)
    obs, off = random_batch(rng, Bn, M, 1, tmax)
    _check(A, B, pi, obs, off)


def test_large_k_batch_groups():
    """The delta history of a large-K batch is processed in groups of row blocks when it does not fit in HBM;
    force groups of one and two row blocks.  B = 300 is five row blocks of 64: 5, 3 and 1 groups, and every group
    launches three kernels (items per step, forward, backtrace)."""
    rng = np.random.default_rng(3200)
    A, B, pi = random_hmm(rng, 140, 9, zero_frac=0.3)
    obs, off = random_batch(rng, 300, 9, 1, 14)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    h = cv.HMM(A, B, pi)
    L = cv._lib.lib()
    launches = {}
    L.cv_debug_set_chunks(1)
    try:
        cv.decode_batch(h, obs, off)                              # the model's device set-up launches kernels too
        for rb in (0, 1, 2):
            L.cv_debug_set_large_group_rb(rb)
            n0 = L.cv_launch_count()
            paths, scores = cv.decode_batch(h, obs, off)
            launches[rb] = L.cv_launch_count() - n0
            assert (paths == rp).all(), f"rb={rb}: path mismatches"
            assert scores.tobytes() == rs.tobytes(), f"rb={rb}: scores differ"
    finally:
        L.cv_debug_set_large_group_rb(0)
        L.cv_debug_set_chunks(-1)
        h.close()
    assert launches[1] - launches[0] == 3 * (5 - 1), launches
    assert launches[2] - launches[0] == 3 * (3 - 1), launches


def test_large_k_ties():
    rng = np.random.default_rng(3100)
    A, B, pi = random_hmm(rng, 150, 5, ties=True)
    obs, off = random_batch(rng, 150, 5, 1, 15)
    _check(A, B, pi, obs, off)


@pytest.mark.parametrize("K", [2, 5, 8, 13, 45])
def test_small_k_ties_and_neg_inf(K):
    """log-probs from a tiny dyadic set incl. -inf and +-0.0: exact ties everywhere, so the
    lowest-index rule (ndarray-stats argmax) decides almost every backpointer."""
    rng = np.random.default_rng(2000 + K)
    M = 6
    A, B, pi = random_hmm(rng, K, M, ties=True)
    obs, off = random_batch(rng, 500, M, 1, 25)
    _check(A, B, pi, obs, off)


def test_edge_lengths_and_single_sequence():
    rng = np.random.default_rng(5)
    A, B, pi = random_hmm(rng, 45, 30)
    for lens in ([1], [2], [1, 1, 1], [300], [1, 500, 2, 1, 77]):
        off = np.zeros(len(lens) + 1, dtype=np.int64); off[1:] = np.cumsum(lens)
        obs = rng.integers(0, 30, size=int(off[-1])).astype(np.uint32)
        _check(A, B, pi, obs, off)
    path = cv.decode([[3], [1], [2], [29]], cv.HMM(A, B, pi))
    ref, _ = po.decode(A, B, np.array([3, 1, 2, 29], dtype=np.uint32))
    assert path.dtype == np.uint64 and (path == ref).all()


def test_all_neg_inf_emissions():
    rng = np.random.default_rng(6)
    A, B, pi = random_hmm(rng, 9, 4)
    B[:] = -np.inf
    obs, off = random_batch(rng, 70, 4, 1, 12)
    _check(A, B, pi, obs, off)


def test_errors_match_reference_panics():
    rng = np.random.default_rng(8)
    A, B, pi = random_hmm(rng, 6, 4)
    h = cv.HMM(A, B, pi)
    with pytest.raises(cv.CvError) as e:                      # empty sequence: usize underflow panic
        cv.decode_batch(h, np.array([0, 1], dtype=np.uint32), np.array([0, 2, 2], dtype=np.int64))
    assert e.value.code == cv._lib.ERR_EMPTY
    with pytest.raises(cv.CvError) as e:                      # obs >= M: ndarray index panic
        cv.decode_batch(h, np.array([0, 9, 1], dtype=np.uint32), np.array([0, 3], dtype=np.int64))
    assert e.value.code == cv._lib.ERR_ARG
    An = A.copy(); An[0, 0] = np.nan
    with pytest.raises(cv.CvError) as e:
        cv.HMM(An, B, pi).device_handle()
    assert e.value.code == cv._lib.ERR_NAN


def test_pos_shape_sample_and_properties():
    """POS shape (K=45, V=20k), 20k sentences: oracle parity on the full sample plus
    size-independent properties: batch == concatenation of singles; permuting the batch
    permutes the output."""
    rng = np.random.default_rng(3019)
    K, M, Bn = 45, 20000, 20000
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.05, alpha=0.1)
    lens = np.clip(np.rint(rng.gamma(2.5, 10.0, size=Bn)), 1, 200).astype(np.int64)
    off = np.zeros(Bn + 1, dtype=np.int64); off[1:] = np.cumsum(lens)
    obs = (rng.zipf(1.1, size=int(off[-1])) % M).astype(np.uint32)
    h = cv.HMM(A, B, pi)
    paths, scores = cv.decode_batch(h, obs, off)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    assert (paths == rp).all() and scores.tobytes() == rs.tobytes()
    perm = rng.permutation(Bn)
    off2 = np.zeros(Bn + 1, dtype=np.int64); off2[1:] = np.cumsum(lens[perm])
    obs2 = np.concatenate([obs[off[b]:off[b + 1]] for b in perm])
    p2, s2 = cv.decode_batch(h, obs2, off2)
    assert s2.tobytes() == scores[perm].tobytes()
    for k in (0, 1, Bn // 2, Bn - 1):
        b = perm[k]
        assert (p2[off2[k]:off2[k + 1]] == paths[off[b]:off[b + 1]]).all()


@pytest.mark.parametrize("K", [9, 20, 33, 45, 47, 64])
def test_tile_kernel_variants_equal_oracle(K):
    """Every launch-time variant of the tile path against the oracle on one ragged batch with -inf entries, many
    length-1 sequences and two chunked host modes: compile-time row pitches on / off (cv_debug_set_fwd_ldc), emission-row
    fetch dealt out by tile work / evenly (cv_debug_set_em_light), backtrace with four lanes per sequence / one thread per
    sequence (cv_debug_set_bt_split; 2 = at every size)."""
    rng = np.random.default_rng(7700 + K)
    M = 35
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.2, ties=(K % 2 == 0))      # even K: dyadic values, exact ties, +-0.0
    obs, off = random_batch(rng, 7000, M, 1, 45)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    h = cv.HMM(A, B, pi)
    L = cv._lib.lib()
    try:
        L.cv_debug_set_chain_max_batch(0)
        for ldc in (1, 0):
            for light in (1, 0):
                for split in (2, 0):
                    for chunks in (1, 3):
                        L.cv_debug_set_fwd_ldc(ldc); L.cv_debug_set_em_light(light); L.cv_debug_set_bt_split(split)
                        L.cv_debug_set_chunks(chunks)
                        p, s = cv.decode_batch(h, obs, off)
                        assert (p == rp).all() and s.tobytes() == rs.tobytes(), (ldc, light, split, chunks)
        # backtrace after the forward kernel (timing mode of the device API runs the kernels one after the other)
        L.cv_debug_set_pipeline(0, 0)
        for split in (2, 0):
            L.cv_debug_set_bt_split(split)
            p, s = cv.decode_batch(h, obs, off)
            assert (p == rp).all() and s.tobytes() == rs.tobytes(), ("sequential", split)
    finally:
        L.cv_debug_set_fwd_ldc(1); L.cv_debug_set_em_light(1); L.cv_debug_set_bt_split(1)
        L.cv_debug_set_pipeline(1, 1)
        L.cv_debug_set_chunks(-1)
        L.cv_debug_set_chain_max_batch(-1)
    h.close()


def test_split_backtrace_all_neg_inf_and_single_steps():
    """The four-lane backtrace on the cases its end-state / -inf rules exist for: every emission -inf (all paths are
    state 0 from the first -inf on), length-1 and length-2 sequences, K below / at the lane split (K = 3, 4, 5)."""
    L = cv._lib.lib()
    try:
        L.cv_debug_set_chain_max_batch(0)
        L.cv_debug_set_bt_split(2)
        for K in (3, 4, 5, 17):
            rng = np.random.default_rng(880 + K)
            M = 6
            A, B, pi = random_hmm(rng, K, M, zero_frac=0.5)
            B[:, 0] = -np.inf                                    # observation 0 is impossible in every state
            lens = rng.integers(1, 4, size=3000)
            off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
            obs = rng.integers(0, M, size=int(off[-1])).astype(np.uint32)
            rp, rs = po.decode_batch(A, B, obs, off, nthreads=4)
            h = cv.HMM(A, B, pi)
            p, s = cv.decode_batch(h, obs, off)
            assert (p == rp).all() and s.tobytes() == rs.tobytes(), K
            h.close()
    finally:
        L.cv_debug_set_bt_split(1)
        L.cv_debug_set_chain_max_batch(-1)


def test_chunked_pipeline_and_device_api():
    """cv_decode_batch cuts large batches into chunks on two internal streams and cv_decode_batch_dev takes
    device-resident buffers (torch tensors here, plain pointers at the ABI): force 3 chunks on a mid-size batch
    and compare both entry points with the oracle."""
    import torch
    rng = np.random.default_rng(4242)
    K, M, Bn = 45, 60, 5000
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.1)
    obs, off = random_batch(rng, Bn, M, 1, 40)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    h = cv.HMM(A, B, pi)
    L = cv._lib.lib()
    try:
        L.cv_debug_set_chain_max_batch(0)
        for chunks in (1, 3, 8):
            L.cv_debug_set_chunks(chunks)
            p, s = cv.decode_batch(h, obs, off)
            assert (p == rp).all() and s.tobytes() == rs.tobytes(), f"host API, chunks={chunks}"
            d_obs = torch.from_numpy(obs.view(np.int32)).cuda()
            d_off = torch.from_numpy(off).cuda()
            d_path = torch.zeros(len(obs), dtype=torch.int32, device="cuda")
            d_score = torch.zeros(Bn, dtype=torch.float64, device="cuda")
            st = torch.cuda.current_stream()
            rc = L.cv_decode_batch_dev(h.device_handle(), d_obs.data_ptr(), d_off.data_ptr(), Bn, len(obs),
                                       int(np.diff(off).max()), d_path.data_ptr(), d_score.data_ptr(), st.cuda_stream, 1)
            cv._lib.check(rc)
            torch.cuda.synchronize()
            assert (d_path.cpu().numpy().view(np.uint32) == rp).all(), f"device API, chunks={chunks}"
            assert d_score.cpu().numpy().tobytes() == rs.tobytes()
    finally:
        L.cv_debug_set_chunks(-1)
        L.cv_debug_set_chain_max_batch(-1)
    h.close()


def test_pipeline_modes_agree():
    """The host path in all its forms -- streamed copies past one launch / one launch per chunk, backtrace next to
    or after the forward kernel -- on a ragged batch with many length-1 sequences and up to 16 chunks."""
    rng = np.random.default_rng(99)
    K, M, Bn = 37, 50, 30000
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.1)
    obs, off = random_batch(rng, Bn, M, 1, 30)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    h = cv.HMM(A, B, pi)
    L = cv._lib.lib()
    try:
        L.cv_debug_set_chain_max_batch(0)
        for conc, streamed in ((1, 1), (1, 0), (0, 0)):
            L.cv_debug_set_pipeline(conc, streamed)
            for chunks in (2, 5, 16):
                L.cv_debug_set_chunks(chunks)
                for _ in range(2):                                # second call reuses flags / counters / buffers
                    p, s = cv.decode_batch(h, obs, off)
                    assert (p == rp).all() and s.tobytes() == rs.tobytes(), (conc, streamed, chunks)
        L.cv_debug_set_pipeline(1, 1)
        L.cv_debug_set_chunks(4)
        bad = off.copy(); bad[1000] = bad[1001]                   # an empty sequence in the third chunk's range... any chunk
        with pytest.raises(cv.CvError) as e:
            cv.decode_batch(h, obs, bad)
        assert e.value.code == cv._lib.ERR_EMPTY
        o2 = obs.copy(); o2[len(o2) // 2] = M                      # observation out of range (index panic)
        with pytest.raises(cv.CvError) as e:
            cv.decode_batch(h, o2, off)
        assert e.value.code == cv._lib.ERR_ARG
        p, s = cv.decode_batch(h, obs, off)                       # and the handle still works afterwards
        assert (p == rp).all() and s.tobytes() == rs.tobytes()
    finally:
        L.cv_debug_set_pipeline(1, 1)
        L.cv_debug_set_chunks(-1)
        L.cv_debug_set_chain_max_batch(-1)
    h.close()


def _path_score(A, B, obs, path):
    """Score of a decoded path under viterbi.rs's association ((d + a) + b), d0 = 0.0 -- plain Python floats."""
    d = 0.0
    for t in range(1, len(obs)):
        d = (d + float(A[path[t - 1], path[t]])) + float(B[path[t], obs[t]])
    return d


def test_full_size_pos_properties():
    """BASELINE configs[2] at full size (1M sentences, ~5e10 cells): too big for the oracle in a test, so check
    size-independent properties: (1) the run is deterministic, (2) every sampled path re-scores, add by add in the
    reference's order, to exactly the returned score (so the path is a valid witness of the value), (3) a sampled
    sub-batch decoded alone gives the same paths/scores, and that sub-batch equals the oracle."""
    import bench
    wl = bench.workload_pos(0, 1_000_000)
    h = cv.HMM(wl["A"], wl["B"], wl["pi"])
    p1, s1 = cv.decode_batch(h, wl["obs"], wl["off"])
    p2, s2 = cv.decode_batch(h, wl["obs"], wl["off"])
    assert (p1 == p2).all() and s1.tobytes() == s2.tobytes()
    rng = np.random.default_rng(1)
    off = wl["off"]
    pick = np.sort(rng.choice(len(off) - 1, size=3000, replace=False))
    for b in pick[:400]:
        o = wl["obs"][off[b]:off[b + 1]]
        sc = _path_score(wl["A"], wl["B"], o, p1[off[b]:off[b + 1]])
        assert np.float64(sc).tobytes() == np.float64(s1[b]).tobytes() or (sc == -np.inf and s1[b] == -np.inf)
    sub_obs = np.concatenate([wl["obs"][off[b]:off[b + 1]] for b in pick])
    sub_off = np.concatenate([[0], np.cumsum([off[b + 1] - off[b] for b in pick])]).astype(np.int64)
    ps, ss = cv.decode_batch(h, sub_obs, sub_off)
    assert ss.tobytes() == s1[pick].tobytes()
    assert (ps == np.concatenate([p1[off[b]:off[b + 1]] for b in pick])).all()
    rp, rs = po.decode_batch(wl["A"], wl["B"], sub_obs, sub_off, nthreads=8)
    assert (ps == rp).all() and ss.tobytes() == rs.tobytes()
    h.close()


def test_large_state_properties():
    """BASELINE configs[3] shape (K=1024, M=4096) at reduced batch/length: determinism, exact re-scoring of
    sampled paths, and oracle parity on a few sequences."""
    import bench
    wl = bench.workload_large(0, 256, 96)
    h = cv.HMM(wl["A"], wl["B"], wl["pi"])
    p1, s1 = cv.decode_batch(h, wl["obs"], wl["off"])
    p2, s2 = cv.decode_batch(h, wl["obs"], wl["off"])
    assert (p1 == p2).all() and s1.tobytes() == s2.tobytes()
    off = wl["off"]
    for b in (0, 17, 128, 255):
        o = wl["obs"][off[b]:off[b + 1]]
        sc = _path_score(wl["A"], wl["B"], o, p1[off[b]:off[b + 1]])
        assert np.float64(sc).tobytes() == np.float64(s1[b]).tobytes()
    sel = [3, 200]
    sub_obs = np.concatenate([wl["obs"][off[b]:off[b + 1]] for b in sel])
    sub_off = np.array([0, 96, 192], dtype=np.int64)
    rp, rs = po.decode_batch(wl["A"], wl["B"], sub_obs, sub_off, nthreads=2)
    assert (np.concatenate([p1[off[b]:off[b + 1]] for b in sel]) == rp).all() and s1[sel].tobytes() == rs.tobytes()
    h.close()


def test_large_k_dataflow_stress():
    """The large-K kernel synchronises work items of consecutive steps across CTAs with release/acquire counters and
    reads the published rows through TMA.  Many row blocks x column blocks x steps, several runs: every run must be
    identical, equal the oracle on the whole batch, and every path must re-score exactly."""
    rng = np.random.default_rng(5150)
    K, M, Bn, T = 260, 11, 1500, 48          # 24 row blocks x 3 column blocks x 47 steps = 3384 work items
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.25)
    off = np.arange(Bn + 1, dtype=np.int64) * T
    obs = rng.integers(0, M, size=Bn * T).astype(np.uint32)
    h = cv.HMM(A, B, pi)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=16)
    for run in range(4):
        p, s = cv.decode_batch(h, obs, off)
        assert (p == rp).all(), f"run {run}: paths differ from the oracle"
        assert s.tobytes() == rs.tobytes(), f"run {run}: scores differ"
    for b in range(0, Bn, 97):
        sc = _path_score(A, B, obs[off[b]:off[b + 1]], p[off[b]:off[b + 1]])
        assert np.float64(sc).tobytes() == np.float64(s[b]).tobytes() or (sc == -np.inf and s[b] == -np.inf)
    h.close()


@pytest.mark.parametrize("K", [13, 37, 45, 47, 61])
def test_forward_kernel_state_splits_equal_oracle(K):
    """The forward tile kernel with the balanced state split (default: groups of near-equal size over slot-permuted
    copies of logA / logB^T, e.g. 8,8,8,7,7,7 for K = 45) and with plain groups of 8 (last one padded), against the
    oracle; ragged lengths, -inf entries."""
    rng = np.random.default_rng(4400 + K)
    M = 40
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.15)
    obs, off = random_batch(rng, 9000, M, 1, 40)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    h = cv.HMM(A, B, pi)
    L = cv._lib.lib()
    try:
        L.cv_debug_set_chain_max_batch(0)
        for on in (1, 0):
            L.cv_debug_set_balanced_split(on)
            p, s = cv.decode_batch(h, obs, off)
            assert (p == rp).all() and s.tobytes() == rs.tobytes(), f"balanced_split={on}"
    finally:
        L.cv_debug_set_balanced_split(1)
        L.cv_debug_set_chain_max_batch(-1)
    h.close()


def test_streamed_uneven_chunks_with_promotion_equal_oracle():
    """The streamed host path with its automatic cut for large batches (10 / 25 / 25 / 20 / 12 / 8 %, long sequences of the last
    chunk ordered with the chunk before it), forced here on a batch the oracle decodes in seconds: ragged lengths with a
    few very long sequences in the last chunk, u32 and u16/u8 host formats, repeated calls."""
    rng = np.random.default_rng(515)
    K, M, Bn = 45, 70, 40000
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.1)
    obs, off = random_batch(rng, Bn, M, 1, 30)
    lens = np.diff(off)
    lens[-50:] = rng.integers(200, 400, size=50)                  # long sequences at the very end: all get promoted
    lens[-2000:-1900] = 1
    off = np.concatenate(([0], np.cumsum(lens))).astype(np.int64)
    obs = rng.integers(0, M, size=int(off[-1])).astype(np.uint32)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    h = cv.HMM(A, B, pi)
    L = cv._lib.lib()
    try:
        L.cv_debug_set_chain_max_batch(0)
        L.cv_debug_set_chunks(4)                                   # take the streamed path at this size ...
        for uneven in (2, 0, 2):
            L.cv_debug_set_uneven_chunks(uneven)                   # ... with the uneven cut forced / equal chunks
            p, s = cv.decode_batch(h, obs, off)
            assert (p == rp).all() and s.tobytes() == rs.tobytes(), uneven
            p8, s8 = cv.decode_batch_narrow(h, obs.astype(np.uint16), off)
            assert (np.asarray(p8, dtype=np.uint32) == rp).all() and s8.tobytes() == rs.tobytes(), uneven
    finally:
        L.cv_debug_set_uneven_chunks(1)
        L.cv_debug_set_chunks(-1)
        L.cv_debug_set_chain_max_batch(-1)
    h.close()


def test_device_api_rejects_a_max_len_that_is_too_small():
    """cv_decode_batch_dev sorts by the bits a length <= max_len can have: a longer sequence must be CV_ERR_ARG, never a
    silently mis-ordered batch; a generous max_len is fine."""
    import torch
    rng = np.random.default_rng(31)
    K, M, Bn = 21, 30, 12000
    A, B, pi = random_hmm(rng, K, M)
    obs, off = random_batch(rng, Bn, M, 1, 70)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    h = cv.HMM(A, B, pi)
    L = cv._lib.lib()
    d_obs = torch.from_numpy(obs.view(np.int32)).cuda()
    d_off = torch.from_numpy(off).cuda()
    d_path = torch.zeros(len(obs), dtype=torch.int32, device="cuda")
    d_score = torch.zeros(Bn, dtype=torch.float64, device="cuda")
    st = torch.cuda.current_stream()
    true_max = int(np.diff(off).max())
    for ml, ok in ((true_max, True), (4 * true_max + 3, True), (0, True), (true_max - 1, False), (15, False)):
        rc = L.cv_decode_batch_dev(h.device_handle(), d_obs.data_ptr(), d_off.data_ptr(), Bn, len(obs), ml,
                                   d_path.data_ptr(), d_score.data_ptr(), st.cuda_stream, 1)
        torch.cuda.synchronize()
        if ok:
            cv._lib.check(rc)
            assert (d_path.cpu().numpy().view(np.uint32) == rp).all() and d_score.cpu().numpy().tobytes() == rs.tobytes(), ml
        else:
            assert rc == cv._lib.ERR_ARG, (ml, rc)
    h.close()


def test_decode_batch_keep_leaves_device_copies():
    """cv_decode_batch_keep: host results as cv_decode_batch, and the same results in the caller's device buffers
    (rows of an all-gather buffer in the multi-GPU path).  Streamed and per-chunk host paths."""
    import ctypes as C

    import torch
    rng = np.random.default_rng(31)
    K, M = 45, 60
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.1)
    obs, off = random_batch(rng, 60000, M, 1, 30)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    h = cv.HMM(A, B, pi)
    L = cv._lib.lib()
    hd = h.device_handle(torch.cuda.current_device())
    N, Bn = len(obs), len(off) - 1
    paths, scores = np.zeros(N, np.uint32), np.zeros(Bn)
    try:
        for chunks, streamed in ((4, 1), (3, 0), (1, 1)):
            L.cv_debug_set_chunks(chunks)
            L.cv_debug_set_pipeline(-1, streamed)
            d_path = torch.full((N,), -1, dtype=torch.int32, device="cuda")
            d_score = torch.zeros(Bn, dtype=torch.float64, device="cuda")
            cv._lib.check(L.cv_decode_batch_keep(hd, obs.ctypes.data, off.ctypes.data, Bn, paths.ctypes.data,
                                                 scores.ctypes.data, d_path.data_ptr(), d_score.data_ptr()))
            assert (paths == rp).all() and scores.tobytes() == rs.tobytes()
            assert (d_path.cpu().numpy().view(np.uint32) == rp).all() and d_score.cpu().numpy().tobytes() == rs.tobytes()
    finally:
        L.cv_debug_set_chunks(-1)
        L.cv_debug_set_pipeline(1, 1)
    h.close()


@pytest.mark.parametrize("K,Bn", [(45, 70000), (20, 500), (64, 30000)])
def test_narrow_host_formats_equal_oracle(K, Bn):
    """cv_decode_batch_u16u8 (u16 observations in, u8 states out): same paths and score bits as the oracle on the
    tile kernel (streamed and per-chunk host paths) and on the warp-per-sequence kernel; error codes as documented."""
    rng = np.random.default_rng(808 + K)
    M = 300
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.1)
    obs, off = random_batch(rng, Bn, M, 1, 30)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    h = cv.HMM(A, B, pi)
    L = cv._lib.lib()
    try:
        for chunks, streamed in ((-1, 1), (3, 0), (4, 1)):
            L.cv_debug_set_chunks(chunks)
            L.cv_debug_set_pipeline(-1, streamed)
            p, s = cv.decode_batch_narrow(h, obs, off)
            assert p.dtype == np.uint8 and (p == rp).all() and s.tobytes() == rs.tobytes()
    finally:
        L.cv_debug_set_chunks(-1)
        L.cv_debug_set_pipeline(1, 1)
    h.close()
    A2, B2, pi2 = random_hmm(rng, 70, 5)
    h2 = cv.HMM(A2, B2, pi2)
    with pytest.raises(cv.CvError) as e:                              # K > 64: not implemented for the narrow formats
        cv.decode_batch_narrow(h2, np.zeros(4, np.uint32), np.array([0, 4], np.int64))
    assert e.value.code == cv._lib.ERR_UNSUPPORTED
    h2.close()


@pytest.mark.parametrize("K", [45, 24])
def test_long_sequence_split_equals_oracle(K):
    """Short batch with a few very long sequences: the tile path hands sequences longer than its threshold to the
    warp-per-sequence kernel (LongSplit, cv_api.cu).  Host path (streamed, two chunks, long sequences in both chunks),
    narrow formats, the per-chunk host path and the device-resident path, all against the oracle."""
    import torch
    rng = np.random.default_rng(5100 + K)
    M = 80
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.1)
    Bn = 40000
    lens = rng.integers(1, 30, size=Bn)
    for b in rng.integers(0, Bn, size=25):
        lens[b] = rng.integers(200, 1500)
    off = np.zeros(Bn + 1, dtype=np.int64)
    off[1:] = np.cumsum(lens)
    obs = rng.integers(0, M, size=int(off[-1])).astype(np.uint32)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    h = cv.HMM(A, B, pi)
    L = cv._lib.lib()
    try:
        for streamed in (1, 0):
            L.cv_debug_set_pipeline(-1, streamed)
            p, s = cv.decode_batch(h, obs, off)
            assert (p == rp).all() and s.tobytes() == rs.tobytes(), f"streamed={streamed}"
            p8, s8 = cv.decode_batch_narrow(h, obs, off)
            assert (p8 == rp).all() and s8.tobytes() == rs.tobytes()
    finally:
        L.cv_debug_set_pipeline(1, 1)
    hd = h.device_handle(torch.cuda.current_device())
    N = len(obs)
    d_obs = torch.from_numpy(obs.view(np.int32)).cuda()
    d_off = torch.from_numpy(off).cuda()
    for fn, dt in ((L.cv_decode_batch_dev, torch.int32), (L.cv_decode_batch_dev_u8, torch.uint8)):
        d_path = torch.zeros(N, dtype=dt, device="cuda")
        d_score = torch.zeros(Bn, dtype=torch.float64, device="cuda")
        for _ in range(2):                                            # twice: the flags / lists are rebuilt every call
            cv._lib.check(fn(hd, d_obs.data_ptr(), d_off.data_ptr(), Bn, N, int(lens.max()), d_path.data_ptr(),
                             d_score.data_ptr(), torch.cuda.current_stream().cuda_stream, 1))
        torch.cuda.synchronize()
        got = d_path.cpu().numpy()
        got = got.astype(np.uint32) if dt == torch.uint8 else got.view(np.uint32)
        assert (got == rp).all() and d_score.cpu().numpy().tobytes() == rs.tobytes()
    h.close()


@pytest.mark.parametrize("K,ties,zero_frac", [(45, False, 0.15), (45, True, 0.0), (24, True, 0.0), (33, False, 0.5), (64, False, 0.05), (17, False, 0.1), (61, True, 0.0)])
def test_tile_path_equals_oracle_on_ties_zeros_and_sparse_models(K, ties, zero_frac):
    """The tile path (forward tile kernel + backtrace) against the oracle: models full of exact ties / +-0.0 / -inf,
    sparse models (half of the entries -inf), long sequences (delta in the thousands), u32 and narrow formats."""
    rng = np.random.default_rng(6600 + K)
    M = 40
    A, B, pi = random_hmm(rng, K, M, zero_frac=zero_frac, ties=ties)
    lens = rng.integers(1, 60, size=7000)
    lens[:6] = rng.integers(2000, 6000, size=6)              # |delta| in the thousands
    off = np.zeros(len(lens) + 1, dtype=np.int64)
    off[1:] = np.cumsum(lens)
    obs = rng.integers(0, M, size=int(off[-1])).astype(np.uint32)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    h = cv.HMM(A, B, pi)
    L = cv._lib.lib()
    try:
        L.cv_debug_set_chain_max_batch(0)
        p, s = cv.decode_batch(h, obs, off)
        assert (p == rp).all(), "paths"
        assert s.tobytes() == rs.tobytes(), "score bits"
        p8, s8 = cv.decode_batch_narrow(h, obs, off)
        assert (p8 == rp).all() and s8.tobytes() == rs.tobytes()
    finally:
        L.cv_debug_set_chain_max_batch(-1)
    h.close()


def test_tile_path_equals_oracle_with_positive_log_scores():
    """A model with positive log-scores (not log-probabilities) on the tile path still equals the oracle."""
    rng = np.random.default_rng(12)
    K, M = 40, 30
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.1)
    A[3, 5] = 0.75
    B[7, 2] = 1.5
    obs, off = random_batch(rng, 9000, M, 1, 40)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    h = cv.HMM(A, B, pi)
    L = cv._lib.lib()
    try:
        L.cv_debug_set_chain_max_batch(0)
        p, s = cv.decode_batch(h, obs, off)
        assert (p == rp).all() and s.tobytes() == rs.tobytes()
    finally:
        L.cv_debug_set_chain_max_batch(-1)
    h.close()


def test_long_sequence_split_beyond_its_capacity():
    """More sequences above the split threshold than the warp-per-sequence list holds (4096): the surplus stays in
    the tiles with its full length -- still the oracle's result."""
    rng = np.random.default_rng(5300)
    K, M, Bn = 45, 60, 40000
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.1)
    lens = rng.integers(1, 30, size=Bn)
    lens[rng.choice(Bn, size=5000, replace=False)] = rng.integers(250, 320, size=5000)
    off = np.zeros(Bn + 1, dtype=np.int64)
    off[1:] = np.cumsum(lens)
    obs = rng.integers(0, M, size=int(off[-1])).astype(np.uint32)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    h = cv.HMM(A, B, pi)
    for _ in range(2):
        p, s = cv.decode_batch(h, obs, off)
        assert (p == rp).all() and s.tobytes() == rs.tobytes()
    h.close()


@pytest.mark.parametrize("K,zero_frac", [(45, 0.05), (24, 0.3), (61, 0.0)])
def test_f32_mode_within_tolerance(K, zero_frac):
    """cv_decode_batch_f32 (optional, not the parity path): scores within 1e-5 relative of the f64 oracle
    (BASELINE.json north_star's tolerance for an f32 mode), -inf exactly where the oracle has -inf, and every
    returned path is a valid witness: re-scored in f64 with the f64 model it is within 1e-5 relative of the optimum.
    Most paths equal the oracle's; they may differ only at near-ties."""
    import torch
    rng = np.random.default_rng(7700 + K)
    M = 50
    A, B, pi = random_hmm(rng, K, M, zero_frac=zero_frac)
    obs, off = random_batch(rng, 20000, M, 1, 80)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=8)
    h = cv.HMM(A, B, pi)
    p, s = cv.decode_batch_f32(h, obs, off)
    fin = np.isfinite(rs)
    assert (np.isneginf(s) == np.isneginf(rs)).all()
    rel = np.abs(s[fin] - rs[fin]) / np.maximum(np.abs(rs[fin]), 1.0)
    assert rel.max() <= 1e-5, rel.max()
    same = np.array([(p[off[b]:off[b + 1]] == rp[off[b]:off[b + 1]]).all() for b in range(len(off) - 1)])
    assert same[fin].mean() > 0.97, same[fin].mean()
    for b in np.flatnonzero(fin & ~same)[:200]:                      # a different path must be (nearly) as good
        sc = _path_score(A, B, obs[off[b]:off[b + 1]], p[off[b]:off[b + 1]])
        assert abs(sc - rs[b]) <= 1e-5 * max(abs(rs[b]), 1.0), (b, sc, rs[b])
    # device-resident entry, deterministic
    hd = h.device_handle(torch.cuda.current_device())
    L = cv._lib.lib()
    N, Bn = len(obs), len(off) - 1
    d_obs = torch.from_numpy(obs.view(np.int32)).cuda(); d_off = torch.from_numpy(off).cuda()
    d_path = torch.zeros(N, dtype=torch.int32, device="cuda"); d_score = torch.zeros(Bn, dtype=torch.float64, device="cuda")
    cv._lib.check(L.cv_decode_batch_dev_f32(hd, d_obs.data_ptr(), d_off.data_ptr(), Bn, N, int(np.diff(off).max()),
                                            d_path.data_ptr(), d_score.data_ptr(), torch.cuda.current_stream().cuda_stream, 1))
    torch.cuda.synchronize()
    assert (d_path.cpu().numpy().view(np.uint32) == p).all() and d_score.cpu().numpy().tobytes() == s.tobytes()
    # and the exact mode is untouched by it
    p64, s64 = cv.decode_batch(h, obs, off)
    assert (p64 == rp).all() and s64.tobytes() == rs.tobytes()
    h.close()


def test_f32_mode_small_batches_take_the_exact_kernel():
    """Batches of <= 8192 sequences go to the warp-per-sequence kernel, which is f64: in f32 mode they simply return the
    exact result (documented in include/cv_b200.h), also while cv_debug_set_chain_max_batch forces the tile kernel."""
    rng = np.random.default_rng(41)
    K, M = 30, 20
    A, B, pi = random_hmm(rng, K, M, zero_frac=0.1)
    obs, off = random_batch(rng, 500, M, 1, 50)
    rp, rs = po.decode_batch(A, B, obs, off, nthreads=4)
    h = cv.HMM(A, B, pi)
    L = cv._lib.lib()
    try:
        for chain_max in (-1, 0):
            L.cv_debug_set_chain_max_batch(chain_max)
            p, s = cv.decode_batch_f32(h, obs, off)
            assert (p == rp).all() and s.tobytes() == rs.tobytes(), f"chain_max={chain_max}"
    finally:
        L.cv_debug_set_chain_max_batch(-1)
    A2, B2, pi2 = random_hmm(rng, 70, 5)
    h2 = cv.HMM(A2, B2, pi2)
    with pytest.raises(cv.CvError) as e:                              # K > 64: no f32 mode
        cv.decode_batch_f32(h2, np.zeros(4, np.uint32), np.array([0, 4], np.int64))
    assert e.value.code == cv._lib.ERR_UNSUPPORTED
    h.close(); h2.close()
