// decode_small.cuh -- batched plain Viterbi (mode R1), K <= 64.
//
// Replaces B calls of viterbi::decode (reference src/viterbi_solver/viterbi.rs:5-32).
//
// Two kernels:
//
// 1. decode_small_fwd_kernel -- forward max-plus recurrence, VALUE ONLY.
//    sm_100a has neither a 64-bit select nor DMNMX, so tracking (value, argmax)
//    per cell costs DADD + DSETP + 3 selects and is bound by the ALU pipe (ncu:
//    alu 74 %, fp64 49 %).  The forward pass therefore keeps only the running
//    maximum (DADD + DSETP + 2 FSEL) and writes every delta row to HBM ("delta
//    history").  The backpointer psi[t][s] = first-argmax_j fl(delta[t-1][j] +
//    logA[j][s]) is a pure function of the stored row, so the backtrace recomputes
//    it only for the one state per step on the decoded path (K cells, not K*K).
//
//    Mapping: persistent CTAs pull tiles of NS = 64 sequences (pre-sorted by
//    length, longest first, so a tile runs in lock step).  Shared memory holds
//      sA  [K][Kp]      logA, staged once per CTA by a TMA bulk copy
//      sD  [2][K][NS]   delta, double buffered, [state][sequence slot]
//      sEm [NS][Kp+2]   this step's emission rows logB^T[o_t(s)][.], fetched by TMA
//                       bulk copies (one 8*Kp-byte row per sequence, L2 resident)
//    A lane owns TP=2 adjacent sequences (one conflict-free LDS.128 per j), a warp
//    owns TQ=8 adjacent target states (four broadcast LDS.128 per j): 16 cells per
//    thread per predecessor from 5 shared loads.  Warps = G state groups
//    (G = ceil(K/8)).  After the j loop the thread adds the
//    emission ((delta + a) + b, viterbi.rs:17; an emission of -inf gives -inf,
//    viterbi.rs:19-21) and stores 8 x double2 into the other buffer; after the
//    step barrier one thread writes the whole [K][NS] slab to the history with a
//    single TMA bulk store.  No per-thread global loads or stores remain in the
//    step loop except the observation prefetch of the producer warp.
//
//    History layout: slab (tile, t) at hist + (tile_base[tile] + t) * K * NS,
//    tile_base = exclusive scan of the tiles' longest lengths.
//
// 2. backtrace_small_kernel -- end state (viterbi.rs:24) and backtrace
//    (viterbi.rs:25-30) with lazy psi; one thread per sequence, a warp holds 32
//    adjacent sequences of a tile so every slab-row read is a coalesced 256-byte
//    run; rows are prefetched in chunks of 16 predecessors ahead of the reduce.
#pragma once

#include "common.cuh"

namespace cvb {

struct DecodeSmallParams {
    const double *A;         // [K][Kp]   logA, columns >= K padded with -inf (natural column order: the backtrace)
    const double *BT;        // [M][Kp]   logB transposed (obs-major), padded -inf
    const double *At, *BTt;  // what the forward tile kernel reads: A / BT, or their slot-permuted copies (balanced split)
    const float *A32n;       // f32 mode (decode_f32.cuh): rn32(logA) [K][Kp], natural columns (backtrace)
    const float *A32s;       //                            rn32(logA) [K][Kp], slot-permuted like At (forward kernel)
    const float *BT32;       //                            rn32(logB^T) [M][Kp], slot-permuted like BTt
    const uint32_t *obs;     // [N]
    const int64_t *seq_off;  // [B+1]
    const uint32_t *order;   // [B] sequence ids, longest first
    const long long *tile_base;  // [ntiles] first slab of each tile
    double *hist;            // delta history slabs, [K][NS] each
    long long hist_cap_slabs;    // slabs the history buffer holds (a tile past it is refused, status 7)
    uint32_t *path;          // [N]
    double *score;           // [B] or nullptr
    unsigned int *tile_counter;
    int *status;             // 0 ok, else CV_ERR_*
    // concurrent backtrace (nullptr = the backtrace runs after the forward kernel): tile_done is a QUEUE of finished
    // tiles in completion order -- a forward CTA appends tile + 1 (slot = atomicAdd(started + 1)) once the tile's
    // history is complete in global memory, backtrace warp q / 2 takes queue slot q.  (Indexed by tile id the first
    // backtrace CTAs would sit on the longest tiles, which finish last, while hundreds of short tiles queue up behind
    // them.)  started[0] counts the forward CTAs that have begun.
    int *tile_done;
    unsigned int *started;
    // streamed host path (nullptr / 0 otherwise): one launch over the whole batch while the observations still
    // arrive chunk by chunk and the paths already leave chunk by chunk.  Sequences are ordered by (chunk, length);
    // a tile may start once *arrived > tile_chunk[tile]; chunk_done[c] counts the finished sequences of chunk c.
    const long long *tile_tmax;      // longest sequence of every tile (a tile can straddle two chunks)
    const int *tile_chunk;           // last chunk a tile takes sequences from
    const unsigned int *arrived;     // chunks whose observations are on the device (written by the copy stream)
    unsigned int *chunk_done;
    int nch;
    int64_t cb[18];                  // chunk boundaries: chunk c = sequences [cb[c], cb[c+1])
    int64_t M, B;
    int K, Kp, G, NS, ntiles;      // NS = sequences per tile (64)
    // balanced state split: state group g owns nq_base + (g < nq_rem) states starting at state
    // g * nq_base + min(g, nq_rem); the columns of A / BT are permuted into 8-wide slots per group (slot 8g + q holds
    // that group's q-th state, unused slots -inf).  nq_base = 0: the plain layout (group g = states 8g .. 8g+7).
    int nq_base, nq_rem;
    int em_light;   // 1: with an uneven balanced split the lighter state groups fetch more of the emission rows
    // narrow host formats (cv_decode_batch_u16u8): obs holds u16 observations, path receives u8 states
    int obs16, path8;
    // long-sequence split: sequences flagged here are decoded by the warp-per-sequence kernel, the tile kernels treat
    // them as inactive slots (nullptr: no split)
    const uint8_t *is_long;
    // certified backtrace (backtrace_small_kernel<.., float, true>): the ids of the sequences it could not certify are
    // appended to cert_list; cert_count[0] = how many, [1] = their longest length, [2..3] = their elements (u64).
    // cert_tol scales the error bound: 1 = the derived bound, 0 = certify every decision, inf = none.
    uint32_t *cert_list;
    unsigned int *cert_count;
    double cert_tol;
};

// element `idx` of the observation array (u32, or u16 when obs16); `coherent`: the copy engine is still writing the
// buffer (streamed host path), so the read-only path and L1 must not be used
__device__ __forceinline__ uint32_t load_obs_at(const DecodeSmallParams &p, int64_t idx, bool coherent)
{
    if (p.obs16) {
        const uint16_t *q = reinterpret_cast<const uint16_t *>(p.obs) + idx;
        return coherent ? (uint32_t)__ldcg(q) : (uint32_t)__ldg(q);
    }
    return coherent ? __ldcg(p.obs + idx) : __ldg(p.obs + idx);
}
__device__ __forceinline__ void store_path_at(const DecodeSmallParams &p, int64_t idx, uint32_t state)
{
    if (p.path8) reinterpret_cast<uint8_t *>(p.path)[idx] = (uint8_t)state;
    else p.path[idx] = state;
}
// reads back a state this thread stored (plain load: the read-only path could serve a stale line)
__device__ __forceinline__ uint32_t load_path_at(const DecodeSmallParams &p, int64_t idx)
{
    return p.path8 ? (uint32_t)reinterpret_cast<const uint8_t *>(p.path)[idx] : p.path[idx];
}

__host__ __device__ inline int em_pitch(int Kp) { return Kp + 2; }   // doubles; bank-conflict-free row pitch

// dynamic smem: [A][delta x2][em][off i64][len i32][mbarA, mbarEm][tile]
// lda = row pitch of logA in shared memory, in doubles: Kp, or FWD_LDC for the constant-stride kernel
__host__ __device__ inline size_t decode_small_smem_bytes(int K, int Kp, int NS, int lda = 0)
{
    return (size_t)K * (lda ? lda : Kp) * 8 + (size_t)2 * K * NS * 8 + (size_t)NS * em_pitch(Kp) * 8 + (size_t)NS * (8 + 4) + 32 + 16;
}

// value-only TP x TQ micro-tile over predecessors [0, nj), nj >= 1: best[p][q] = max_j ( dcol[j*ldd + p] + arow[j*lda + q] )
// (strict > keeps the first maximum's bits, e.g. the sign of a zero, as the reference does).
// NQ <= TQ: only the first NQ target states of the slot group are computed (balanced split: the slots behind them
// are padding); the operand loads stay 16-byte pairs.
// LDC > 0: both row pitches are the compile-time constant LDC (doubles) -- every operand load of an unrolled iteration is
// base + immediate off two pointers that advance once per iteration (with run-time pitches: two IMADs per predecessor)
template <int NQ, int LDC>
__device__ __forceinline__ void maxplus_tile_val(const double *__restrict__ dcol, int ldd_rt,
                                                 const double *__restrict__ arow, int lda_rt, int nj,
                                                 double (&best)[TP][TQ])
{
    const int ldd = LDC ? LDC : ldd_rt, lda = LDC ? LDC : lda_rt;
    // operands of one predecessor: dp / ap point at its delta row and its logA row
    auto load = [&](const double *dp, const double *ap, double (&dd)[TP], double (&a)[TQ]) {
#pragma unroll
        for (int p = 0; p < TP / 2; p++) {
            const double2 d = *reinterpret_cast<const double2 *>(dp + 2 * p);
            dd[2 * p] = d.x; dd[2 * p + 1] = d.y;
        }
#pragma unroll
        for (int q = 0; q < (NQ + 1) / 2; q++) {
            const double2 aa = *reinterpret_cast<const double2 *>(ap + 2 * q);
            a[2 * q] = aa.x; a[2 * q + 1] = aa.y;
        }
    };
    // the two row pointers walk the predecessors (no index arithmetic in the loop)
    const double *dp = dcol, *ap = arow;
    const double *const dend = dcol + (size_t)nj * ldd;
    {
        // predecessor 0 starts the running maximum: `best = -inf; if (v > best) best = v` leaves best = v for every v
        // that can occur (v is never NaN), so the initialisation and the first compare/select are dropped
        double dd[TP], a[TQ];
        load(dp, ap, dd, a);
#pragma unroll
        for (int p = 0; p < TP; p++)
#pragma unroll
            for (int q = 0; q < NQ; q++) best[p][q] = dd[p] + a[q];
        dp += ldd; ap += lda;
    }
    // two predecessors are reduced before they meet the running maximum: the dependent chain on `best` is one
    // compare/select per two predecessors.  `b > a ? b : a` keeps the EARLIER value on a tie at
    // every level, so the result carries the bits of the first maximum exactly as the sequential scan does.
    // Measured at the POS shape (K = 45), forward kernel alone / whole step: pairs, two per iteration, 10.60 / 11.30 ms;
    // one predecessor at a time unrolled 2: 10.94 / 11.49 ms, 4: 10.63 / 11.36 ms, 11: 10.27 / 12.64 ms -- the
    // loop-carried register moves at the back edge amortise with the unroll factor, but the 13 KB loop bodies (one per
    // state-group width) then fight the concurrent backtrace for the instruction cache.
    const double *const dend2 = dp + (size_t)((nj - 1) & ~1) * ldd;      // an even number of predecessors
#pragma unroll 2
    for (; dp != dend2; dp += 2 * ldd, ap += 2 * lda) {
        double d0[TP], d1[TP], a0[TQ], a1[TQ];
        load(dp, ap, d0, a0); load(dp + ldd, ap + lda, d1, a1);
#pragma unroll
        for (int p = 0; p < TP; p++)
#pragma unroll
            for (int q = 0; q < NQ; q++) {
                const double v0 = d0[p] + a0[q], v1 = d1[p] + a1[q];
                const double m = v1 > v0 ? v1 : v0;
                best[p][q] = m > best[p][q] ? m : best[p][q];
            }
    }
#pragma unroll 1
    for (; dp != dend; dp += ldd, ap += lda) {                       // at most one predecessor is left
        double dd[TP], a[TQ];
        load(dp, ap, dd, a);
#pragma unroll
        for (int p = 0; p < TP; p++)
#pragma unroll
            for (int q = 0; q < NQ; q++) {
                const double v = dd[p] + a[q];
                best[p][q] = v > best[p][q] ? v : best[p][q];
            }
    }
}

__device__ __forceinline__ void tma_bulk_s2g(void *dst_gmem, const void *src_smem, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem),
                 "r"(smem_u32(src_smem)), "r"(bytes)
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait_read_all()
{
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
// all bulk stores of this thread have been written (not only read out of shared memory)
__device__ __forceinline__ void tma_store_wait_all()
{
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// One step of one thread: its TP sequences x NQ target states.  best = max_j (delta[t-1][j] + a[j][i]) over all
// predecessors (value only), then (.. + b) (viterbi.rs:17) into the other delta buffer.  `row0` points at the row of the
// group's first state in that buffer, `nreal` = how many of the NQ states exist (the last group of the plain layout
// may reach past K).
template <int NQ, int LDC>
__device__ __forceinline__ void fwd_step(const double *__restrict__ dcur, double *__restrict__ row0, int NS_rt,
                                         const double *__restrict__ arow, int lda, int K, const double *__restrict__ e0, int EP,
                                         uint64_t *em_bar, uint32_t em_phase, int nreal)
{
    const int NS = LDC ? LDC : NS_rt;
    double best[TP][TQ];
    maxplus_tile_val<NQ, LDC>(dcur, NS, arow, lda, K, best);     // K >= 1: predecessor 0 exists

    mbar_wait(em_bar, em_phase);      // emission rows of step t have landed
#pragma unroll
    for (int k = 0; k < (NQ + 1) / 2; k++) {
        double2 x[TP];
#pragma unroll
        for (int q = 0; q < TP; q++) x[q] = *reinterpret_cast<const double2 *>(e0 + (size_t)q * EP + 2 * k);
        // (delta + a) + b (viterbi.rs:17).  Sequences that already ended compute garbage in their
        // own column only; their last row is already in the history.
#pragma unroll
        for (int q = 0; q < TP; q += 2) {
            if (2 * k < nreal)
                *reinterpret_cast<double2 *>(row0 + (size_t)(2 * k) * NS + q) =
                    make_double2(best[q][2 * k] + x[q].x, best[q + 1][2 * k] + x[q + 1].x);
            if (2 * k + 1 < NQ && 2 * k + 1 < nreal)
                *reinterpret_cast<double2 *>(row0 + (size_t)(2 * k + 1) * NS + q) =
                    make_double2(best[q][2 * k + 1] + x[q].y, best[q + 1][2 * k + 1] + x[q + 1].y);
        }
    }
}

// One warp per state group of TQ = 8 target states, TP = 2 sequences per lane: 32 * G threads per CTA.
// LDC > 0 (= FWD_LDC = 64): tiles of exactly LDC sequences and logA rows at a pitch of LDC doubles in shared memory,
// both known at compile time (see maxplus_tile_val); 0: run-time NS and pitch Kp.
constexpr int FWD_LDC = 64;
template <int LDC>
__global__ void __launch_bounds__(512, 1) decode_small_fwd_kernel(const DecodeSmallParams p)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int K = p.K, Kp = p.Kp, NS = LDC ? LDC : p.NS, EP = em_pitch(Kp);
    const int lda = LDC ? LDC : Kp;
    double *sA = reinterpret_cast<double *>(smem_raw);
    double *sD = sA + (size_t)K * lda;
    double *sEm = sD + (size_t)2 * K * NS;
    int64_t *sOff = reinterpret_cast<int64_t *>(sEm + (size_t)NS * EP);
    int *sLen = reinterpret_cast<int *>(sOff + NS);
    uint64_t *sBar = reinterpret_cast<uint64_t *>(sLen + NS);   // [0] logA, [1] emissions
    int *sTile = reinterpret_cast<int *>(sBar + 4);

    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int g = w % p.G, sg = w / p.G;
    const int i0 = g * TQ;                                   // first column slot of the group in sA / sEm
    // first state (= delta row) of the group and how many of its TQ slots are real states
    const int srow0 = p.nq_base ? g * p.nq_base + min(g, p.nq_rem) : i0;
    const int nreal = p.nq_base ? p.nq_base + (g < p.nq_rem ? 1 : 0) : max(0, min(TQ, K - i0));
    const int s0 = sg * (32 * TP) + lane * TP;
    const uint32_t slab_bytes = (uint32_t)((size_t)K * NS * 8);
    const uint32_t row_bytes = (uint32_t)(Kp * 8);
    constexpr int EMK = 2 * TP;    // emission slots a lane may serve: NS / (32 * warps) <= TP, x2 slack

    // Who fetches the emission rows.  The per-step barrier makes the slowest warp's step the CTA's, so the fetch work
    // (one elected-lane TMA issue per row, ~10 instructions) is dealt out by how much tile work a warp has: with an
    // uneven balanced split the groups behind the first nq_rem own one state less -- K predecessors x 2 cells per lane
    // x ~4.5 instructions = ~9 K instructions per step less, worth ~0.9 K rows -- and take that many more rows each
    // (K = 45: the three 7-state warps fetch all 64 rows, the 8-state warps none).  Warp w owns the slots
    // [em_beg, em_beg + em_cnt); lane l serves em_beg + l + 32 k.  Otherwise every warp takes an equal share.
    const int nwarps = (int)blockDim.x >> 5;
    int em_beg = 0, em_cnt = 0, n_fetch = 0;
    {
        const bool uneven = p.em_light && p.nq_base && p.nq_rem;
        const int nlight = uneven ? p.G - p.nq_rem : 0;
        const int extra = uneven ? min(NS / nlight, (9 * K + 5) / 10) : 0;      // additional rows per lighter warp
        const int rest = NS - extra * nlight, base = rest / nwarps, left = rest - base * nwarps;
        // the `left` rows that remain go one each to the last warps (the lighter ones, if any)
        int beg = 0;
        for (int v = 0; v < nwarps; v++) {
            const int c = base + ((uneven && v % p.G >= p.nq_rem) ? extra : 0) + (v >= nwarps - left ? 1 : 0);
            if (v == w) { em_beg = beg; em_cnt = c; }
            if (c > 0) n_fetch++;
            beg += c;
        }
    }
    const int emk = (em_cnt + 31) / 32;                                                            // slots per lane that exist
    const int st_tid = (p.em_light && p.nq_base && p.nq_rem) ? 32 * p.nq_rem : 0;      // the thread that issues (and waits for) the history slab stores: one of a lighter warp
    // ---- stage logA once per CTA (TMA bulk copy, UBLKCP) ----
    if (tid == 0) {
        if (p.started) atomicAdd(p.started, 1u);   // the backtrace kernel is released once every forward CTA is resident
        mbar_init(sBar, 1);
        mbar_init(sBar + 1, n_fetch);              // one arrival per fetching warp and step
        fence_proxy_async_smem();
        const uint32_t bytes = (uint32_t)((size_t)K * Kp * 8);
        mbar_expect_tx(sBar, bytes);
        if (LDC && lda != Kp) {
            for (int r = 0; r < K; r++) tma_bulk_g2s(sA + (size_t)r * lda, p.At + (size_t)r * Kp, row_bytes, sBar);   // row by row into the wider pitch
        } else {
            tma_bulk_g2s(sA, p.At, bytes, sBar);
        }
    }
    __syncthreads();
    mbar_wait(sBar, 0);
    uint32_t em_phase = 0;

    // Emission rows of step t for every sequence still running: each fetching warp issues one TMA row copy per slot of
    // its share (see em_beg / em_cnt above) and arrives once on the emission mbarrier with the byte count of that share.
    auto issue_emissions = [&](int t, const uint32_t (&o_cur)[EMK]) {
        int nact = 0;
#pragma unroll
        for (int k = 0; k < EMK; k++) {
            if (k >= emk) break;
            const int s = em_beg + lane + 32 * k;
            if (lane + 32 * k < em_cnt && t < sLen[s]) nact++;
        }
        const int total = __reduce_add_sync(0xffffffffu, nact);
        if (lane == 0) mbar_expect_tx(sBar + 1, (uint32_t)total * row_bytes);   // arrive + expected bytes (0 is fine)
        __syncwarp();
#pragma unroll
        for (int k = 0; k < EMK; k++) {
            if (k >= emk) break;
            const int s = em_beg + lane + 32 * k;
            if (lane + 32 * k < em_cnt && t < sLen[s]) {
                uint32_t o = o_cur[k];
                if ((int64_t)o >= p.M) { *p.status = 3; o = 0; }   // index panic in the reference
                tma_bulk_g2s(sEm + (size_t)s * EP, p.BTt + (size_t)o * Kp, row_bytes, sBar + 1);
            }
        }
    };

    // Observations.  On the streamed host path the copy engine is still writing later chunks of p.obs while this
    // kernel runs, so the read-only (non-coherent) path and L1 must not be used: a sector that straddles a chunk
    // boundary could be served stale.  ld.global.cg reads through to L2, where the copy engine's writes land before
    // the `arrived` word that releases the chunk.
    const bool obs_streamed = p.arrived != nullptr;
    auto ld_obs = [&](int64_t idx) -> uint32_t { return load_obs_at(p, idx, obs_streamed); };

    unsigned int arrived_seen = 0;      // (thread 0) chunks of observations known to be on the device
    for (;;) {
        if (tid == 0) *sTile = (int)atomicAdd(p.tile_counter, 1u);
        __syncthreads();
        const int tile = *sTile;
        if (tile >= p.ntiles) break;

        // ---- tile set-up: sequence slots, delta(0) = 0.0 (viterbi.rs:6) ----
        for (int s = tid; s < NS; s += blockDim.x) {
            const int64_t r = (int64_t)tile * NS + s;
            int64_t off = 0; int len = 0;
            if (r < p.B) {
                const uint32_t b = p.order[r];
                off = p.seq_off[b];
                len = (int)(p.seq_off[b + 1] - off);
                if (p.is_long && p.is_long[b]) len = 0;              // decoded by the warp-per-sequence kernel
            }
            sOff[s] = off; sLen[s] = len;
        }
        for (int e = tid; e < K * NS; e += blockDim.x) sD[e] = 0.0;
        if (p.arrived && tid == 0) {
            // streamed input: the tile's observations must have arrived (bounded wait, then error).  The count only
            // grows, so the system-scope load is skipped once this thread has seen enough chunks arrive.
            const unsigned int need = (unsigned int)p.tile_chunk[tile] + 1u;
            const long long t0 = clock64();
            while (arrived_seen < need) {
                asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(arrived_seen) : "l"(p.arrived) : "memory");
                if (arrived_seen >= need) break;
                if (clock64() - t0 > (1LL << 32)) { *p.status = 5; break; }
                __nanosleep(128);
            }
        }
        fence_proxy_async_smem();
        __syncthreads();

        // the longest sequence of the tile: slot 0 when the tile is sorted by length, else precomputed
        int Tmax = p.tile_tmax ? (int)p.tile_tmax[tile] : sLen[0];
        if (p.tile_base[tile] + (long long)Tmax > p.hist_cap_slabs) {
            // cannot happen with the host's sizing (launch_decode_small); never store past the history buffer
            if (tid == 0) atomicMax(p.status, 7);
            Tmax = 0;
        }
        double *slab = p.hist + (size_t)p.tile_base[tile] * K * NS;
        if (tid == st_tid && Tmax > 0) tma_bulk_s2g(slab, sD, slab_bytes);   // history slab 0 = delta(0)

        uint32_t o_nxt[EMK];                                                  // obs of the NEXT step to fetch
        {
            uint32_t o1[EMK];
#pragma unroll
            for (int k = 0; k < EMK; k++) {
                const int s = em_beg + lane + 32 * k;
                const bool in = lane + 32 * k < em_cnt;
                o1[k] = (in && 1 < sLen[s]) ? ld_obs(sOff[s] + 1) : 0u;
                o_nxt[k] = (in && 2 < sLen[s]) ? ld_obs(sOff[s] + 2) : 0u;
            }
            if (Tmax > 1 && em_cnt > 0) issue_emissions(1, o1);
        }

        for (int t = 1; t < Tmax; t++) {
            const double *dcur = sD + (size_t)((t - 1) & 1) * K * NS + s0;
            double *row0 = sD + (size_t)(t & 1) * K * NS + (size_t)srow0 * NS + s0;
            const double *e0 = sEm + (size_t)s0 * EP + i0;
            bool done = false;
            if (p.nq_base != 0) {
                // balanced split: this group's state count (warp-uniform); groups of fewer than 5 states take the
                // full-width path below (their unused slots hold -inf and are not stored)
                done = true;
                switch (nreal) {
                    case 7: fwd_step<7, LDC>(dcur, row0, NS, sA + i0, lda, K, e0, EP, sBar + 1, em_phase, nreal); break;
                    case 6: fwd_step<6, LDC>(dcur, row0, NS, sA + i0, lda, K, e0, EP, sBar + 1, em_phase, nreal); break;
                    case 5: fwd_step<5, LDC>(dcur, row0, NS, sA + i0, lda, K, e0, EP, sBar + 1, em_phase, nreal); break;
                    default: done = false;
                }
            }
            if (!done) fwd_step<TQ, LDC>(dcur, row0, NS, sA + i0, lda, K, e0, EP, sBar + 1, em_phase, nreal);
            em_phase ^= 1;
            fence_proxy_async_smem();           // make this thread's delta writes visible to the TMA store
            if (tid == st_tid) tma_store_wait_read_all();   // slab t-1 has left the buffer step t+1 will overwrite
            __syncthreads();
            if (tid == st_tid) tma_bulk_s2g(slab + (size_t)t * K * NS, sD + (size_t)(t & 1) * K * NS, slab_bytes);
            if (t + 1 < Tmax && em_cnt > 0) {
                issue_emissions(t + 1, o_nxt);
#pragma unroll
                for (int k = 0; k < EMK; k++) {
                    if (k >= emk) break;
                    const int s = em_beg + lane + 32 * k;
                    o_nxt[k] = (lane + 32 * k < em_cnt && t + 2 < sLen[s]) ? ld_obs(sOff[s] + t + 2) : 0u;
                }
            }
        }
        if (tid == st_tid) {
            if (p.tile_done) {
                // the tile's history is complete in global memory: hand it to the concurrent backtrace
                tma_store_wait_all();
                asm volatile("fence.proxy.async;" ::: "memory");
                __threadfence();
                const unsigned int slot = atomicAdd(p.started + 1, 1u);
                asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p.tile_done + slot), "r"(tile + 1) : "memory");
            } else {
                tma_store_wait_read_all();         // last slab read out before the buffers are reused
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------
// End state + backtrace with lazy backpointers: one thread per sequence.
//
// Why no emission lookup is needed: the reference leaves psi[t][s] = 0 when b[s][o_t] = -inf
// (viterbi.rs:7,19-21) and otherwise stores argmax_j(delta[t-1][j] + a[j][s]).  If delta[t][s] > -inf the
// emission was finite and the argmax is recomputed here.  If delta[t][s] = -inf then either the emission was
// -inf (psi = 0) or every candidate was -inf (argmax of an all -inf vector = 0): psi = 0 both ways.  That needs
// finite sums never to round to -inf: cv_hmm_create refuses finite entries beyond 2^900 (the f32 mode: 2^64), which
// keeps every sum of fewer than 2^63 entries finite.
// ---------------------------------------------------------------------------
// BT_CHUNK = predecessors per prefetch chunk: 16 when the kernel has the GPU to itself (124 registers), 8 with at most
// 64 registers for the concurrent mode, where it lives on the 16 K registers per SM two forward CTAs leave free

// One thread per sequence; the 32 lanes of a warp hold 32 adjacent sequences of one tile, so the loads of
// predecessor j are one coalesced 256-byte run of the slab row.  Rows do not depend on the decoded path, so
// the next chunk of 16 predecessors is always in flight while the current one is reduced; the only dependent
// chain per step is 16 x (DADD, DSETP, select) x ceil(K/16).
// streamed host path: sequence b is decoded -- its path and score may be copied out once its whole chunk is
__device__ __forceinline__ int bt_chunk_of(const DecodeSmallParams &p, uint32_t b)
{
    int c = 0;
    while (c + 1 < p.nch && (int64_t)b >= p.cb[c + 1]) c++;
    return c;
}
// Called by ALL 32 lanes of a warp once their sequences of this round are decoded (c = chunk of the lane's sequence,
// -1 = none): one system-scope fence and one atomic per warp and chunk instead of one per sequence.  The lanes' path /
// score stores are ordered before the leader's fence by the warp-level synchronisation of the match.
__device__ __forceinline__ void bt_mark_done_warp(const DecodeSmallParams &p, int c)
{
    if (!p.chunk_done) return;
    const unsigned int same = __match_any_sync(0xffffffffu, c);
    if (c >= 0 && (threadIdx.x & 31) == __ffs(same) - 1) {
        __threadfence_system();                              // path / score stores before the count the copy stream waits for
        atomicAdd(p.chunk_done + c, (unsigned int)__popc(same));
    }
}

// History rows are read with the default L2 policy (ld.global.cg), not evict-first (ld.global.cs): the one value of the
// row that a step reads again -- delta[tt-1][state], a per-lane gather -- then still hits L2.  With evict-first the
// backtrace read 11.6 GB from DRAM for a 9.0 GB history and took 2.1 ms alone; now 1.03x the history and 1.7 ms.
template <typename T>
__device__ __forceinline__ T bt_ld(const T *q) { return __ldcg(q); }

// ---------------------------------------------------------------------------
// Certified backtrace (CERT = true, T = float): the exact f64 decode from the f32 history of decode_f32_fwd_kernel.
//
// Model (cv_hmm_create, cv_hmm::cert_ok): every finite entry of logA / logB is <= 0 and has |x| <= 2^64.  Then every
// delta and every candidate is <= 0, no finite sum of fewer than 2^63 entries overflows in f32 or f64, and the f32 and
// f64 recurrences have the same -inf pattern (a cell is -inf iff every path into it holds a -inf entry).  On values of
// one sign fl(x + y) and max are monotone, so with C = the exact max-plus value of a cell (real arithmetic on the f64
// entries) and n roundings along the way, a rounded result lies in [C (1+u)^n, C (1-u)^n], plus an absolute term for
// entries that rn32 puts in the f32 subnormal range (|error| <= 2^-150 each; an add whose result is subnormal is exact).
//
// Decision at step t (t = tt for the backpointer of step tt, whose candidates fl(delta[tt-1][j] + a[j][cur]) take 2tt-1
// adds; t = len-1 for the end state): the f32 candidate carries <= 2t roundings of u32 = 2^-24 (adds plus the one
// rounding of the entries), the f64 candidate <= 2t of u64 = 2^-53.  Let v = the f32 first maximum (index m) and
// r = the largest other f32 candidate.  For j != m: c64[j] <= c32[j] (1-e64)/(1+e32) <= r + |r| E, and
// c64[m] >= v - |v| E, with E = (1+u32)^(2t) (1+u64)^(2t) / (1 - ...) - 1 <= (2t+2) u32 while (2t+2) u32 < 1/2.  So
//     v - r > E (|v| + |r|) + 2 eta,   eta = 2t 2^-150 (times at most 2 for the relative factors),
// makes c64[m] strictly the largest f64 candidate: the f64 first-argmax is m as well.  The test below uses
//     v - r > s ((2t+4) 2^-23 (|v| + |r|) + (2t+2) 2^-148),   s = cert_tol (1 by default),
// a factor of 2 over E and 2 eta, which also absorbs the f64 rounding of the test itself (a few 2^-53 relative);
// the gap is evaluated in f64.  A runner-up of -inf (one finite candidate) always passes: the f64 row has the same single
// finite candidate.  A decision with delta[tt][cur] = -inf is psi = 0 in both recurrences and needs no test.
//
// If every decision of a path passes, the f32 path is the f64 path, and along it every f64 maximum is the path's own
// candidate, so the f64 score is the chain  d = fl(fl(d + a[p(t-1)][p(t)]) + b[p(t)][o(t)])  from d = 0.0 -- bit for bit
// what the f64 forward kernel computes (a -inf along the way stays -inf: the -inf => psi = 0 rule puts a -inf term in the
// chain).  A sequence with a failed test is appended to cert_list and decoded again by the exact f64 kernels.
// ---------------------------------------------------------------------------
__device__ __forceinline__ bool cert_pass(float v, float r, int t, double tol)
{
    if (!(r > -INFINITY) || tol == 0.0) return true;
    const double dv = v, dr = r;
    return dv - dr > tol * ((2.0 * t + 4.0) * 0x1p-23 * (fabs(dv) + fabs(dr)) + (2.0 * t + 2.0) * 0x1p-148);
}

// History slabs [K][64] (decode_small_fwd_kernel, decode_f32_fwd_kernel); the tile size is a compile-time constant
// so that the load offsets become immediates.
// T = double (exact, the reference's arithmetic) or float (cv_decode_batch_f32: the f32 history of decode_f32.cuh and
// rn32(logA), same first-maximum rule on fl32 sums).  CERT (T = float only): the certified backtrace described above.
template <int BT_CHUNK, int MINB, typename T = double, bool CERT = false>
__global__ void __launch_bounds__(128, MINB) backtrace_small_kernel(const DecodeSmallParams p)
{
    static_assert(!CERT || sizeof(T) == 4, "the certified backtrace reads the f32 history");
    const T NEG = (T)neg_inf();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int NS = 64;
    const int K = p.K, Kp = p.Kp;
    const int ATP = K | 1;                                   // odd pitch: rows of different states spread over banks
    T *sAT = reinterpret_cast<T *>(smem_raw);               // sAT[s*ATP + j] = logA[j][s]
    if (CERT) {
        // padding columns and the chunk padding behind the last row are zeros: they meet -inf operands only, and the
        // runner-up must never see a NaN
        for (int e = threadIdx.x; e < K * ATP + BT_CHUNK; e += blockDim.x) {
            const int s = e / ATP, j = e % ATP;
            sAT[e] = (s < K && j < K) ? (T)p.A32n[(size_t)j * Kp + s] : (T)0;
        }
    } else {
        for (int e = threadIdx.x; e < K * Kp; e += blockDim.x) {
            const int j = e / Kp, s = e % Kp;
            if (s < K) sAT[(size_t)s * ATP + j] = sizeof(T) == 4 ? (T)p.A32n[e] : (T)p.A[e];
        }
    }
    __syncthreads();

    const size_t sl = (size_t)K * NS;
    const int nfull = K / BT_CHUNK, ktail = K - nfull * BT_CHUNK;   // full chunks, predecessors of the partial last chunk
    const int nchunk = nfull + (ktail ? 1 : 0);
    const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
    const int64_t total = (int64_t)p.ntiles * NS;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < total; r += nthreads) {
        int tile = (int)(r / NS);
        const int s = (int)(r % NS);
        if (p.tile_done) {
            // concurrent mode: the forward kernel is still running; this warp (32 sequences of one tile) takes queue
            // slot r / NS and waits until a finished tile is published there (bounded: ~17 s -- a tile of a million
            // steps takes ~3 s --, then error).  One lane polls, about once a microsecond: tens of thousands of
            // threads polling L2 would slow the forward kernel.
            int v = 0;
            if ((threadIdx.x & 31) == 0) {
                const long long t0 = clock64();
                for (;;) {
                    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p.tile_done + tile) : "memory");
                    if (v) break;
                    if (clock64() - t0 > (1LL << 35)) { *p.status = 5; v = tile + 1; break; }
                    __nanosleep(1000);
                }
            }
            tile = __shfl_sync(0xffffffffu, v, 0) - 1;
            __threadfence();                                   // the leader's acquire, extended to the lanes that waited
        }
        // the lane's sequence; returns the chunk it belongs to on the streamed host path (-1: nothing to report)
        const int done_chunk = [&]() -> int {
        const int64_t rr = (int64_t)tile * NS + s;                     // rank in the length-sorted order
        if (rr >= p.B) return -1;
        const uint32_t b = p.order[rr];
        if (p.is_long && p.is_long[b]) return -1;                     // the warp-per-sequence kernel owns this sequence
        const int my_chunk = p.chunk_done ? bt_chunk_of(p, b) : -1;
        const int64_t off = p.seq_off[b];
        const int len = (int)(p.seq_off[b + 1] - off);
        if (len <= 0 || p.tile_base[tile] + (long long)len > p.hist_cap_slabs) return my_chunk;   // tile refused by the forward kernel (status 7)
        const T *col = reinterpret_cast<const T *>(p.hist) + (size_t)p.tile_base[tile] * sl + (size_t)s;   // sequence s of slab 0

        // certified backtrace: every decision passed its test so far (inf tolerance: none does)
        bool ok = p.cert_tol < INFINITY;
        // certified: the f64 score along the decoded path, or the sequence goes to the exact fallback
        auto cert_finish = [&]() {
            if (!ok) {
                p.cert_list[atomicAdd(p.cert_count, 1u)] = b;
                atomicMax(p.cert_count + 1, (unsigned int)len);
                atomicAdd(reinterpret_cast<unsigned long long *>(p.cert_count + 2), (unsigned long long)len);
                return;
            }
            if (!p.score) return;
            double d = 0.0;                                   // viterbi.rs:6
            uint32_t prev = load_path_at(p, off);
#pragma unroll 4
            for (int t = 1; t < len; t++) {
                const uint32_t st = load_path_at(p, off + t);
                uint32_t o = load_obs_at(p, off + t, false);
                if ((int64_t)o >= p.M) o = 0;                    // reported by the forward kernel (status 3)
                d = (d + __ldg(p.A + (size_t)prev * Kp + st)) + __ldg(p.BT + (size_t)o * Kp + st);   // viterbi.rs:17
                prev = st;
            }
            p.score[b] = d;
        };

        // end state: argmax of the last row (viterbi.rs:24)
        const T *row = col + (size_t)(len - 1) * sl;
        T bv = bt_ld(row), br = NEG; int cur = 0;
        for (int j = 1; j < K; j++) {
            const T v = bt_ld(row + (size_t)j * NS);
            if (CERT) br = max(br, min(v, bv));            // runner-up: the largest value that is not the first maximum
            if (v > bv) { bv = v; cur = j; }
        }
        if (CERT) ok = ok && (!(bv > NEG) || cert_pass(bv, br, len - 1, p.cert_tol));
        else if (p.score) p.score[b] = (double)bv;
        store_path_at(p, off + len - 1, (uint32_t)cur);
        if (len == 1) {
            if (CERT) cert_finish();
            return my_chunk;
        }

        // walk back (viterbi.rs:27-30): steps tt = len-1 .. 1, each a scan of row tt-1 in chunks of BT_CHUNK predecessors;
        // the next chunk (of this step, or the first of the next step -- rows do not depend on the path) is always
        // in flight while the current one is reduced.  Pointers advance by constants: no division in the loop.
        T dcur = bv;                                          // delta[tt][cur]
        T bufA[BT_CHUNK], bufB[BT_CHUNK];                     // two chunk buffers used alternately: no register copies
        const T *rowp = col + (size_t)(len - 2) * sl;         // row tt-1
        int64_t pout = off + (len - 2);
        auto load_chunk = [&](const T *prow, int c, T (&dst)[BT_CHUNK]) {
            const T *q = prow + (size_t)c * (BT_CHUNK * NS);
            if (c < nfull) {
#pragma unroll
                for (int k = 0; k < BT_CHUNK; k++) dst[k] = bt_ld(q + (size_t)k * NS);
            } else {
#pragma unroll
                for (int k = 0; k < BT_CHUNK; k++) dst[k] = (k < ktail) ? bt_ld(q + (size_t)k * NS) : NEG;
            }
        };
        T mv = 0, rv = NEG; int mi = 0;
        const T *at = sAT;
        // chunk c of the current step: candidates fl(delta[tt-1][j] + logA[j][cur]), first maximum (viterbi.rs:15-16);
        // predecessors >= K hold -inf and can never be strictly greater (logA is read up to BT_CHUNK-1 doubles past
        // K: padded).  CERT: rv = the runner-up (the largest candidate other than the first maximum)
        auto reduce_chunk = [&](const T (&cu)[BT_CHUNK], int c) {
            const T *ac = at + c * BT_CHUNK;
            if (c == 0) {
                mv = cu[0] + ac[0]; mi = 0;
                if (CERT) rv = NEG;
#pragma unroll
                for (int k = 1; k < BT_CHUNK; k++) {
                    const T v = cu[k] + ac[k];
                    if (CERT) rv = max(rv, min(v, mv));
                    if (v > mv) { mv = v; mi = k; }
                }
            } else {
                const int j0 = c * BT_CHUNK;
#pragma unroll
                for (int k = 0; k < BT_CHUNK; k++) {
                    const T v = cu[k] + ac[k];
                    if (CERT) rv = max(rv, min(v, mv));
                    if (v > mv) { mv = v; mi = j0 + k; }
                }
            }
        };
        // one step: X holds chunk 0 on entry; the chunk after the one being reduced is always in flight (the next
        // chunk of this step, or chunk 0 of the next step -- rows do not depend on the path)
        auto step = [&](T (&X)[BT_CHUNK], T (&Y)[BT_CHUNK], int tt) {
            at = sAT + (size_t)cur * ATP;
            int c = 0;
            for (; c + 1 < nchunk; c += 2) {
                load_chunk(rowp, c + 1, Y);
                reduce_chunk(X, c);
                if (c + 2 < nchunk) load_chunk(rowp, c + 2, X);
                else if (tt > 1) load_chunk(rowp - sl, 0, X);
                reduce_chunk(Y, c + 1);
            }
            if (c < nchunk) {                                  // odd number of chunks: the next step starts in Y
                if (tt > 1) load_chunk(rowp - sl, 0, Y);
                reduce_chunk(X, c);
            }
            // psi = 0 when delta[tt][cur] = -inf (emission -inf or all candidates -inf; see header comment)
            if (CERT && dcur > NEG) ok = ok && cert_pass(mv, rv, tt, p.cert_tol);
            cur = (dcur > NEG) ? mi : 0;
            dcur = __ldcg(rowp + (size_t)cur * NS);              // delta[tt-1][cur]
            store_path_at(p, pout, (uint32_t)cur);
            pout--; rowp -= sl;
        };
        load_chunk(rowp, 0, bufA);
        if (nchunk & 1) {
            int tt = len - 1;
            for (; tt >= 2; tt -= 2) { step(bufA, bufB, tt); step(bufB, bufA, tt - 1); }
            if (tt >= 1) step(bufA, bufB, tt);
        } else {
            for (int tt = len - 1; tt >= 1; tt--) step(bufA, bufB, tt);
        }
        if (CERT) cert_finish();
        return my_chunk;
        }();
        bt_mark_done_warp(p, done_chunk);
    }
}

// ---------------------------------------------------------------------------
// The same end state + backtrace with FOUR lanes per sequence (f64).
//
// One thread per sequence is bound by memory latency: a lane has one chunk of 8 predecessors in flight and a step costs
// six dependent round trips (6-10 us per step; 0.41 ms for the 125 k sentences a rank of an 8-GPU run decodes, most of
// it left over when the forward kernel ends).  Here lane (part, sl) of a warp owns the predecessors
// [part * JP, (part + 1) * JP) of sequence sl -- a warp holds 8 sequences, the loads of one predecessor are 64-byte
// runs -- so a whole row is in flight at once (JP loads per lane), the dependent chain of a step is JP compares plus
// two shuffle rounds, and no load depends on the decoded state: the delta value of the winning predecessor (the
// `dcur` of the next step) is carried through the reduction instead of being fetched.  The first maximum survives the
// cross-lane combine because parts are ordered by predecessor index: a later part wins only if strictly greater.
// The end state (viterbi.rs:24) is the same scan against a column of zeros (delta + 0.0 = delta bit for bit: no delta is -0.0).
// ---------------------------------------------------------------------------
template <int JP, int MINB>
__global__ void __launch_bounds__(128, MINB) backtrace_split_kernel(const DecodeSmallParams p)
{
    constexpr int NS = 64, LPS = 4;
    const double NEG = neg_inf();
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int K = p.K, Kp = p.Kp;
    const int ATP = K | 1;                                     // odd pitch: rows of different states spread over banks
    // sAT[s*ATP + j] = logA[j][s]; row K = zeros (+ padding: a part may read up to LPS * JP - K entries past a row's end --
    // whatever it finds there is added to a -inf operand)
    double *sAT = reinterpret_cast<double *>(smem_raw);
    for (int e = threadIdx.x; e < (K + 1) * ATP + LPS * JP; e += blockDim.x) {
        const int s = e / ATP, j = e % ATP;
        sAT[e] = (s >= K || j >= K) ? 0.0 : p.A[(size_t)j * Kp + s];
    }
    __syncthreads();

    const size_t sl = (size_t)K * NS;
    const int lane = threadIdx.x & 31, part = lane >> 3;
    const unsigned int grp_mask = 0x01010101u << (lane & 7);  // the four lanes of this sequence
    const int j0 = part * JP;
    const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
    const int64_t total = (int64_t)p.ntiles * NS * LPS;
    for (int64_t r4 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r4 < total; r4 += nthreads) {
        // warp = 8 adjacent sequences of one tile: sequence index r = (warp index) * 8 + (lane & 7)
        const int64_t r = (r4 >> 5) * 8 + (lane & 7);
        int tile = (int)(r / NS);
        const int s = (int)(r % NS);
        if (p.tile_done) {
            // concurrent mode: queue slot `tile` holds a finished tile (see backtrace_small_kernel)
            int v = 0;
            if (lane == 0) {
                const long long t0 = clock64();
                for (;;) {
                    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p.tile_done + tile) : "memory");
                    if (v) break;
                    if (clock64() - t0 > (1LL << 35)) { *p.status = 5; v = tile + 1; break; }
                    __nanosleep(1000);
                }
            }
            tile = __shfl_sync(0xffffffffu, v, 0) - 1;
            __threadfence();
        }
        const int done_chunk = [&]() -> int {
        const int64_t rr = (int64_t)tile * NS + s;
        if (rr >= p.B) return -1;
        const uint32_t b = p.order[rr];
        if (p.is_long && p.is_long[b]) return -1;
        const int my_chunk = (p.chunk_done && part == 0) ? bt_chunk_of(p, b) : -1;    // one report per sequence
        const int64_t off = p.seq_off[b];
        const int len = (int)(p.seq_off[b + 1] - off);
        if (len <= 0 || p.tile_base[tile] + (long long)len > p.hist_cap_slabs) return my_chunk;
        // this lane's predecessors of row len-1 of sequence s
        const double *rowp = p.hist + (size_t)p.tile_base[tile] * sl + (size_t)(len - 1) * sl + (size_t)j0 * NS + s;
        double buf[JP];
        auto load_row = [&](const double *q) {
#pragma unroll
            for (int k = 0; k < JP; k++) buf[k] = (j0 + k < K) ? bt_ld(q + (size_t)k * NS) : NEG;
        };
        load_row(rowp);
        const double *at = sAT + (size_t)K * ATP + j0;         // the column of zeros: the end state is a plain argmax
        double dcur = 0.0;
        int64_t pout = off + (len - 1);
        for (int tt = len - 1; tt >= 0; tt--) {
            // candidates fl(delta[tt][j] + logA[j][state(tt+1)]) of this lane's part, first maximum, with the delta operand
            double mv = buf[0] + at[0], md = buf[0];
            int mi = j0;
#pragma unroll
            for (int k = 1; k < JP; k++) {
                const double v = buf[k] + at[k];
                if (v > mv) { mv = v; md = buf[k]; mi = j0 + k; }
            }
            // the row below is path independent: fetch it while the four parts are combined
            if (tt > 0) { rowp -= sl; load_row(rowp); }
#pragma unroll
            for (int d = 8; d <= 16; d <<= 1) {
                const double ov = __shfl_xor_sync(grp_mask, mv, d), od = __shfl_xor_sync(grp_mask, md, d);
                const int oi = __shfl_xor_sync(grp_mask, mi, d);
                // the other lane holds later predecessors iff its index is higher: later wins only if strictly greater
                const bool take = oi > mi ? ov > mv : !(mv > ov);
                if (take) { mv = ov; md = od; mi = oi; }
            }
            // psi = 0 when delta[tt+1][state(tt+1)] = -inf (emission -inf or all candidates -inf; see header comment)
            const int cur = (dcur > NEG) ? mi : 0;
            if (part == 0) {
                if (tt == len - 1 && p.score) p.score[b] = mv;
                store_path_at(p, pout, (uint32_t)cur);
            }
            pout--;
            // delta[tt][cur]: the winning operand, unless the -inf rule replaced the argmax by state 0
            dcur = (cur == mi) ? md : __ldcg(p.hist + (size_t)p.tile_base[tile] * sl + (size_t)tt * sl + (size_t)cur * NS + s);
            at = sAT + (size_t)cur * ATP + j0;
        }
        return my_chunk;
        }();
        bt_mark_done_warp(p, done_chunk);
    }
}

}  // namespace cvb
