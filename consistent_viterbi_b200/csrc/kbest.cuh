// kbest.cuh -- exact k-best (list) Viterbi, cv_decode_batch_kbest (include/cv_b200.h): ONE WARP PER SEQUENCE.
//
// The list L[t][i] holds the min(k, K^t) best prefixes ending in state i at step t, ordered (c descending, j ascending,
// r ascending) with c = fl(L[t-1][j][r] + a[j][i]); its values are fl(c + b[i][o_t]).  Lane i (and i + 32 when
// K > 32) builds the list of state i in registers by stable insertion while it walks the predecessors j ascending and
// each predecessor's sorted list r ascending.  A predecessor's walk stops at the first candidate that does not beat
// the current k-th entry: fl(x + a) is monotone, so every later entry of that list is no larger and loses the tie
// order as well.  The previous row [Kp][KC] f64 sits in per-warp shared memory, double-buffered; logA is in shared
// memory, emissions are read from the handle's logB^T.  Backpointers (j << 5 | r) go to HBM as u16 rows [Kp][KC]
// per position, written by every lane as vector stores of its own KC slots.  The end selection merges the K lists
// with k rounds of a warp argmax keyed (value, state); lane r then follows rank r back through the backpointers.
#pragma once

#include "chain_warp.cuh"

namespace cvb {

constexpr int KB_K_MAX = 32;        // ranks per sequence: one lane of the backtrace per rank
constexpr int KB_WARPS_MAX = 8;     // warps (sequences in flight) per block

struct KbestParams {
    const double *A;          // [K][Kp]
    const double *BT;         // [M][Kp]
    const uint32_t *obs;      // [N] the chunk's observations
    const int64_t *seq_off;   // [B+1] chunk-local offsets, seq_off[0] = 0
    const uint32_t *order;    // [B] longest first
    uint16_t *bp;             // [N][Kp][KC] backpointers of position x (row 0 of a sequence is not written)
    uint32_t *path;           // [k][N] rank-major planes
    double *score;            // [k][B]
    unsigned int *counter;    // sequences taken
    int64_t B, N;
    int K, Kp, k;
};

// Register list of capacity KC holding the k entries of one state in slots KC-k .. KC-1 (slot KC-1 is the k-th
// entry); slots below KC-k hold +inf and never move.  A free slot holds NaN, which `!(x >= c)` orders below every
// candidate, so the first k candidates always enter and a full list admits c only when c beats its k-th entry.
// The new entry goes behind every entry that is >= c: stable in the candidate order.
template <int KC>
__device__ __forceinline__ void kb_insert(double (&v)[KC], uint32_t (&q)[KC], double c, uint32_t bp)
{
#pragma unroll
    for (int s = KC - 1; s >= 1; s--) {
        const bool below_prev = !(v[s - 1] >= c), below = !(v[s] >= c);
        v[s] = below_prev ? v[s - 1] : (below ? c : v[s]);
        q[s] = below_prev ? q[s - 1] : (below ? bp : q[s]);
    }
    if (!(v[0] >= c)) { v[0] = c; q[0] = bp; }
}

template <int KC>
__device__ __forceinline__ void kb_store_bp(uint16_t *dst, const uint32_t (&q)[KC])
{
    if constexpr (KC == 1) {
        dst[0] = (uint16_t)q[0];
    } else if constexpr (KC == 2) {
        *reinterpret_cast<uint32_t *>(dst) = q[0] | q[1] << 16;
    } else if constexpr (KC == 4) {
        *reinterpret_cast<uint2 *>(dst) = make_uint2(q[0] | q[1] << 16, q[2] | q[3] << 16);
    } else {
#pragma unroll
        for (int g = 0; g < KC / 8; g++)
            reinterpret_cast<uint4 *>(dst)[g] = make_uint4(q[8 * g] | q[8 * g + 1] << 16, q[8 * g + 2] | q[8 * g + 3] << 16,
                                                           q[8 * g + 4] | q[8 * g + 5] << 16, q[8 * g + 6] | q[8 * g + 7] << 16);
    }
}

__host__ __device__ constexpr size_t kbest_smem_bytes(int K, int Kp, int KC, int warps)
{
    return (size_t)K * Kp * 8 + (size_t)warps * 2 * Kp * KC * 8;
}

// register cap per instantiation: ptxas left to itself spills at KC = 8 (64 registers); the list takes 3 KC of them
constexpr int kb_max_regs(int KC) { return KC <= 4 ? 64 : KC == 8 ? 96 : KC == 16 ? 160 : 255; }

// KC = list capacity (1, 2, 4, 8, 16, 32), k <= KC ranks
template <int KC>
__global__ void __launch_bounds__(32 * KB_WARPS_MAX) __maxnreg__(kb_max_regs(KC)) kbest_kernel(const KbestParams p)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int K = p.K, Kp = p.Kp, k = p.k, pad = KC - k;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    double *sA = reinterpret_cast<double *>(smem_raw);
    double *rows = sA + (size_t)K * Kp + (size_t)w * 2 * Kp * KC;      // this warp's rows [2][Kp][KC], entry r at [i][r]
    for (int e = threadIdx.x; e < K * Kp; e += blockDim.x) sA[e] = p.A[e];
    __syncthreads();
    const int nsl = K > 32 ? 2 : 1;
    const double pos_inf = __longlong_as_double(0x7ff0000000000000LL), nan = __longlong_as_double(0x7ff8000000000000LL);

    for (;;) {
        unsigned int sq = 0;
        if (lane == 0) sq = atomicAdd(p.counter, 1u);
        sq = __shfl_sync(0xffffffffu, sq, 0);
        if ((int64_t)sq >= p.B) break;
        const uint32_t b = p.order[sq];
        const int64_t off = p.seq_off[b];
        const int len = (int)(p.seq_off[b + 1] - off);

        for (int s = 0; s < nsl; s++)
            if (lane + 32 * s < K) rows[(lane + 32 * s) * KC] = 0.0;          // t = 0: one entry per state, 0.0
        __syncwarp();
        int n = 1;                                                              // entries per state in row t-1
        for (int t = 1; t < len; t++) {
            const double *prev = rows + ((t - 1) & 1) * Kp * KC;
            double *cur = rows + (t & 1) * Kp * KC;
            const int ncur = min(k, n * K);
            const uint32_t o = __ldg(p.obs + off + t);
            uint16_t *bprow = p.bp + (size_t)(off + t) * Kp * KC;
#pragma unroll 1
            for (int s = 0; s < nsl; s++) {
                const int i = lane + 32 * s;
                if (i >= K) continue;
                const double e = __ldg(p.BT + (size_t)o * Kp + i);
                double v[KC];
                uint32_t q[KC];
#pragma unroll
                for (int x = 0; x < KC; x++) { v[x] = x < pad ? pos_inf : nan; q[x] = 0; }
                if (e > neg_inf()) {
                    for (int j = 0; j < K; j++) {
                        const double a = sA[j * Kp + i];
                        const double *lj = prev + j * KC;
                        for (int r = 0; r < n; r++) {
                            const double c = lj[r] + a;
                            if (v[KC - 1] >= c) break;                          // the rest of list j loses too
                            kb_insert(v, q, c, (uint32_t)(j << 5 | r));
                        }
                    }
#pragma unroll
                    for (int x = 0; x < KC; x++) v[x] = v[x] + e;
                } else {
                    // the state cannot emit o_t: the first candidates in (j, r) order, every value -inf (R1's psi = 0)
#pragma unroll
                    for (int x = 0; x < KC; x++) {
                        const int r = max(x - pad, 0);
                        q[x] = (uint32_t)((r / n) << 5 | (r % n));
                        v[x] = neg_inf();
                    }
                }
#pragma unroll
                for (int x = 0; x < KC; x++)
                    if (x >= pad && x - pad < ncur) cur[i * KC + x - pad] = v[x];
                kb_store_bp<KC>(bprow + (size_t)i * KC, q);
            }
            n = ncur;
            __syncwarp();
        }

        // end selection: k rounds of a warp argmax over the list heads, (value descending, state ascending); within a
        // state the list order is already (value descending, r ascending)
        const double *last = rows + ((len - 1) & 1) * Kp * KC;
        const int nr = min(k, n * K);
        int head0 = 0, head1 = 0, my_i = 0, my_r = 0;
        double my_v = neg_inf();
        for (int rk = 0; rk < nr; rk++) {
            double bv = neg_inf();
            int bi = 0x7fffffff;
            if (lane < K && head0 < n) { bv = last[lane * KC + head0]; bi = lane; }
            if (lane + 32 < K && head1 < n) {
                const double x = last[(lane + 32) * KC + head1];
                if (bi == 0x7fffffff || x > bv) { bv = x; bi = lane + 32; }
            }
            warp_argmax(bv, bi);
            const int hr = __shfl_sync(0xffffffffu, bi >= 32 ? head1 : head0, bi & 31);
            if (lane == (bi & 31)) { if (bi >= 32) head1++; else head0++; }
            if (lane == rk) { my_i = bi; my_r = hr; my_v = bv; }
        }
        // backtrace: lane r follows rank r; ranks beyond the paths that exist are "no path"
        if (lane < k) {
            uint32_t *pl = p.path + (size_t)lane * p.N + off;
            if (lane < nr) {
                p.score[(size_t)lane * p.B + b] = my_v;
                int i = my_i, r = my_r;
                pl[len - 1] = (uint32_t)i;
                for (int t = len - 1; t >= 1; t--) {
                    const uint32_t x = p.bp[(size_t)(off + t) * Kp * KC + i * KC + pad + r];
                    i = (int)(x >> 5); r = (int)(x & 31);
                    pl[t - 1] = (uint32_t)i;
                }
            } else {
                p.score[(size_t)lane * p.B + b] = neg_inf();
                for (int t = 0; t < len; t++) pl[t] = 0xffffffffu;
            }
        }
        __syncwarp();                                                           // rows are reused by the next sequence
    }
}

}  // namespace cvb
