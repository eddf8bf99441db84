// decode_f32.cuh -- batched plain Viterbi, OPTIONAL f32 mode (cv_decode_batch_f32 / cv_decode_batch_dev_f32), K <= 64.
//
// BASELINE.json's north_star allows an f32 mode with path log-scores within 1e-5 relative of the f64 reference.
// This is that mode, NOT the parity path: the recurrence of viterbi::decode (src/viterbi_solver/viterbi.rs:5-32) with
// every operand rounded to f32 once (rn32(logA), rn32(logB)) and every add an IEEE binary32 add,
//   delta[t][i] = fl32( max_j fl32(delta[t-1][j] + a[j][i]) + b[i][o_t] ),  -inf emission => -inf, psi = 0,
// first-maximum backpointers recomputed by the backtrace from the f32 history (backtrace_small_kernel<.., float>), so
// the decoded path is the exact optimum of the f32 recurrence; it can differ from the f64 path where two candidates
// are within f32 rounding of each other.
//
// Why it is much faster: a cell is FADD + FMNMX, and sm_100a has packed adds (FADD2, two cells per instruction) and
// 3-input maxima (FMNMX3, two cells per instruction): ~1.2 issue slots per cell instead of 5.  Same mapping as
// decode_small_fwd_kernel (persistent CTAs, tiles of 64 sequences, a lane owns 2 adjacent sequences, a warp one group
// of <= 8 target states of the balanced split, emission rows by TMA, one TMA bulk store of the [K][64] slab per step),
// at half the shared memory (46 KB at K = 45: four CTAs per SM).
//
// MINB = 4 caps the kernel at 64 registers (78 uncapped; the 8 + 24 bytes of spills are in the per-tile prologue and
// epilogue, none in the step loop): then four forward CTAs of six warps (K = 45) and two CTAs of the concurrent
// backtrace share an SM's registers, and the backtrace of a long batch runs beside the forward pass instead of after it.
// The cap costs the kernel ~10 % alone, so short batches run the uncapped build (MINB = 3; launch_decode_small).
//
// The exact decode of an eligible model (cv_hmm_create: every finite entry <= 0 and |x| <= 2^64) runs this kernel as
// well: backtrace_small_kernel<.., float, true> then certifies every backpointer against the f64 recurrence (the
// bound is derived above that kernel) and the sequences it cannot certify are decoded again in f64.
#pragma once

#include "decode_small.cuh"

namespace cvb {

// packed f32 add (FADD2): two cells per instruction
__device__ __forceinline__ float2 fadd2(float2 a, float2 b)
{
    float2 r;
    asm("{ .reg .b64 ra, rb, rc; mov.b64 ra, {%2, %3}; mov.b64 rb, {%4, %5}; add.rn.f32x2 rc, ra, rb; mov.b64 {%0, %1}, rc; }"
        : "=f"(r.x), "=f"(r.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return r;
}

__host__ __device__ inline int f32_em_pitch(int Kp) { return Kp + 4; }   // floats; rows stay 16-byte aligned
__host__ __device__ inline size_t decode_f32_smem_bytes(int K, int Kp)
{
    return (size_t)K * Kp * 4 + (size_t)2 * K * 64 * 4 + (size_t)64 * f32_em_pitch(Kp) * 4 + 64 * (8 + 4) + 32 + 16;
}

template <int MINB>
__global__ void __launch_bounds__(256, MINB) decode_f32_fwd_kernel(const DecodeSmallParams p)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int NS = 64;
    const float NEGF = __int_as_float(0xff800000);
    const int K = p.K, Kp = p.Kp, EP = f32_em_pitch(Kp);
    float *sA = reinterpret_cast<float *>(smem_raw);                // [K][Kp] slot-permuted columns
    float *sD = sA + (size_t)K * Kp;                                // [2][K][64]
    float *sEm = sD + (size_t)2 * K * NS;                           // [64][EP]
    int64_t *sOff = reinterpret_cast<int64_t *>(sEm + (size_t)NS * EP);
    int *sLen = reinterpret_cast<int *>(sOff + NS);
    uint64_t *sBar = reinterpret_cast<uint64_t *>(sLen + NS);
    int *sTile = reinterpret_cast<int *>(sBar + 4);

    const int tid = threadIdx.x, lane = tid & 31, g = tid >> 5;
    const int nw = (int)blockDim.x >> 5;
    const int c0 = g * 8;
    const int srow0 = p.nq_base ? g * p.nq_base + min(g, p.nq_rem) : c0;
    const int nreal = p.nq_base ? p.nq_base + (g < p.nq_rem ? 1 : 0) : max(0, min(8, K - c0));
    const int s0 = 2 * lane;
    const uint32_t slab_bytes = (uint32_t)((size_t)K * NS * 4);
    const uint32_t row_bytes = (uint32_t)(Kp * 4);
    constexpr int EMK = 4;

    if (tid == 0) {
        if (p.started) atomicAdd(p.started, 1u);
        mbar_init(sBar, 1);
        mbar_init(sBar + 1, nw);
        fence_proxy_async_smem();
        const uint32_t bytes = (uint32_t)((size_t)K * Kp * 4);
        mbar_expect_tx(sBar, bytes);
        tma_bulk_g2s(sA, p.A32s, bytes, sBar);
    }
    __syncthreads();
    mbar_wait(sBar, 0);
    uint32_t em_phase = 0;

    const bool obs_streamed = p.arrived != nullptr;
    auto ld_obs = [&](int64_t idx) -> uint32_t { return load_obs_at(p, idx, obs_streamed); };
    auto issue_emissions = [&](int t, const uint32_t (&o_cur)[EMK]) {
        int nact = 0;
#pragma unroll
        for (int k = 0; k < EMK; k++) {
            const int s = g + nw * (lane + 32 * k);
            if (s < NS && t < sLen[s]) nact++;
        }
        const int total = __reduce_add_sync(0xffffffffu, nact);
        if (lane == 0) mbar_expect_tx(sBar + 1, (uint32_t)total * row_bytes);
        __syncwarp();
#pragma unroll
        for (int k = 0; k < EMK; k++) {
            const int s = g + nw * (lane + 32 * k);
            if (s < NS && t < sLen[s]) {
                uint32_t o = o_cur[k];
                if ((int64_t)o >= p.M) { *p.status = 3; o = 0; }
                tma_bulk_g2s(sEm + (size_t)s * EP, p.BT32 + (size_t)o * Kp, row_bytes, sBar + 1);
            }
        }
    };

    for (;;) {
        if (tid == 0) *sTile = (int)atomicAdd(p.tile_counter, 1u);
        __syncthreads();
        const int tile = *sTile;
        if (tile >= p.ntiles) break;

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
        for (int e = tid; e < K * NS; e += blockDim.x) sD[e] = 0.0f;          // delta(0) = 0 (viterbi.rs:6)
        if (p.arrived && tid == 0) {
            const unsigned int need = (unsigned int)p.tile_chunk[tile] + 1u;
            const long long t0 = clock64();
            for (;;) {
                unsigned int v;
                asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p.arrived) : "memory");
                if (v >= need) break;
                if (clock64() - t0 > (1LL << 32)) { *p.status = 5; break; }
                __nanosleep(128);
            }
        }
        fence_proxy_async_smem();
        __syncthreads();

        int Tmax = p.tile_tmax ? (int)p.tile_tmax[tile] : sLen[0];
        if (p.tile_base[tile] + (long long)Tmax > p.hist_cap_slabs) {
            if (tid == 0) atomicMax(p.status, 7);
            Tmax = 0;
        }
        float *slab = reinterpret_cast<float *>(p.hist) + (size_t)p.tile_base[tile] * K * NS;
        if (tid == 0 && Tmax > 0) tma_bulk_s2g(slab, sD, slab_bytes);

        uint32_t o_nxt[EMK];
        {
            uint32_t o1[EMK];
#pragma unroll
            for (int k = 0; k < EMK; k++) {
                const int s = g + nw * (lane + 32 * k);
                const bool in = s < NS;
                o1[k] = (in && 1 < sLen[s]) ? ld_obs(sOff[s] + 1) : 0u;
                o_nxt[k] = (in && 2 < sLen[s]) ? ld_obs(sOff[s] + 2) : 0u;
            }
            if (Tmax > 1) issue_emissions(1, o1);
        }

        for (int t = 1; t < Tmax; t++) {
            const float *dcur = sD + (size_t)((t - 1) & 1) * K * NS + s0;
            const float *arow = sA + c0;
            float best[2][8];
#pragma unroll
            for (int pp = 0; pp < 2; pp++)
#pragma unroll
                for (int q = 0; q < 8; q++) best[pp][q] = NEGF;
            // two predecessors per iteration: 16 packed adds + 16 three-input maxima for 32 cells
            int j = 0;
#pragma unroll 2
            for (; j + 1 < K; j += 2) {
                float y[2][2][8];
#pragma unroll
                for (int u = 0; u < 2; u++) {
                    const float2 d = *reinterpret_cast<const float2 *>(dcur + (size_t)(j + u) * NS);
                    const float4 a0 = *reinterpret_cast<const float4 *>(arow + (size_t)(j + u) * Kp);
                    const float4 a1 = *reinterpret_cast<const float4 *>(arow + (size_t)(j + u) * Kp + 4);
                    const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
                    for (int pp = 0; pp < 2; pp++) {
                        const float dp = pp ? d.y : d.x;
#pragma unroll
                        for (int q = 0; q < 8; q += 2) {
                            const float2 v = fadd2(make_float2(dp, dp), make_float2(a[q], a[q + 1]));
                            y[u][pp][q] = v.x; y[u][pp][q + 1] = v.y;
                        }
                    }
                }
#pragma unroll
                for (int pp = 0; pp < 2; pp++)
#pragma unroll
                    for (int q = 0; q < 8; q++) best[pp][q] = fmaxf(fmaxf(best[pp][q], y[0][pp][q]), y[1][pp][q]);
            }
            if (j < K) {                                                      // odd K: the last predecessor
                const float2 d = *reinterpret_cast<const float2 *>(dcur + (size_t)j * NS);
                const float4 a0 = *reinterpret_cast<const float4 *>(arow + (size_t)j * Kp);
                const float4 a1 = *reinterpret_cast<const float4 *>(arow + (size_t)j * Kp + 4);
                const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
                for (int q = 0; q < 8; q++) {
                    best[0][q] = fmaxf(best[0][q], d.x + a[q]);
                    best[1][q] = fmaxf(best[1][q], d.y + a[q]);
                }
            }
            mbar_wait(sBar + 1, em_phase);
            em_phase ^= 1;
            {
                float *dnext = sD + (size_t)(t & 1) * K * NS + s0;
                const float *e0 = sEm + (size_t)s0 * EP + c0, *e1 = e0 + EP;
                const float4 x00 = *reinterpret_cast<const float4 *>(e0), x01 = *reinterpret_cast<const float4 *>(e0 + 4);
                const float4 x10 = *reinterpret_cast<const float4 *>(e1), x11 = *reinterpret_cast<const float4 *>(e1 + 4);
                const float b0[8] = {x00.x, x00.y, x00.z, x00.w, x01.x, x01.y, x01.z, x01.w};
                const float b1[8] = {x10.x, x10.y, x10.z, x10.w, x11.x, x11.y, x11.z, x11.w};
#pragma unroll
                for (int q = 0; q < 8; q++)
                    if (q < nreal)
                        *reinterpret_cast<float2 *>(dnext + (size_t)(srow0 + q) * NS) = make_float2(best[0][q] + b0[q], best[1][q] + b1[q]);
            }
            fence_proxy_async_smem();
            if (tid == 0) tma_store_wait_read_all();
            __syncthreads();
            if (tid == 0) tma_bulk_s2g(slab + (size_t)t * K * NS, sD + (size_t)(t & 1) * K * NS, slab_bytes);
            if (t + 1 < Tmax) {
                issue_emissions(t + 1, o_nxt);
#pragma unroll
                for (int k = 0; k < EMK; k++) {
                    const int s = g + nw * (lane + 32 * k);
                    o_nxt[k] = (s < NS && t + 2 < sLen[s]) ? ld_obs(sOff[s] + t + 2) : 0u;
                }
            }
        }
        if (tid == 0) {
            if (p.tile_done) {
                tma_store_wait_all();
                asm volatile("fence.proxy.async;" ::: "memory");
                __threadfence();
                const unsigned int slot = atomicAdd(p.started + 1, 1u);
                asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p.tile_done + slot), "r"(tile + 1) : "memory");
            } else {
                tma_store_wait_read_all();
            }
        }
        __syncthreads();
    }
}

}  // namespace cvb
