// common.cuh -- shared device helpers for the consistent-viterbi B200 kernels.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace cvb {

constexpr int TQ = 8;   // target states per thread (operand broadcast from smem)
constexpr int TP = 2;   // sequences per thread   (operand per lane, one LDS.128)
constexpr int SEQ_PER_WARP = 32 * TP;
constexpr int SMALL_K_MAX = 64;   // K above this uses the tiled (large-K) kernel
constexpr int LARGE_BN = 128;     // target states per work item of the large-K kernel

__device__ __forceinline__ double neg_inf() { return __longlong_as_double(0xfff0000000000000LL); }

// HMM::log (hmm.rs:192-205) of one probability: 0 -> -inf, else x.log(10.0) = ln(x) / ln(10).  Used by cv_mle on the
// host and by the Baum-Welch M-step on the device.
__host__ __device__ inline double hmm_log10(double x) { return x == 0.0 ? -INFINITY : log(x) / log(10.0); }

// ---------------------------------------------------------------------------
// One max-plus cell: v = d + a; if (v > best) { best = v; idx = j; }
//
// The update is the reference's ndarray-stats argmax rule (first element that is
// strictly greater than the running maximum wins, viterbi.rs:16 / cp.rs:53)
// because predecessors are visited in ascending j.
//
// sm_100a has no 64-bit select and no DMNMX, so a cell is
//   DADD + DSETP (FP64 pipe) + 2 x 32-bit select (value) + 1 x select (index),
// and SEL/FSEL issue on the ALU pipe only.  VARIANT 1-3 were attempts to move selects onto the FMA pipe as
// predicated IMADs; ptxas turns every predicated move back into op + SEL (checked in SASS, even at -O0), so they
// compile to the same select count and are kept only for the probe (cv_debug_probe_fp64 modes 3-5).  The production
// kernels use VARIANT 0 where the index is part of the state (constrained decode) and the value-only tile of
// decode_small.cuh / decode_large.cuh otherwise.
// ---------------------------------------------------------------------------
template <int VARIANT>
__device__ __forceinline__ void cell(double d, double a, double &best, int &idx, int j, int zero)
{
    if constexpr (VARIANT == 0) {
        (void)zero;
        double v = d + a;
        if (v > best) { best = v; idx = j; }
    } else if constexpr (VARIANT == 1) {
        asm("{\n\t.reg .pred p;\n\t.reg .f64 v;\n\t"
            "add.rn.f64 v, %2, %3;\n\t"
            "setp.gt.f64 p, v, %0;\n\t"
            "selp.f64 %0, v, %0, p;\n\t"
            "@p mad.lo.s32 %1, %4, %4, %5;\n\t}"
            : "+d"(best), "+r"(idx) : "d"(d), "d"(a), "r"(zero), "r"(j));
    } else if constexpr (VARIANT == 2) {
        asm("{\n\t.reg .pred p;\n\t.reg .f64 v;\n\t.reg .b32 vl, vh, bl, bh;\n\t"
            "add.rn.f64 v, %2, %3;\n\t"
            "setp.gt.f64 p, v, %0;\n\t"
            "mov.b64 {vl, vh}, v;\n\t"
            "mov.b64 {bl, bh}, %0;\n\t"
            "selp.b32 bl, vl, bl, p;\n\t"
            "@p mad.lo.u32 bh, %4, %4, vh;\n\t"
            "mov.b64 %0, {bl, bh};\n\t"
            "@p mad.lo.s32 %1, %4, %4, %5;\n\t}"
            : "+d"(best), "+r"(idx) : "d"(d), "d"(a), "r"(zero), "r"(j));
    } else {
        asm("{\n\t.reg .pred p;\n\t.reg .f64 v;\n\t.reg .b32 vl, vh, bl, bh;\n\t"
            "add.rn.f64 v, %2, %3;\n\t"
            "setp.gt.f64 p, v, %0;\n\t"
            "mov.b64 {vl, vh}, v;\n\t"
            "mov.b64 {bl, bh}, %0;\n\t"
            "@p mad.lo.u32 bl, %4, %4, vl;\n\t"
            "@p mad.lo.u32 bh, %4, %4, vh;\n\t"
            "mov.b64 %0, {bl, bh};\n\t"
            "@p mad.lo.s32 %1, %4, %4, %5;\n\t}"
            : "+d"(best), "+r"(idx) : "d"(d), "d"(a), "r"(zero), "r"(j));
    }
}

#ifndef CVB_CELL_VARIANT
#define CVB_CELL_VARIANT 0
#endif

// ---------------------------------------------------------------------------
// TP x TQ register micro-tile over all predecessors j in [0, K):
//   best[p][q], idx[p][q] <- first-max_j ( dcol[j*ldd + p] + arow[j*lda + q] )
// dcol points at this lane's TP adjacent sequences (16-byte aligned),
// arow at this warp's TQ adjacent target states (64-byte aligned, uniform).
// ---------------------------------------------------------------------------
template <int VARIANT>
__device__ __forceinline__ void maxplus_tile(const double *__restrict__ dcol, int ldd,
                                             const double *__restrict__ arow, int lda, int K,
                                             double (&best)[TP][TQ], int (&idx)[TP][TQ], int zero)
{
#pragma unroll
    for (int p = 0; p < TP; p++)
#pragma unroll
        for (int q = 0; q < TQ; q++) { best[p][q] = neg_inf(); idx[p][q] = 0; }

#pragma unroll 2
    for (int j = 0; j < K; j++) {
        const double2 d = *reinterpret_cast<const double2 *>(dcol + (size_t)j * ldd);
        const double2 a01 = *reinterpret_cast<const double2 *>(arow + (size_t)j * lda);
        const double2 a23 = *reinterpret_cast<const double2 *>(arow + (size_t)j * lda + 2);
        const double2 a45 = *reinterpret_cast<const double2 *>(arow + (size_t)j * lda + 4);
        const double2 a67 = *reinterpret_cast<const double2 *>(arow + (size_t)j * lda + 6);
        const double a[TQ] = {a01.x, a01.y, a23.x, a23.y, a45.x, a45.y, a67.x, a67.y};
        const double dd[TP] = {d.x, d.y};
#pragma unroll
        for (int p = 0; p < TP; p++)
#pragma unroll
            for (int q = 0; q < TQ; q++) cell<VARIANT>(dd[p], a[q], best[p][q], idx[p][q], j, zero);
    }
}

// ---- TMA 1-D bulk copy global -> shared, completion on an mbarrier ----------
__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}
// bytes must be a multiple of 16; src/dst 16-byte aligned.
__device__ __forceinline__ void tma_bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

}  // namespace cvb
