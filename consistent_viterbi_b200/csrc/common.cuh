// common.cuh -- shared device helpers for the consistent-viterbi B200 kernels.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace cvb {

constexpr int TQ = 8;   // target states per thread (operand broadcast from smem)
constexpr int TP = 2;   // sequences per thread   (operand per lane, one LDS.128)
constexpr int SMALL_K_MAX = 64;   // K above this uses the tiled (large-K) kernel
constexpr int LARGE_BN = 128;     // target states per work item of the large-K kernel

__device__ __forceinline__ double neg_inf() { return __longlong_as_double(0xfff0000000000000LL); }

// HMM::log (hmm.rs:192-205) of one probability: 0 -> -inf, else x.log(10.0) = ln(x) / ln(10).  Used by cv_mle on the
// host and by the Baum-Welch M-step on the device.
__host__ __device__ inline double hmm_log10(double x) { return x == 0.0 ? -INFINITY : log(x) / log(10.0); }

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
