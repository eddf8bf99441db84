// probe.cuh -- FP64 issue-rate micro-benchmark (roofline denominator, cv_debug_probe_fp64).
#pragma once

#include "common.cuh"

namespace cvb {

// MODE 0: independent DADD chains; 1: DADD + DSETP (predicate OR-chained, no selects); 2: independent DFMA chains
template <int MODE>
__global__ void __launch_bounds__(512, 1) probe_fp64_kernel(double *out, int iters, double seed)
{
    constexpr int NCH = 16;
    double acc[NCH];
    bool pr = false;
#pragma unroll
    for (int c = 0; c < NCH; c++) acc[c] = seed * (threadIdx.x + c);
    const double inc = seed * 1e-3;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int c = 0; c < NCH; c++) {
            if constexpr (MODE == 0) {
                acc[c] += inc;
            } else if constexpr (MODE == 2) {
                acc[c] = fma(acc[c], seed, inc);          // DFMA (seed = 1.0 at run time: the compiler cannot fold it)
            } else {
                acc[c] += inc;
                pr = pr || (acc[c] > seed);
            }
        }
    }
    double s = 0.0;
#pragma unroll
    for (int c = 0; c < NCH; c++) s += acc[c];
    if (s == 12345.678 || (pr && seed == -1.0)) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

}  // namespace cvb
