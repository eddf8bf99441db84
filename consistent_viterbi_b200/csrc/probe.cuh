// probe.cuh -- FP64 issue-rate micro-benchmarks (roofline denominator) and the
// decode inner loop run in isolation with each select-placement variant.
#pragma once

#include "common.cuh"
#include "decode_small.cuh"

namespace cvb {

// (probe only) Software-pipelined variant: the adds of predecessor j+1 are issued next to the compare/selects of j, so the
// FP64 adds never wait behind a batch of selects in the in-order issue stream.
template <int TQT, int TPT = TP>
__device__ __forceinline__ void maxplus_tile_val_pipe(const double *__restrict__ dcol, int ldd,
                                                      const double *__restrict__ arow, int lda, int nj,
                                                      double (&best)[TPT][TQT])
{
    double v[TPT][TQT];
    auto load_add = [&](int j, double (&out)[TPT][TQT]) {
        double dd[TPT], a[TQT];
#pragma unroll
        for (int p = 0; p < TPT / 2; p++) {
            const double2 d = *reinterpret_cast<const double2 *>(dcol + (size_t)j * ldd + 2 * p);
            dd[2 * p] = d.x; dd[2 * p + 1] = d.y;
        }
#pragma unroll
        for (int q = 0; q < TQT / 2; q++) {
            const double2 aa = *reinterpret_cast<const double2 *>(arow + (size_t)j * lda + 2 * q);
            a[2 * q] = aa.x; a[2 * q + 1] = aa.y;
        }
#pragma unroll
        for (int p = 0; p < TPT; p++)
#pragma unroll
            for (int q = 0; q < TQT; q++) out[p][q] = dd[p] + a[q];
    };
    load_add(0, v);
#pragma unroll 2
    for (int j = 1; j < nj; j++) {
        double vn[TPT][TQT];
        load_add(j, vn);
#pragma unroll
        for (int p = 0; p < TPT; p++)
#pragma unroll
            for (int q = 0; q < TQT; q++) {
                best[p][q] = v[p][q] > best[p][q] ? v[p][q] : best[p][q];
                v[p][q] = vn[p][q];
            }
    }
#pragma unroll
    for (int p = 0; p < TPT; p++)
#pragma unroll
        for (int q = 0; q < TQT; q++) best[p][q] = v[p][q] > best[p][q] ? v[p][q] : best[p][q];
}


// mode 0: independent DADD chains; mode 1: DADD + DSETP (predicate OR-chained, no selects)
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

// The real micro-tile on synthetic shared-memory operands (K predecessors, `iters` steps).
template <int VARIANT>
__global__ void __launch_bounds__(512, 1) probe_tile_kernel(double *out, int K, int iters, int zero, double seed)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int Kp = ((K + 7) / 8) * 8;
    const int G = Kp / 8;
    const int NS = ((blockDim.x / 32 + G - 1) / G) * SEQ_PER_WARP;   // warps = G state groups x sequence groups
    double *sA = reinterpret_cast<double *>(smem_raw);
    double *sD = sA + (size_t)K * Kp;
    for (int e = threadIdx.x; e < K * Kp; e += blockDim.x) sA[e] = -seed * ((e * 37) % 101);
    for (int e = threadIdx.x; e < K * NS; e += blockDim.x) sD[e] = -seed * ((e * 53) % 89);
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int i0 = (w % G) * TQ;
    const int s0 = (w / G) * SEQ_PER_WARP + lane * TP;
    double tot = 0.0; int ti = 0;
    for (int it = 0; it < iters; it++) {
        double best[TP][TQ]; int idx[TP][TQ];
        maxplus_tile<VARIANT>(sD + s0, NS, sA + i0, Kp, K, best, idx, zero);
#pragma unroll
        for (int p = 0; p < TP; p++)
#pragma unroll
            for (int q = 0; q < TQ; q++) { tot += best[p][q]; ti += idx[p][q]; }
        // perturb one operand so iterations are not hoisted
        if (i0 == 0) sD[(size_t)(it % K) * NS + s0] = tot * 1e-30;
    }
    if (tot == 12345.678 || ti == -7) out[blockIdx.x * blockDim.x + threadIdx.x] = tot + ti;
}


// value-only micro-tile (the forward kernel's inner loop) in isolation
template <int UNR>
__global__ void __launch_bounds__(512, 1) probe_tile_val_kernel(double *out, int K, int iters, double seed)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int Kp = ((K + 7) / 8) * 8;
    const int G = Kp / 8;
    const int NS = ((blockDim.x / 32 + G - 1) / G) * SEQ_PER_WARP;
    double *sA = reinterpret_cast<double *>(smem_raw);
    double *sD = sA + (size_t)K * Kp;
    for (int e = threadIdx.x; e < K * Kp; e += blockDim.x) sA[e] = -seed * ((e * 37) % 101);
    for (int e = threadIdx.x; e < K * NS; e += blockDim.x) sD[e] = -seed * ((e * 53) % 89);
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int i0 = (w % G) * TQ;
    const int s0 = (w / G) * SEQ_PER_WARP + lane * TP;
    double tot = 0.0;
    for (int it = 0; it < iters; it++) {
        double best[TP][TQ];
#pragma unroll
        for (int p = 0; p < TP; p++)
#pragma unroll
            for (int q = 0; q < TQ; q++) best[p][q] = neg_inf();
        if (UNR == 0) maxplus_tile_val_pipe<TQ, TP>(sD + s0, NS, sA + i0, Kp, K, best);
        else maxplus_tile_val<TQ, (UNR > 0 ? UNR : 2), TP>(sD + s0, NS, sA + i0, Kp, K, best);
#pragma unroll
        for (int p = 0; p < TP; p++)
#pragma unroll
            for (int q = 0; q < TQ; q++) tot += best[p][q];
        if (i0 == 0) sD[(size_t)(it % K) * NS + s0] = tot * 1e-30;
    }
    if (tot == 12345.678) out[blockIdx.x * blockDim.x + threadIdx.x] = tot;
}


// value-only micro-tile with operands in REGISTERS (no shared loads): compute-only ceiling of the inner loop
__global__ void __launch_bounds__(512, 1) probe_tile_val_reg_kernel(double *out, int K, int iters, double seed)
{
    double a[TQ], d[TP];
#pragma unroll
    for (int q = 0; q < TQ; q++) a[q] = -seed * ((threadIdx.x * 7 + q * 3) % 11);
#pragma unroll
    for (int p = 0; p < TP; p++) d[p] = -seed * ((threadIdx.x * 5 + p) % 13);
    double tot = 0.0;
    for (int it = 0; it < iters; it++) {
        double best[TP][TQ];
#pragma unroll
        for (int p = 0; p < TP; p++)
#pragma unroll
            for (int q = 0; q < TQ; q++) best[p][q] = neg_inf();
#pragma unroll 2
        for (int j = 0; j < K; j++) {
#pragma unroll
            for (int p = 0; p < TP; p++)
#pragma unroll
                for (int q = 0; q < TQ; q++) {
                    const double v = d[p] + a[q];
                    best[p][q] = v > best[p][q] ? v : best[p][q];
                }
#pragma unroll
            for (int q = 0; q < TQ; q++) a[q] = a[q] * 1.0000001;     // keep the adds from being hoisted (8 DMUL per 16 cells)
        }
#pragma unroll
        for (int p = 0; p < TP; p++)
#pragma unroll
            for (int q = 0; q < TQ; q++) tot += best[p][q];
    }
    if (tot == 12345.678) out[blockIdx.x * blockDim.x + threadIdx.x] = tot;
}


// compute-only ceiling, variants of instruction ordering (VAR 0: as the kernel; 1: adds of predecessor j+1 issued
// before the compare/selects of j (explicit software pipelining); 2: unroll 4)
template <int VAR>
__global__ void __launch_bounds__(512, 1) probe_tile_val_var_kernel(double *out, int K, int iters, double seed)
{
    double a[TQ], d[TP];
#pragma unroll
    for (int q = 0; q < TQ; q++) a[q] = -seed * ((threadIdx.x * 7 + q * 3) % 11);
#pragma unroll
    for (int p = 0; p < TP; p++) d[p] = -seed * ((threadIdx.x * 5 + p) % 13);
    double tot = 0.0;
    for (int it = 0; it < iters; it++) {
        double best[TP][TQ];
#pragma unroll
        for (int p = 0; p < TP; p++)
#pragma unroll
            for (int q = 0; q < TQ; q++) best[p][q] = neg_inf();
        if (VAR == 1) {
            double v[TP][TQ];
#pragma unroll
            for (int p = 0; p < TP; p++)
#pragma unroll
                for (int q = 0; q < TQ; q++) v[p][q] = d[p] + a[q];
#pragma unroll 2
            for (int j = 0; j < K; j++) {
#pragma unroll
                for (int q = 0; q < TQ; q++) a[q] = a[q] * 1.0000001;
                double vn[TP][TQ];
#pragma unroll
                for (int p = 0; p < TP; p++)
#pragma unroll
                    for (int q = 0; q < TQ; q++) {
                        vn[p][q] = d[p] + a[q];                                  // next predecessor's add ...
                        best[p][q] = v[p][q] > best[p][q] ? v[p][q] : best[p][q];   // ... next to this one's select
                    }
#pragma unroll
                for (int p = 0; p < TP; p++)
#pragma unroll
                    for (int q = 0; q < TQ; q++) v[p][q] = vn[p][q];
            }
        } else {
#pragma unroll 4
            for (int j = 0; j < K; j++) {
#pragma unroll
                for (int p = 0; p < TP; p++)
#pragma unroll
                    for (int q = 0; q < TQ; q++) {
                        const double v = d[p] + a[q];
                        best[p][q] = v > best[p][q] ? v : best[p][q];
                    }
#pragma unroll
                for (int q = 0; q < TQ; q++) a[q] = a[q] * 1.0000001;
            }
        }
#pragma unroll
        for (int p = 0; p < TP; p++)
#pragma unroll
            for (int q = 0; q < TQ; q++) tot += best[p][q];
    }
    if (tot == 12345.678) out[blockIdx.x * blockDim.x + threadIdx.x] = tot;
}

// dispatch-port test: NF independent FFMA per DADD (ND = 0 -> FFMA only)
template <int ND, int NF>
__global__ void __launch_bounds__(512, 1) probe_mix_kernel(double *out, int iters, double seed)
{
    constexpr int NCH = 8;
    double acc[NCH]; float facc[NCH * (NF > 0 ? NF : 1)];
#pragma unroll
    for (int c = 0; c < NCH; c++) acc[c] = seed * (threadIdx.x + c);
#pragma unroll
    for (int c = 0; c < NCH * (NF > 0 ? NF : 1); c++) facc[c] = (float)seed * (threadIdx.x + c);
    const double inc = seed * 1e-3; const float finc = (float)seed * 1e-3f;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int c = 0; c < NCH; c++) {
            if (ND) acc[c] += inc;
#pragma unroll
            for (int f = 0; f < NF; f++) facc[c * NF + f] = fmaf(facc[c * NF + f], finc, finc);
        }
    }
    double s = 0.0;
#pragma unroll
    for (int c = 0; c < NCH; c++) s += acc[c];
#pragma unroll
    for (int c = 0; c < NCH * (NF > 0 ? NF : 1); c++) s += facc[c];
    if (s == 12345.678) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}



// dispatch-port test 2: NI independent integer ALU ops (LOP3/IADD3 class) per DADD; ND = 0 -> ALU only
template <int ND, int NI>
__global__ void __launch_bounds__(512, 1) probe_mix_alu_kernel(double *out, int iters, double seed)
{
    constexpr int NCH = 8;
    double acc[NCH]; unsigned iacc[NCH * (NI > 0 ? NI : 1)];
#pragma unroll
    for (int c = 0; c < NCH; c++) acc[c] = seed * (threadIdx.x + c);
#pragma unroll
    for (int c = 0; c < NCH * (NI > 0 ? NI : 1); c++) iacc[c] = threadIdx.x * 2654435761u + c;
    const double inc = seed * 1e-3; const unsigned m = (unsigned)(seed * 12345.0) | 1u;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int c = 0; c < NCH; c++) {
            if (ND) acc[c] += inc;
#pragma unroll
            for (int f = 0; f < NI; f++) iacc[c * NI + f] = (iacc[c * NI + f] ^ m) + (iacc[c * NI + f] >> 3);   // LOP3 + SHF/IADD
        }
    }
    double s = 0.0;
#pragma unroll
    for (int c = 0; c < NCH; c++) s += acc[c];
    unsigned si = 0;
#pragma unroll
    for (int c = 0; c < NCH * (NI > 0 ? NI : 1); c++) si += iacc[c];
    if (s == 12345.678 || si == 0x12345678u) out[blockIdx.x * blockDim.x + threadIdx.x] = s + si;
}

// dependent-chain latency probe: one warp, `iters` x 16 dependent ops; mode 0 DADD, 1 DSETP+FSEL (max), 2 SHFL+DADD
template <int MODE>
__global__ void probe_latency_kernel(double *out, int iters, double seed, long long *cycles)
{
    double acc = seed * (threadIdx.x + 1), best = -seed;
    const double inc = seed * 1e-3;
    const long long t0 = clock64();
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int k = 0; k < 16; k++) {
            if (MODE == 0) acc += inc;
            else if (MODE == 1) { const double v = inc * (k + it); best = v > best ? v : best; }
            else { acc = __shfl_sync(0xffffffffu, acc, (threadIdx.x + 1) & 31) + inc; }
        }
    }
    const long long t1 = clock64();
    if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;
    if (acc + best == 12345.678) out[threadIdx.x] = acc;
}

}  // namespace cvb
