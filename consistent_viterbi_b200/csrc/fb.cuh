// fb.cuh -- forward-backward inference on the device, K <= 64: per-sequence log10 P(O), posterior marginals gamma_t
// and posterior (maximum posterior marginal) decoding.  Semantics at cv_loglik_batch / cv_posterior_batch in
// include/cv_b200.h; the host side is fb_host.inl.
//
// The forward pass is bw_fwd_kernel of bw.cuh (tiles of 64 sequences sorted longest first, exact power-of-two scaling
// applied one step late): bw_fwd_kernel<false> for cv_loglik_batch, bw_fwd_kernel<true> (r_t kept in the history) for
// cv_posterior_batch.  Both instantiations run the same arithmetic, so the log-likelihoods of the two calls are the same
// bytes.  Kernels of a posterior chunk, in launch order:
//   bw_fwd_kernel<true>   scaled forward pass, r_t as [K][64] per history slab; log10 P(O) and the valid flag per rank
//   fb_bwd_kernel         scaled backward pass; gamma_t = r_t beta_t / Z_t written over the slab as [64][K]
//   fb_out_kernel         one warp per sequence: per position the first argmax and the maximum of the gamma row, the
//                         row itself into the [N][K] output when asked for, log10 P(O) at the caller's index
// A log-likelihood chunk runs bw_fwd_kernel<false> and fb_ll_kernel.
// Nothing is reduced across sequences: every value of a sequence comes from its own cells in an order fixed by K, so
// it does not depend on the batch, the slot or the tile the sequence lands in.
#pragma once
#include "bw.cuh"

namespace cvb {

// Largest finite model entry (log10) the forward-backward calls accept.  With every probability <= 10^x: the scaled
// forward rows sum to < K 10^(2x) (a predecessor row summing to < 1 times a and b), the scaled backward vectors stay
// < 10^x (a times a vector summing to < 1), so u_t = b o beta_t < 10^(2x) and Z_t = sum r_t beta_t < K 10^(3x).  At
// x = 64, K = 64: forward sums < 1e130 (far below the 1e300 above which bw_fwd_kernel treats a sum as an overflow) and
// Z_t < 1e194, so no product or sum overflows.  Real log-probability models (entries <= 0) are never refused.
constexpr double FB_MAX_ENTRY = 64.0;

struct FbParams {
    int K, Kp, G;
    int64_t B;                      // sequences of the chunk
    int ntiles;
    const double *AT;               // [K][Kp]  AT[j][i] = a[i][j]
    const double *BT;               // [M][Kp]
    const uint32_t *obs;            // [N] of the chunk
    const int64_t *seq_off;         // [B+1] of the chunk, from 0
    const uint32_t *order;          // [B] chunk-local sequence ids, longest first
    const long long *tile_base;     // [ntiles]
    double *hist;                   // r_t [K][64] per slab (forward), gamma_t [64][K] (backward)
    const double *ll;               // [B] log10 P(O) per rank (bw_fwd_kernel)
    const uint8_t *valid;           // [B] per rank
    uint32_t *path;                 // [N] or null
    double *pmax;                   // [N] or null
    double *post;                   // [N][K] or null
    double *loglik;                 // [B] per chunk-local sequence id
};

__host__ __device__ inline size_t fb_bwd_smem(int K, int Kp, int G)
{
    return ((size_t)K * Kp + 2 * (size_t)Kp * BW_NS + 4 * (size_t)G * BW_NS) * 8 + (size_t)BW_NS * (8 + 4 + 4);
}

// Backward pass, the mapping of bw_bwd_kernel without the transition expectations: warp g owns states [8g, 8g+8),
// lane l the sequences 2l, 2l+1.  Per step t (descending), one barrier:
//   phase A  own cells: r_t from the history, u_t = b(o_t) o beta_t -> sU[t&1], partial sums of r_t beta_t (Z) and u_t
//   phase B  gamma_t = r_t beta_t / Z_t over the history slab ([64][K]); beta_{t-1} = a u_t, scaled by the exponent of
//            sum_j u_t(j)
// Phase B of step t reads the buffers t&1 only; phase A of step t-1 writes the other ones, and phase A of step t-2 runs
// after the barrier of step t-1, which every warp reaches after its phase B of step t.
// 1/Z_t is formed from Z's mantissa m in [0.5, 1) and exponent e: gamma = (r beta (1/m)) 2^-e, so a Z in the subnormal
// range (emissions near 1e-300) cannot overflow 1/Z to inf.
__global__ void __launch_bounds__(32 * BW_KMAX / 8) fb_bwd_kernel(const FbParams p)
{
    extern __shared__ __align__(16) unsigned char fb_smem[];
    const int K = p.K, Kp = p.Kp, G = p.G;
    double *sAT = reinterpret_cast<double *>(fb_smem);      // [K][Kp]
    double *sU = sAT + (size_t)K * Kp;                         // [2][Kp][NS]
    double *sZ = sU + (size_t)2 * Kp * BW_NS;                  // [2][G][NS]
    double *sUs = sZ + (size_t)2 * G * BW_NS;                  // [2][G][NS]
    int64_t *sOff = reinterpret_cast<int64_t *>(sUs + (size_t)2 * G * BW_NS);
    int *sLen = reinterpret_cast<int *>(sOff + BW_NS);
    int *sValid = sLen + BW_NS;
    const int tid = threadIdx.x, lane = tid & 31, g = tid >> 5, i0 = 8 * g, s0 = 2 * lane;
    for (int e = tid; e < K * Kp; e += blockDim.x) sAT[e] = p.AT[e];
    auto gsum = [&](const double *buf, int s) {               // sum of the G group partials of slot s, fixed order
        double v = 0.0;
        for (int h = 0; h < G; h++) v += buf[(size_t)h * BW_NS + s];
        return v;
    };

    for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
        __syncthreads();
        for (int s = tid; s < BW_NS; s += blockDim.x) {
            const int64_t r = (int64_t)tile * BW_NS + s;
            int64_t off = 0; int len = 0, ok = 0;
            if (r < p.B) { const uint32_t b = p.order[r]; off = p.seq_off[b]; len = (int)(p.seq_off[b + 1] - off); ok = p.valid[r]; }
            sOff[s] = off; sLen[s] = len; sValid[s] = ok;
        }
        __syncthreads();
        const int Tmax = sLen[0];
        const long long slab0 = p.tile_base[tile];
        int len[2]; int64_t off[2]; bool ok[2];
#pragma unroll
        for (int q = 0; q < 2; q++) { len[q] = sLen[s0 + q]; off[q] = sOff[s0 + q]; ok[q] = sValid[s0 + q] != 0; }
        double beta[2][8];

        for (int t = Tmax - 1; t >= 0; t--) {
            const int b2 = t & 1;
            double r[2][8], u[2][8], zp[2], us[2];
            // ---- phase A ----
#pragma unroll
            for (int q = 0; q < 2; q++) {
                const bool act = t < len[q] && ok[q];
                if (t == len[q] - 1) {
#pragma unroll
                    for (int k = 0; k < 8; k++) beta[q][k] = i0 + k < K ? 1.0 : 0.0;
                }
                const uint32_t o = act ? __ldg(p.obs + off[q] + t) : 0u;
                const double *hp = p.hist + (size_t)(slab0 + t) * K * BW_NS + s0 + q;
                const double *bp = p.BT + (size_t)o * Kp + i0;
                zp[q] = 0.0; us[q] = 0.0;
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    r[q][k] = (act && i0 + k < K) ? hp[(size_t)(i0 + k) * BW_NS] : 0.0;
                    u[q][k] = act ? __ldg(bp + k) * beta[q][k] : 0.0;
                    zp[q] = fma(r[q][k], beta[q][k], zp[q]);
                    us[q] += u[q][k];
                }
            }
#pragma unroll
            for (int k = 0; k < 8; k++)
                *reinterpret_cast<double2 *>(sU + (size_t)b2 * Kp * BW_NS + (size_t)(i0 + k) * BW_NS + s0) = make_double2(u[0][k], u[1][k]);
            *reinterpret_cast<double2 *>(sZ + (size_t)b2 * G * BW_NS + (size_t)g * BW_NS + s0) = make_double2(zp[0], zp[1]);
            *reinterpret_cast<double2 *>(sUs + (size_t)b2 * G * BW_NS + (size_t)g * BW_NS + s0) = make_double2(us[0], us[1]);
            __syncthreads();
            // ---- phase B ----
#pragma unroll
            for (int q = 0; q < 2; q++) {
                if (t >= len[q]) continue;
                double *gp = p.hist + ((size_t)(slab0 + t) * BW_NS + s0 + q) * K + i0;
                const double Z = ok[q] ? gsum(sZ + (size_t)b2 * G * BW_NS, s0 + q) : 0.0;
                int ez = 0;
                const double inv = Z > 0.0 ? 1.0 / frexp(Z, &ez) : 0.0;   // P(O) = 0: a row of zeros
#pragma unroll
                for (int k = 0; k < 8; k++)
                    if (i0 + k < K) gp[k] = ldexp(r[q][k] * beta[q][k] * inv, -ez);
            }
            if (t > 0) {
                int f[2];
#pragma unroll
                for (int q = 0; q < 2; q++) f[q] = bw_exponent(gsum(sUs + (size_t)b2 * G * BW_NS, s0 + q));
                double nb[2][8];
#pragma unroll
                for (int k = 0; k < 8; k++) nb[0][k] = nb[1][k] = 0.0;
                const double *up = sU + (size_t)b2 * Kp * BW_NS + s0;
                const double *ap = sAT + i0;
#pragma unroll 4
                for (int j = 0; j < K; j++) {
                    const double2 d = *reinterpret_cast<const double2 *>(up + (size_t)j * BW_NS);
                    double a[8];
#pragma unroll
                    for (int k = 0; k < 8; k += 2) {
                        const double2 aa = *reinterpret_cast<const double2 *>(ap + (size_t)j * Kp + k);
                        a[k] = aa.x; a[k + 1] = aa.y;
                    }
#pragma unroll
                    for (int k = 0; k < 8; k++) { nb[0][k] = fma(a[k], d.x, nb[0][k]); nb[1][k] = fma(a[k], d.y, nb[1][k]); }
                }
#pragma unroll
                for (int q = 0; q < 2; q++)
#pragma unroll
                    for (int k = 0; k < 8; k++) beta[q][k] = ldexp(nb[q][k], -f[q]);
            }
        }
    }
}

// One warp per sequence (by rank), its positions in order.  Lane l holds states l and l + 32 of the gamma row; the
// first argmax is the largest value with the lowest index, found by a butterfly whose result does not depend on the
// order of the comparisons (max is exact, ties go to the lower index).
__global__ void fb_out_kernel(const FbParams p)
{
    const int lane = threadIdx.x & 31, K = p.K;
    const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < p.B; r += nw) {
        const uint32_t b = p.order[r];
        const int64_t off = p.seq_off[b], len = p.seq_off[b + 1] - off;
        if (lane == 0 && p.loglik) p.loglik[b] = p.valid[r] ? p.ll[r] : -INFINITY;
        const double *gp = p.hist + ((size_t)p.tile_base[r / BW_NS] * BW_NS + r % BW_NS) * K;
        for (int64_t t = 0; t < len; t++, gp += (size_t)BW_NS * K) {
            const double v0 = lane < K ? __ldcs(gp + lane) : -1.0;
            const double v1 = lane + 32 < K ? __ldcs(gp + lane + 32) : -1.0;
            double v = v0; int i = lane;
            if (v1 > v) { v = v1; i = lane + 32; }
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) {
                const double ov = __shfl_xor_sync(0xffffffffu, v, d);
                const int oi = __shfl_xor_sync(0xffffffffu, i, d);
                if (ov > v || (ov == v && oi < i)) { v = ov; i = oi; }
            }
            const int64_t x = off + t;
            if (lane == 0) {
                if (p.path) p.path[x] = (uint32_t)i;
                if (p.pmax) p.pmax[x] = v;
            }
            if (p.post) {
                if (lane < K) __stcs(p.post + (size_t)x * K + lane, v0);
                if (lane + 32 < K) __stcs(p.post + (size_t)x * K + lane + 32, v1);
            }
        }
    }
}

// cv_loglik_batch: log10 P(O) from rank order to the caller's order, -inf where P(O) = 0
__global__ void fb_ll_kernel(const FbParams p)
{
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < p.B) p.loglik[p.order[r]] = p.valid[r] ? p.ll[r] : -INFINITY;
}

}  // namespace cvb
