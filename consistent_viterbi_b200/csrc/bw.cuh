// bw.cuh -- one Baum-Welch (EM) iteration of the HMM on the device, K <= 64.
//
// Semantics (the expected counts, the M-step, skipped sequences) are documented at cv_baum_welch in
// include/cv_b200.h.  The E-step is the sum-product counterpart of the batched Viterbi forward pass
// (decode_small.cuh): the same tiles of 64 sequences sorted longest first, the same [state][sequence] slabs, but
// every cell is one DFMA on probabilities instead of DADD + DSETP + selects.
//
// Kernels of one iteration, in launch order:
//   bw_prep_kernel      log10 model -> probabilities (10^x, -inf -> 0) in the padded layouts the kernels read
//   bw_fwd_kernel       scaled forward pass; writes r_t (below) and the scale exponents e_t to the history
//   bw_ll_kernel        log10 P(O) summed over the contributing sequences in rank order; counts the skipped ones
//   bw_bwd_kernel       scaled backward pass; transition expectations X, occupancies; gamma over the history
//   bw_reduce_kernel    per-CTA partials summed in CTA order
//   bw_emit_kernel      gamma summed per chunk of positions sorted by observation
//   bw_mstep_b_kernel   chunk sums per observation in chunk order -> log10 b
//   bw_mstep_a_kernel   log10 a, log10 pi
// No floating-point atomics anywhere, tiles are dealt to CTAs round-robin (not by a work counter), and every
// reduction runs in an order fixed by the data: two calls with the same inputs on the same GPU give the same bytes.
//
// Scaling.  r_0(i) = pi_i b_i(o_0);  r_t(i) = 2^-e_{t-1} (sum_j r_{t-1}(j) a_ji) b_i(o_t), with e_t the binary exponent
// of sum_i r_t(i) (frexp).  The scale of step t is applied one step late, from the per-state-group partial sums every
// thread writes before the step barrier, so the forward pass needs no barrier beyond the one of the double buffer.
// Powers of two are exact, so r_t = alpha_t 2^-(e_0 + .. + e_{t-1}) and log10 P(O) = log10 sum_i r_{T-1}(i) +
// (e_0 + .. + e_{T-2}) log10 2.  The backward pass scales beta the same way (by the exponent of sum_j u_t(j),
// u_t = b(o_t) o beta_t); its scales cancel in every normalised quantity:
//   gamma_t(i)  = r_t(i) beta_t(i) / Z_t,                      Z_t = sum_i r_t(i) beta_t(i)
//   xi_t(i,j)   = [r_{t-1}(i) 2^-e_{t-1} / Z_t] a_ij u_t(j)    (sum_ij of the bracket times a u = 2^e Z / 2^e Z = 1)
// X[i][j] = sum of r_{t-1}(i) 2^-e_{t-1} / Z_t * u_t(j) is accumulated and multiplied by a_ij once, in the M-step.
// A sequence whose forward sum is 0 (P(O) = 0, or underflow) is skipped: it contributes nothing.
#pragma once
#include "common.cuh"

namespace cvb {

constexpr int BW_NS = 64;           // sequences per tile
constexpr int BW_KMAX = 64;
constexpr int BW_CHUNK = 512;       // positions per emission chunk

struct BwParams {
    int K, Kp, G;                   // Kp = 8 G, G = state groups of 8 (one warp each)
    int64_t M, B;
    int ntiles;
    // model, probabilities, padded with 0
    double *A;                      // [K][Kp]  a[from][to]
    double *AT;                     // [K][Kp]  AT[j][i] = a[i][j]
    double *BT;                     // [M][Kp]  b[state][o] transposed
    double *pi;                     // [Kp]
    // model, log10 (what the call returns)
    double *logA, *logB, *logPi;    // [K*K] [K*M] [K]
    const uint32_t *obs;            // [N]
    const int64_t *seq_off;         // [B+1]
    const uint32_t *order;          // [B] sequence ids, longest first (rank order)
    const long long *tile_base;     // [ntiles] first slab of each tile
    double *hist;                   // slabs of K*64 doubles: r_t as [K][64] (forward), gamma_t as [64][K] (backward)
    int *ehist;                     // [slabs][64] e_t
    double *ll;                     // [B] log10 P(O) per rank
    uint8_t *valid;                 // [B] 1 = contributing sequence
    double *part;                   // [grid][NP] per-CTA partials, NP = K*K + 3K: X, occ_a, occ_b, occ_first
    double *sums;                   // [NP]
    const int64_t *sorted;          // [N] history positions (slab * 64 + slot), stably sorted by observation
    const int64_t *chunk_pos;       // [nchunk + 1] first sorted position of every chunk
    const int *obs_chunk;           // [M + 1] first chunk of every observation
    int64_t nchunk;
    double *chunk_sum;              // [nchunk][Kp]
    double *loglik;                 // [n_iter]
    long long *skipped;             // [n_iter]
    int iter;
};

__host__ __device__ inline int bw_np(int K) { return K * K + 3 * K; }
__host__ __device__ inline size_t bw_fwd_smem(int K, int Kp, int G)
{
    return ((size_t)K * Kp + 2 * (size_t)Kp * BW_NS + 2 * (size_t)G * BW_NS) * 8 + (size_t)BW_NS * (8 + 4);
}
__host__ __device__ inline size_t bw_bwd_smem(int K, int Kp, int G)
{
    return ((size_t)K * Kp + 5 * (size_t)Kp * BW_NS + 6 * (size_t)G * BW_NS) * 8 + (size_t)BW_NS * (8 + 4 + 4);
}

// binary exponent e of S as frexp gives it (S = m 2^e, m in [0.5, 1)); 0 for S = 0
__device__ __forceinline__ int bw_exponent(double S) { return S > 0.0 ? ilogb(S) + 1 : 0; }

__device__ __forceinline__ double pow10_or_zero(double x) { return x == -INFINITY ? 0.0 : exp10(x); }

__global__ void bw_prep_kernel(const BwParams p)
{
    const int K = p.K, Kp = p.Kp;
    const int64_t n = (int64_t)max(p.M, (int64_t)K) * Kp;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t o = e / Kp;
        const int s = (int)(e % Kp);
        if (o < p.M) p.BT[e] = s < K ? pow10_or_zero(p.logB[(size_t)s * p.M + o]) : 0.0;
        if (e < (int64_t)K * Kp) {
            const int r = (int)(e / Kp);
            p.A[e] = s < K ? pow10_or_zero(p.logA[(size_t)r * K + s]) : 0.0;
            p.AT[e] = s < K ? pow10_or_zero(p.logA[(size_t)s * K + r]) : 0.0;
        }
        if (e < Kp) p.pi[e] = e < K ? pow10_or_zero(p.logPi[e]) : 0.0;
    }
}

// Forward pass.  Warp g owns states [8g, 8g+8), lane l the sequences 2l, 2l+1 of the tile: 16 cells per thread,
// K DFMAs each per step, operands from shared memory (r_{t-1}: one LDS.128 per predecessor, a: four broadcast LDS.128).
// HIST = false (cv_loglik_batch, fb.cuh) skips the stores of r_t and e_t to the history; the arithmetic is the same.
template <bool HIST>
__global__ void __launch_bounds__(32 * BW_KMAX / 8) bw_fwd_kernel(const BwParams p)
{
    extern __shared__ __align__(16) unsigned char bw_smem[];
    const int K = p.K, Kp = p.Kp, G = p.G;
    double *sA = reinterpret_cast<double *>(bw_smem);       // [K][Kp]
    double *sD = sA + (size_t)K * Kp;                          // [2][Kp][NS]
    double *sP = sD + (size_t)2 * Kp * BW_NS;                  // [2][G][NS] partial sums of r_t per state group
    int64_t *sOff = reinterpret_cast<int64_t *>(sP + (size_t)2 * G * BW_NS);
    int *sLen = reinterpret_cast<int *>(sOff + BW_NS);
    const int tid = threadIdx.x, lane = tid & 31, g = tid >> 5, i0 = 8 * g, s0 = 2 * lane;
    for (int e = tid; e < K * Kp; e += blockDim.x) sA[e] = p.A[e];
    const double LOG10_2 = log10(2.0);

    for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
        __syncthreads();                                       // the previous tile is done with sOff / sLen
        for (int s = tid; s < BW_NS; s += blockDim.x) {
            const int64_t r = (int64_t)tile * BW_NS + s;
            int64_t off = 0; int len = 0;
            if (r < p.B) { const uint32_t b = p.order[r]; off = p.seq_off[b]; len = (int)(p.seq_off[b + 1] - off); }
            sOff[s] = off; sLen[s] = len;
        }
        __syncthreads();
        const int Tmax = sLen[0];
        const long long slab0 = p.tile_base[tile];
        int len[2]; int64_t off[2]; long long E[2] = {0, 0}; int e_prev[2] = {0, 0};
#pragma unroll
        for (int q = 0; q < 2; q++) { len[q] = sLen[s0 + q]; off[q] = sOff[s0 + q]; }

        for (int t = 0; t <= Tmax; t++) {
            if (t > 0) {
                // exponent of row t-1 (partials published by the barrier of step t-1); the end of a sequence: log10 P(O)
#pragma unroll
                for (int q = 0; q < 2; q++) {
                    double S = 0.0;
                    for (int h = 0; h < G; h++) S += sP[(size_t)((t - 1) & 1) * G * BW_NS + (size_t)h * BW_NS + s0 + q];
                    const int e = bw_exponent(S);
                    e_prev[q] = e;
                    if (t - 1 < len[q]) {
                        if (HIST && g == 0) p.ehist[(size_t)(slab0 + t - 1) * BW_NS + s0 + q] = e;
                        if (t - 1 == len[q] - 1) {
                            if (g == 0) {
                                const int64_t r = (int64_t)tile * BW_NS + s0 + q;
                                const bool ok = S > 0.0 && S <= 1e300;
                                p.valid[r] = ok ? 1 : 0;
                                p.ll[r] = ok ? log10(S) + (double)E[q] * LOG10_2 : 0.0;
                            }
                        } else {
                            E[q] += e;
                        }
                    }
                }
            }
            if (t == Tmax) break;
            double acc[2][8];
            if (t == 0) {
#pragma unroll
                for (int k = 0; k < 8; k++) acc[0][k] = acc[1][k] = p.pi[i0 + k];
            } else {
#pragma unroll
                for (int k = 0; k < 8; k++) acc[0][k] = acc[1][k] = 0.0;
                const double *dp = sD + (size_t)((t - 1) & 1) * Kp * BW_NS + s0;
                const double *ap = sA + i0;
#pragma unroll 4
                for (int j = 0; j < K; j++) {
                    const double2 d = *reinterpret_cast<const double2 *>(dp + (size_t)j * BW_NS);
                    double a[8];
#pragma unroll
                    for (int k = 0; k < 8; k += 2) {
                        const double2 aa = *reinterpret_cast<const double2 *>(ap + (size_t)j * Kp + k);
                        a[k] = aa.x; a[k + 1] = aa.y;
                    }
#pragma unroll
                    for (int k = 0; k < 8; k++) { acc[0][k] = fma(d.x, a[k], acc[0][k]); acc[1][k] = fma(d.y, a[k], acc[1][k]); }
                }
            }
            double ps[2];
#pragma unroll
            for (int q = 0; q < 2; q++) {
                ps[q] = 0.0;
                const bool act = t < len[q];
                const uint32_t o = act ? __ldg(p.obs + off[q] + t) : 0u;
                const double *bp = p.BT + (size_t)o * Kp + i0;
#pragma unroll
                for (int k = 0; k < 8; k += 2) {
                    const double2 bb = __ldg(reinterpret_cast<const double2 *>(bp + k));
                    acc[q][k] = act ? ldexp(acc[q][k] * bb.x, -e_prev[q]) : 0.0;
                    acc[q][k + 1] = act ? ldexp(acc[q][k + 1] * bb.y, -e_prev[q]) : 0.0;
                }
#pragma unroll
                for (int k = 0; k < 8; k++) ps[q] += acc[q][k];
            }
            double *dn = sD + (size_t)(t & 1) * Kp * BW_NS + s0;
            double *hp = p.hist + (size_t)(slab0 + t) * K * BW_NS + s0;
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const double2 v = make_double2(acc[0][k], acc[1][k]);
                *reinterpret_cast<double2 *>(dn + (size_t)(i0 + k) * BW_NS) = v;
                if (HIST && i0 + k < K) *reinterpret_cast<double2 *>(hp + (size_t)(i0 + k) * BW_NS) = v;
            }
            *reinterpret_cast<double2 *>(sP + (size_t)(t & 1) * G * BW_NS + (size_t)g * BW_NS + s0) = make_double2(ps[0], ps[1]);
            __syncthreads();
        }
    }
}

// log10 P(O) over the contributing sequences, summed in rank order by a fixed tree; skipped sequences counted
__global__ void __launch_bounds__(1024) bw_ll_kernel(const BwParams p)
{
    __shared__ double sh[1024];
    __shared__ long long shn[1024];
    double v = 0.0; long long n = 0;
    for (int64_t r = threadIdx.x; r < p.B; r += blockDim.x) {
        if (p.valid[r]) v += p.ll[r];
        else n++;
    }
    sh[threadIdx.x] = v; shn[threadIdx.x] = n;
    __syncthreads();
    for (int w = blockDim.x / 2; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) { sh[threadIdx.x] += sh[threadIdx.x + w]; shn[threadIdx.x] += shn[threadIdx.x + w]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { p.loglik[p.iter] = sh[0]; p.skipped[p.iter] = shn[0]; }
}

// Backward pass + expected counts, same thread mapping as the forward pass.  Per step t (descending), one barrier:
//   phase A  own cells: r_t from the history, u_t = b(o_t) o beta_t -> sU[t%3], r_t 2^-e_t / Z_{t+1} -> sR[t&1],
//            partial sums of r_t beta_t (Z) and of u_t (beta scale)
//   phase B  gamma_t = r_t beta_t / Z_t over the history slab ([64][K]: rows of a position are contiguous for the
//            emission pass) and into the occupancies; beta_{t-1} = a u_t (scaled); X += sR[t&1] (x) sU[(t+1)%3]
// Phase B of step t reads only what phase A of steps t and t+1 wrote; phase A of step t-1 writes other buffers.
__global__ void __launch_bounds__(32 * BW_KMAX / 8) bw_bwd_kernel(const BwParams p)
{
    extern __shared__ __align__(16) unsigned char bw_smem[];
    const int K = p.K, Kp = p.Kp, G = p.G;
    double *sAT = reinterpret_cast<double *>(bw_smem);      // [K][Kp]
    double *sU = sAT + (size_t)K * Kp;                         // [3][Kp][NS]
    double *sR = sU + (size_t)3 * Kp * BW_NS;                  // [2][Kp][NS]
    double *sZ = sR + (size_t)2 * Kp * BW_NS;                  // [3][G][NS]
    double *sUs = sZ + (size_t)3 * G * BW_NS;                  // [3][G][NS]
    int64_t *sOff = reinterpret_cast<int64_t *>(sUs + (size_t)3 * G * BW_NS);
    int *sLen = reinterpret_cast<int *>(sOff + BW_NS);
    int *sValid = sLen + BW_NS;
    const int tid = threadIdx.x, lane = tid & 31, g = tid >> 5, i0 = 8 * g, s0 = 2 * lane;
    for (int e = tid; e < K * Kp; e += blockDim.x) sAT[e] = p.AT[e];
    const int nxb = 2 * G;                                     // X blocks of 4 x 4 per dimension
    const bool xown = tid < nxb * nxb;
    const int ib = xown ? tid / nxb : 0, jb = xown ? tid % nxb : 0;
    double X[4][4], occA[8], occB[8], occF[8];
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) X[a][b] = 0.0;
#pragma unroll
    for (int k = 0; k < 8; k++) occA[k] = occB[k] = occF[k] = 0.0;
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
            const int b3 = t % 3, b3n = (t + 1) % 3;
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
                double c = 0.0;
                if (act && t + 1 < len[q]) {
                    const int e = p.ehist[(size_t)(slab0 + t) * BW_NS + s0 + q];
                    c = ldexp(1.0 / gsum(sZ + (size_t)b3n * G * BW_NS, s0 + q), -e);
                }
                // sR = r_t 2^-e_t / Z_{t+1}: c carries both factors (exact power-of-two scaling of 1/Z)
#pragma unroll
                for (int k = 0; k < 8; k++) sR[(size_t)(t & 1) * Kp * BW_NS + (size_t)(i0 + k) * BW_NS + s0 + q] = r[q][k] * c;
            }
#pragma unroll
            for (int k = 0; k < 8; k++)
                *reinterpret_cast<double2 *>(sU + (size_t)b3 * Kp * BW_NS + (size_t)(i0 + k) * BW_NS + s0) = make_double2(u[0][k], u[1][k]);
            *reinterpret_cast<double2 *>(sZ + (size_t)b3 * G * BW_NS + (size_t)g * BW_NS + s0) = make_double2(zp[0], zp[1]);
            *reinterpret_cast<double2 *>(sUs + (size_t)b3 * G * BW_NS + (size_t)g * BW_NS + s0) = make_double2(us[0], us[1]);
            __syncthreads();
            // ---- phase B ----
#pragma unroll
            for (int q = 0; q < 2; q++) {
                if (t >= len[q]) continue;
                double *gp = p.hist + ((size_t)(slab0 + t) * BW_NS + s0 + q) * K + i0;
                if (!ok[q]) {                                  // skipped sequence: no emission counts
#pragma unroll
                    for (int k = 0; k < 8; k++) if (i0 + k < K) gp[k] = 0.0;
                    continue;
                }
                const double Z = gsum(sZ + (size_t)b3 * G * BW_NS, s0 + q);
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    if (i0 + k >= K) break;
                    const double gm = r[q][k] * beta[q][k] / Z;
                    gp[k] = gm;
                    occB[k] += gm;
                    if (t < len[q] - 1) occA[k] += gm;
                    if (t == 0) occF[k] += gm;
                }
            }
            if (t > 0) {
                int f[2];
#pragma unroll
                for (int q = 0; q < 2; q++) f[q] = bw_exponent(gsum(sUs + (size_t)b3 * G * BW_NS, s0 + q));
                double nb[2][8];
#pragma unroll
                for (int k = 0; k < 8; k++) nb[0][k] = nb[1][k] = 0.0;
                const double *up = sU + (size_t)b3 * Kp * BW_NS + s0;
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
            if (xown && t + 1 < Tmax) {
                const double *rp = sR + (size_t)(t & 1) * Kp * BW_NS + (size_t)(4 * ib) * BW_NS;
                const double *up = sU + (size_t)b3n * Kp * BW_NS + (size_t)(4 * jb) * BW_NS;
#pragma unroll 2
                for (int s = 0; s < BW_NS; s += 2) {
                    double2 rv[4], uv[4];
#pragma unroll
                    for (int a = 0; a < 4; a++) {
                        rv[a] = *reinterpret_cast<const double2 *>(rp + (size_t)a * BW_NS + s);
                        uv[a] = *reinterpret_cast<const double2 *>(up + (size_t)a * BW_NS + s);
                    }
#pragma unroll
                    for (int a = 0; a < 4; a++)
#pragma unroll
                        for (int b = 0; b < 4; b++) X[a][b] = fma(rv[a].y, uv[b].y, fma(rv[a].x, uv[b].x, X[a][b]));
                }
            }
        }
    }
    // per-CTA partials: X blocks as they are, occupancies reduced over the lanes of each warp (fixed butterfly)
    double *pp = p.part + (size_t)blockIdx.x * bw_np(K);
    if (xown) {
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int b = 0; b < 4; b++) {
                const int i = 4 * ib + a, j = 4 * jb + b;
                if (i < K && j < K) pp[(size_t)i * K + j] = X[a][b];
            }
    }
#pragma unroll
    for (int k = 0; k < 8; k++) {
        double va = occA[k], vb = occB[k], vf = occF[k];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            va += __shfl_xor_sync(0xffffffffu, va, d);
            vb += __shfl_xor_sync(0xffffffffu, vb, d);
            vf += __shfl_xor_sync(0xffffffffu, vf, d);
        }
        if (lane == 0 && i0 + k < K) {
            pp[(size_t)K * K + i0 + k] = va;
            pp[(size_t)K * K + K + i0 + k] = vb;
            pp[(size_t)K * K + 2 * K + i0 + k] = vf;
        }
    }
}

__global__ void bw_reduce_kernel(const BwParams p, int nparts)
{
    const int NP = bw_np(p.K);
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= NP) return;
    double v = 0.0;
    for (int c = 0; c < nparts; c++) v += p.part[(size_t)c * NP + e];
    p.sums[e] = v;
}

// one warp per chunk of BW_CHUNK positions of one observation; lane l sums gamma of states l and l + 32 in order
__global__ void bw_emit_kernel(const BwParams p)
{
    const int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31, K = p.K;
    if (c >= p.nchunk) return;
    double v0 = 0.0, v1 = 0.0;
    const int64_t end = p.chunk_pos[c + 1];
    for (int64_t x = p.chunk_pos[c]; x < end; x++) {
        const double *gp = p.hist + (size_t)__ldg(p.sorted + x) * K;
        if (lane < K) v0 += __ldcs(gp + lane);
        if (lane + 32 < K) v1 += __ldcs(gp + lane + 32);
    }
    double *out = p.chunk_sum + (size_t)c * p.Kp;
    if (lane < K) out[lane] = v0;
    if (lane + 32 < K) out[lane + 32] = v1;
}

// one warp per observation: expected emission counts (chunks in order) / occupancy -> log10 b
__global__ void bw_mstep_b_kernel(const BwParams p)
{
    const int64_t m = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31, K = p.K;
    if (m >= p.M) return;
    const double *occB = p.sums + (size_t)K * K + K;
    for (int j = lane; j < K; j += 32) {
        double v = 0.0;
        for (int c = p.obs_chunk[m]; c < p.obs_chunk[m + 1]; c++) v += p.chunk_sum[(size_t)c * p.Kp + j];
        p.logB[(size_t)j * p.M + m] = occB[j] > 0.0 ? hmm_log10(v / occB[j]) : -INFINITY;
    }
}

// log10 a = log10 (X a / occ_a), log10 pi = log10 (occ_first / contributing sequences); zero denominators give zero rows
__global__ void bw_mstep_a_kernel(const BwParams p)
{
    const int K = p.K;
    const double *occA = p.sums + (size_t)K * K, *occF = occA + 2 * K;
    const long long ncontrib = p.B - p.skipped[p.iter];
    for (int e = threadIdx.x; e < K * K; e += blockDim.x) {
        const int i = e / K, j = e % K;
        p.logA[e] = occA[i] > 0.0 ? hmm_log10(p.sums[e] * p.A[(size_t)i * p.Kp + j] / occA[i]) : -INFINITY;
    }
    for (int i = threadIdx.x; i < K; i += blockDim.x)
        p.logPi[i] = ncontrib > 0 ? hmm_log10(occF[i] / (double)ncontrib) : -INFINITY;
}

}  // namespace cvb
