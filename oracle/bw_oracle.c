/*
 * bw_oracle.c -- CPU oracle of cv_baum_welch (Baum-Welch EM), see bw_oracle.h.
 *
 * TEST INFRASTRUCTURE ONLY, like cv_oracle.c: only tests/, __graft_entry__.smoke() and tools/bw_bench.py load it.
 * Compile WITHOUT fast-math and without FMA contraction (bw.mk: -O2 -ffp-contract=off -fno-fast-math).
 */
#include "bw_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <omp.h>

/* ---- Baum-Welch (EM), the semantics of cv_baum_welch (include/cv_b200.h) ----------------------------------------
 * A literal restatement in LOG space (natural logarithms, log-sum-exp), independent of the device's scaled
 * probabilities: forward alpha and backward beta with every row shifted by its log-sum-exp, log P(O) = sum of the
 * forward shifts, gamma_t / xi_t normalised per t; expected counts summed per OpenMP thread (static schedule over
 * sequences) and combined in thread order. */
static double lse(const double *x, int n)
{
    double m = -INFINITY;
    for (int k = 0; k < n; k++) if (x[k] > m) m = x[k];
    if (m == -INFINITY) return -INFINITY;
    double s = 0.0;
    for (int k = 0; k < n; k++) s += exp(x[k] - m);
    return m + log(s);
}

static double log10_or_ninf(double x) { return x == 0.0 ? -INFINITY : log(x) / log(10.0); }

int cvo_baum_welch(int K, int64_t M, double *logA, double *logB, double *logPi, const uint32_t *obs,
                   const int64_t *seq_off, int64_t B, int n_iter, double tol, double *loglik_out, int *iters_out,
                   int64_t *skipped_out, int nthreads)
{
    if (K <= 0 || M <= 0 || B < 1 || n_iter < 1 || !logA || !logB || !logPi || !obs || !seq_off) return CVO_ERR_ARG;
    for (int64_t i = 0; i < B; i++)
        if (seq_off[i + 1] <= seq_off[i]) return CVO_ERR_EMPTY;
    for (int64_t x = 0; x < seq_off[B]; x++)
        if ((int64_t)obs[x] >= M) return CVO_ERR_ARG;
    for (int64_t e = 0; e < (int64_t)K * K; e++) if (logA[e] != logA[e] || logA[e] == INFINITY) return CVO_ERR_NAN;
    for (int64_t e = 0; e < (int64_t)K * M; e++) if (logB[e] != logB[e] || logB[e] == INFINITY) return CVO_ERR_NAN;
    for (int e = 0; e < K; e++) if (logPi[e] != logPi[e] || logPi[e] == INFINITY) return CVO_ERR_NAN;
    if (nthreads < 1) nthreads = 1;
    int64_t Tmax = 0;
    for (int64_t i = 0; i < B; i++) if (seq_off[i + 1] - seq_off[i] > Tmax) Tmax = seq_off[i + 1] - seq_off[i];
    const double ln10 = log(10.0);
    const size_t NA = (size_t)K * K, NB = (size_t)K * M, NC = NA + NB + 3 * (size_t)K;   /* X, emis, occA, occB, occF */
    double *lA = malloc(NA * sizeof(double)), *lB = malloc(NB * sizeof(double)), *lP = malloc((size_t)K * sizeof(double));
    double *acc = calloc(NC * (size_t)nthreads, sizeof(double));
    double *tll = calloc((size_t)nthreads, sizeof(double));
    int64_t *tsk = calloc((size_t)nthreads, sizeof(int64_t));
    if (!lA || !lB || !lP || !acc || !tll || !tsk) { free(lA); free(lB); free(lP); free(acc); free(tll); free(tsk); return CVO_ERR_ARG; }
    int iters = 0;
    int64_t skipped = 0;
    for (int it = 0; it < n_iter; it++) {
        for (size_t e = 0; e < NA; e++) lA[e] = logA[e] * ln10;
        for (size_t e = 0; e < NB; e++) lB[e] = logB[e] * ln10;
        for (int e = 0; e < K; e++) lP[e] = logPi[e] * ln10;
        memset(acc, 0, NC * (size_t)nthreads * sizeof(double));
        memset(tll, 0, (size_t)nthreads * sizeof(double));
        memset(tsk, 0, (size_t)nthreads * sizeof(int64_t));
#pragma omp parallel num_threads(nthreads)
        {
            const int th = omp_get_thread_num();
            double *X = acc + NC * (size_t)th, *em = X + NA, *occA = em + NB, *occB = occA + K, *occF = occB + K;
            double *la = malloc((size_t)Tmax * K * sizeof(double)), *lb = malloc((size_t)Tmax * K * sizeof(double));
            double *tmp = malloc((size_t)K * sizeof(double)), *xi = malloc(NA * sizeof(double));
#pragma omp for schedule(static)
            for (int64_t i = 0; i < B; i++) {
                const uint32_t *o = obs + seq_off[i];
                const int64_t T = seq_off[i + 1] - seq_off[i];
                /* forward, every row shifted by its own log-sum-exp c_t: log P(O) = sum_t c_t, and no log value
                 * grows with t (unshifted, ln alpha of a 10 000-step sequence is ~1e5 and carries ~1e-11 absolute
                 * error per operation into every posterior) */
                double lp = 0.0;
                for (int s = 0; s < K; s++) la[s] = lP[s] + lB[(size_t)s * M + o[0]];
                for (int64_t t = 0; t < T && lp != -INFINITY; t++) {
                    if (t > 0)
                        for (int s = 0; s < K; s++) {
                            for (int j = 0; j < K; j++) tmp[j] = la[(t - 1) * K + j] + lA[(size_t)j * K + s];
                            la[t * K + s] = lse(tmp, K) + lB[(size_t)s * M + o[t]];
                        }
                    const double c = lse(la + t * K, K);
                    lp = c == -INFINITY ? -INFINITY : lp + c;
                    if (c != -INFINITY) for (int s = 0; s < K; s++) la[t * K + s] -= c;
                }
                if (lp == -INFINITY) { tsk[th]++; continue; }
                tll[th] += lp / ln10;
                for (int s = 0; s < K; s++) lb[(T - 1) * K + s] = 0.0;
                for (int64_t t = T - 1; t >= 1; t--) {
                    for (int s = 0; s < K; s++) {
                        for (int j = 0; j < K; j++) tmp[j] = lA[(size_t)s * K + j] + lB[(size_t)j * M + o[t]] + lb[t * K + j];
                        lb[(t - 1) * K + s] = lse(tmp, K);
                    }
                    const double c = lse(lb + (t - 1) * K, K);
                    for (int s = 0; s < K; s++) lb[(t - 1) * K + s] -= c;
                }
                /* posteriors, normalised per t: gamma_t = exp(la + lb) / sum, xi_t = exp(la_{t-1} + lA + lB + lb_t) / sum */
                for (int64_t t = 0; t < T; t++) {
                    for (int s = 0; s < K; s++) tmp[s] = la[t * K + s] + lb[t * K + s];
                    const double z = lse(tmp, K);
                    for (int s = 0; s < K; s++) {
                        const double g = exp(tmp[s] - z);
                        occB[s] += g;
                        if (t < T - 1) occA[s] += g;
                        if (t == 0) occF[s] += g;
                        em[(size_t)s * M + o[t]] += g;
                    }
                }
                for (int64_t t = 1; t < T; t++) {
                    for (int s = 0; s < K; s++)
                        for (int j = 0; j < K; j++)
                            xi[(size_t)s * K + j] = la[(t - 1) * K + s] + lA[(size_t)s * K + j] + lB[(size_t)j * M + o[t]] + lb[t * K + j];
                    const double z = lse(xi, K * K);
                    for (size_t e = 0; e < NA; e++) X[e] += exp(xi[e] - z);
                }
            }
            free(la); free(lb); free(tmp); free(xi);
        }
        double ll = 0.0;
        skipped = 0;
        for (int th = 1; th < nthreads; th++)
            for (size_t e = 0; e < NC; e++) acc[e] += acc[NC * (size_t)th + e];
        for (int th = 0; th < nthreads; th++) { ll += tll[th]; skipped += tsk[th]; }
        const double *X = acc, *em = X + NA, *occA = em + NB, *occB = occA + K, *occF = occB + K;
        const int64_t ncontrib = B - skipped;
        for (int s = 0; s < K; s++) {
            for (int j = 0; j < K; j++) logA[(size_t)s * K + j] = log10_or_ninf(occA[s] > 0.0 ? X[(size_t)s * K + j] / occA[s] : 0.0);
            for (int64_t m = 0; m < M; m++) logB[(size_t)s * M + m] = log10_or_ninf(occB[s] > 0.0 ? em[(size_t)s * M + m] / occB[s] : 0.0);
            logPi[s] = log10_or_ninf(ncontrib > 0 ? occF[s] / (double)ncontrib : 0.0);
        }
        loglik_out[it] = ll;
        iters = it + 1;
        if (tol > 0.0 && it > 0 && loglik_out[it] - loglik_out[it - 1] < tol * fabs(loglik_out[it - 1])) break;
    }
    *iters_out = iters;
    *skipped_out = skipped;
    free(lA); free(lB); free(lP); free(acc); free(tll); free(tsk);
    return CVO_OK;
}
