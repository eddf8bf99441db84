/*
 * fb_oracle.c -- CPU oracle of cv_loglik_batch / cv_posterior_batch (forward-backward inference), see fb_oracle.h.
 *
 * TEST INFRASTRUCTURE ONLY, like bw_oracle.c: only tests/, __graft_entry__.smoke() and tools/fb_bench.py load it.
 * Compile WITHOUT fast-math and without FMA contraction (fb.mk: -O2 -ffp-contract=off -fno-fast-math).
 */
#include "fb_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <omp.h>

/* log-sum-exp of n values, shifted by their maximum (the helper of bw_oracle.c) */
static double lse(const double *x, int n)
{
    double m = -INFINITY;
    for (int k = 0; k < n; k++) if (x[k] > m) m = x[k];
    if (m == -INFINITY) return -INFINITY;
    double s = 0.0;
    for (int k = 0; k < n; k++) s += exp(x[k] - m);
    return m + log(s);
}
/* ---- forward-backward, the semantics of cv_loglik_batch / cv_posterior_batch (include/cv_b200.h) ----------------
 * The E-step of cvo_baum_welch on its own: forward and backward rows shifted by their log-sum-exp, gamma_t normalised
 * per t.  loglik_out[b] = log10 P(O_b) (-inf for P(O) = 0), post_out[x*K + i] = gamma_t(i) (rows of 0.0 for P(O) = 0;
 * may be NULL).  OpenMP over sequences; every sequence is computed by one thread on its own, so the result does not
 * depend on nthreads. */
int cvo_forward_backward(int K, int64_t M, const double *logA, const double *logB, const double *logPi,
                         const uint32_t *obs, const int64_t *seq_off, int64_t B, double *loglik_out, double *post_out,
                         int nthreads)
{
    if (K <= 0 || M <= 0 || B < 0 || !logA || !logB || !logPi || !obs || !seq_off || !loglik_out) return CVO_ERR_ARG;
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
    const size_t NA = (size_t)K * K, NB = (size_t)K * M;
    double *lA = malloc(NA * sizeof(double)), *lB = malloc(NB * sizeof(double)), *lP = malloc((size_t)K * sizeof(double));
    if (!lA || !lB || !lP) { free(lA); free(lB); free(lP); return CVO_ERR_ARG; }
    for (size_t e = 0; e < NA; e++) lA[e] = logA[e] * ln10;
    for (size_t e = 0; e < NB; e++) lB[e] = logB[e] * ln10;
    for (int e = 0; e < K; e++) lP[e] = logPi[e] * ln10;
#pragma omp parallel num_threads(nthreads)
    {
        double *la = malloc((size_t)(Tmax > 0 ? Tmax : 1) * K * sizeof(double));
        double *lb = malloc((size_t)(Tmax > 0 ? Tmax : 1) * K * sizeof(double));
        double *tmp = malloc((size_t)K * sizeof(double));
#pragma omp for schedule(static)
        for (int64_t i = 0; i < B; i++) {
            const uint32_t *o = obs + seq_off[i];
            const int64_t T = seq_off[i + 1] - seq_off[i];
            double *post = post_out ? post_out + (size_t)seq_off[i] * K : NULL;
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
            if (lp == -INFINITY) {
                loglik_out[i] = -INFINITY;
                if (post) memset(post, 0, (size_t)T * K * sizeof(double));
                continue;
            }
            loglik_out[i] = lp / ln10;
            if (!post) continue;
            for (int s = 0; s < K; s++) lb[(T - 1) * K + s] = 0.0;
            for (int64_t t = T - 1; t >= 1; t--) {
                for (int s = 0; s < K; s++) {
                    for (int j = 0; j < K; j++) tmp[j] = lA[(size_t)s * K + j] + lB[(size_t)j * M + o[t]] + lb[t * K + j];
                    lb[(t - 1) * K + s] = lse(tmp, K);
                }
                const double c = lse(lb + (t - 1) * K, K);
                for (int s = 0; s < K; s++) lb[(t - 1) * K + s] -= c;
            }
            for (int64_t t = 0; t < T; t++) {
                for (int s = 0; s < K; s++) tmp[s] = la[t * K + s] + lb[t * K + s];
                const double z = lse(tmp, K);
                for (int s = 0; s < K; s++) post[t * K + s] = exp(tmp[s] - z);
            }
        }
        free(la); free(lb); free(tmp);
    }
    free(lA); free(lB); free(lP);
    return CVO_OK;
}
