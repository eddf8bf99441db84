/*
 * kbest_oracle.c -- CPU oracle of cv_decode_batch_kbest (k-best list Viterbi), see kbest_oracle.h.
 *
 * TEST INFRASTRUCTURE ONLY, like fb_oracle.c.  A literal restatement of the contract in include/cv_b200.h: the list
 * of (t, i) is every candidate (j, r) of row t-1 sorted by (c descending, j ascending, r ascending) and cut to k.  It
 * deliberately builds and sorts all candidates instead of inserting with an early exit as the kernel does, so that
 * the two stay independent.  Compile WITHOUT fast-math and without FMA contraction (kbest.mk).
 */
#include "kbest_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <omp.h>

typedef struct {
    double key;   /* c (row t) or the entry's value (end selection) */
    int j, r;     /* predecessor state and its rank (row t); state and rank (end selection) */
} Cand;

/* a precedes b in the order (key descending, j ascending, r ascending); keys are compared with IEEE < and > so that
 * -0.0 and +0.0 tie */
static int precedes(const Cand *a, const Cand *b)
{
    if (a->key > b->key) return 1;
    if (a->key < b->key) return 0;
    return a->j < b->j || (a->j == b->j && a->r < b->r);
}

/* moves the first min(k, n) candidates of that order, in order, to the front of c (selection sort cut at k) */
static int select_first(Cand *c, int n, int k)
{
    const int keep = n < k ? n : k;
    for (int q = 0; q < keep; q++) {
        int best = q;
        for (int x = q + 1; x < n; x++)
            if (precedes(&c[x], &c[best])) best = x;
        const Cand tmp = c[q]; c[q] = c[best]; c[best] = tmp;
    }
    return keep;
}

int cvo_decode_batch_kbest(int K, int64_t M, const double *logA, const double *logB, const uint32_t *obs,
                           const int64_t *seq_off, int64_t B, int k, uint32_t *path_out, double *score_out,
                           int nthreads)
{
    if (K <= 0 || M <= 0 || B < 0 || k < 1 || !logA || !logB || !obs || !seq_off || !path_out) return CVO_ERR_ARG;
    for (int64_t b = 0; b < B; b++)
        if (seq_off[b + 1] <= seq_off[b]) return CVO_ERR_EMPTY;
    const int64_t N = seq_off[B];
    for (int64_t x = 0; x < N; x++)
        if ((int64_t)obs[x] >= M) return CVO_ERR_ARG;
    int64_t Tmax = 0;
    for (int64_t b = 0; b < B; b++) if (seq_off[b + 1] - seq_off[b] > Tmax) Tmax = seq_off[b + 1] - seq_off[b];
    if (nthreads < 1) nthreads = 1;
    const size_t row = (size_t)K * k;      /* entries of one position: [i][r] */
#pragma omp parallel num_threads(nthreads)
    {
        double *val = malloc((size_t)Tmax * row * sizeof(double));
        int *bj = malloc((size_t)Tmax * row * sizeof(int)), *br = malloc((size_t)Tmax * row * sizeof(int));
        Cand *cand = malloc((size_t)K * row * sizeof(Cand));
#pragma omp for schedule(dynamic, 16)
        for (int64_t b = 0; b < B; b++) {
            const int64_t off = seq_off[b], T = seq_off[b + 1] - off;
            int n = 1;                                      /* entries per state in the current row */
            for (int i = 0; i < K; i++) val[(size_t)i * k] = 0.0;
            for (int64_t t = 1; t < T; t++) {
                const double *pv = val + (size_t)(t - 1) * row;
                double *cv = val + (size_t)t * row;
                int *cj = bj + (size_t)t * row, *cr = br + (size_t)t * row;
                const uint32_t o = obs[off + t];
                int ncand = 0;
                for (int i = 0; i < K; i++) {
                    const double e = logB[(size_t)i * M + o];
                    ncand = 0;
                    for (int j = 0; j < K; j++)
                        for (int r = 0; r < n; r++) {
                            cand[ncand].key = pv[(size_t)j * k + r] + logA[(size_t)j * K + i];
                            cand[ncand].j = j; cand[ncand].r = r;
                            ncand++;
                        }
                    /* b = -inf: the (j, r) order in which the candidates were built */
                    const int keep = e > -INFINITY ? select_first(cand, ncand, k) : (ncand < k ? ncand : k);
                    for (int q = 0; q < keep; q++) {
                        cv[(size_t)i * k + q] = e > -INFINITY ? cand[q].key + e : -INFINITY;
                        cj[(size_t)i * k + q] = cand[q].j;
                        cr[(size_t)i * k + q] = cand[q].r;
                    }
                }
                n = ncand < k ? ncand : k;
            }
            /* end selection: every entry (i, r) of row T-1 by (value descending, i ascending, r ascending) */
            const double *lv = val + (size_t)(T - 1) * row;
            int ne = 0;
            for (int i = 0; i < K; i++)
                for (int r = 0; r < n; r++) { cand[ne].key = lv[(size_t)i * k + r]; cand[ne].j = i; cand[ne].r = r; ne++; }
            select_first(cand, ne, k);
            for (int q = 0; q < k; q++) {
                uint32_t *p = path_out + (size_t)q * N + off;
                if (q >= ne) {
                    if (score_out) score_out[(size_t)q * B + b] = -INFINITY;
                    for (int64_t t = 0; t < T; t++) p[t] = 0xFFFFFFFFu;
                    continue;
                }
                if (score_out) score_out[(size_t)q * B + b] = cand[q].key;
                int i = cand[q].j, r = cand[q].r;
                p[T - 1] = (uint32_t)i;
                for (int64_t t = T - 1; t >= 1; t--) {
                    const size_t e = (size_t)t * row + (size_t)i * k + r;
                    i = bj[e]; r = br[e];
                    p[t - 1] = (uint32_t)i;
                }
            }
        }
        free(val); free(bj); free(br); free(cand);
    }
    return CVO_OK;
}
