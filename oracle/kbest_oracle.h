/*
 * kbest_oracle.h -- CPU oracle of cv_decode_batch_kbest (include/cv_b200.h).  TEST INFRASTRUCTURE ONLY: the product
 * path never links or calls it.  Status codes are those of cv_oracle.h.
 */
#ifndef KBEST_ORACLE_H
#define KBEST_ORACLE_H

#include <stdint.h>

#include "cv_oracle.h"

#ifdef __cplusplus
extern "C" {
#endif

/* k-best Viterbi with the contract of cv_decode_batch_kbest, restated literally: every candidate of (t, i) is built,
 * sorted by the stated key and cut to k.  path_out[k*N] and score_out[k*B] are rank-major planes; ranks beyond a
 * sequence's min(k, K^T) paths get score -inf and path elements 0xFFFFFFFF.  OpenMP over sequences with nthreads
 * threads; the result does not depend on nthreads. */
int cvo_decode_batch_kbest(int K, int64_t M, const double *logA, const double *logB, const uint32_t *obs,
                           const int64_t *seq_off, int64_t B, int k, uint32_t *path_out, double *score_out,
                           int nthreads);

#ifdef __cplusplus
}
#endif
#endif
