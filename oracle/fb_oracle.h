/*
 * fb_oracle.h -- CPU oracle of cv_loglik_batch / cv_posterior_batch (include/cv_b200.h).  TEST INFRASTRUCTURE ONLY:
 * the product path never links or calls it.  Status codes are those of cv_oracle.h.
 */
#ifndef FB_ORACLE_H
#define FB_ORACLE_H

#include <stdint.h>

#include "cv_oracle.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Forward-backward with the semantics of cv_loglik_batch / cv_posterior_batch: the log-space E-step of cvo_baum_welch
 * (bw_oracle.h) per sequence.  loglik_out[B] = log10 P(O) (-inf when P(O) = 0), post_out[N*K] (may be NULL) =
 * gamma_t(i) per position, rows of 0.0 when P(O) = 0.  OpenMP over sequences with nthreads threads. */
int cvo_forward_backward(int K, int64_t M, const double *logA, const double *logB, const double *logPi,
                         const uint32_t *obs, const int64_t *seq_off, int64_t B, double *loglik_out, double *post_out,
                         int nthreads);

#ifdef __cplusplus
}
#endif
#endif
