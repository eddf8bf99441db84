/*
 * bw_oracle.h -- CPU oracle of cv_baum_welch (include/cv_b200.h).  TEST INFRASTRUCTURE ONLY: the product path never
 * links or calls it.  Status codes are those of cv_oracle.h.
 *
 * The Baum-Welch semantics are the ones documented at cv_baum_welch; they are defined by this project and are not a
 * restatement of the reference's HMM::train (hmm.rs:69-190), whose random start rules out bit parity.
 */
#ifndef BW_ORACLE_H
#define BW_ORACLE_H

#include <stdint.h>

#include "cv_oracle.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Baum-Welch (EM) with the semantics of cv_baum_welch: log-space restatement (log-sum-exp), f64, OpenMP over
 * sequences with nthreads threads.  logA/logB/logPi log10 in and out, loglik_out[n_iter], *iters_out, *skipped_out
 * (last iteration). */
int cvo_baum_welch(int K, int64_t M, double *logA, double *logB, double *logPi, const uint32_t *obs,
                   const int64_t *seq_off, int64_t B, int n_iter, double tol, double *loglik_out, int *iters_out,
                   int64_t *skipped_out, int nthreads);

#ifdef __cplusplus
}
#endif
#endif
