/*
 * cv_b200_debug.h -- test / bench hooks of libcv_b200.so.  NOT part of the drop-in boundary (cv_b200.h is):
 * a Rust binding of the reference's interface never needs anything declared here.  tests/, tools/ and bench.py
 * use these to force launch shapes, to dump solver state for parity checks and to measure the FP64 issue peak
 * that the roofline is quoted against.  Implemented in csrc/cv_debug.cu (setters, probe) and csrc/cv_cp.cu
 * (state dumps, ordered sum).
 */
#ifndef CV_B200_DEBUG_H
#define CV_B200_DEBUG_H

#include <stdint.h>

#include "cv_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* force the small-K launch shape, cfg = 10*S + MINB (S sequence groups of 64 per CTA, MINB co-resident CTAs per
 * SM); -1 = automatic */
void cv_debug_set_small_config(int cfg);
/* number of chunks a batch is cut into (chunks overlap on two internal streams); -1 = automatic */
void cv_debug_set_chunks(int n);
/* batches of at most b sequences (K <= 64) use the warp-per-sequence kernel; -1 = default (8192), 0 = always the
 * tile kernel */
void cv_debug_set_chain_max_batch(long long b);
/* bt_concurrent = 1 runs the backtrace kernel next to the forward kernel (tile by tile), streamed = 1 lets
 * cv_decode_batch stream its copies past ONE launch instead of launching once per chunk; -1 = leave as is */
void cv_debug_set_pipeline(int bt_concurrent, int streamed);
/* forward tile kernel: 1 (default) = balanced state split (state groups of near-equal size over slot-permuted copies
 * of logA / logB^T, no padded target states), 0 = groups of 8 states with the last one padded */
void cv_debug_set_balanced_split(int on);
/* forward tile kernel: 1 (default) = the instantiation with compile-time row pitches (tiles of 64 sequences, logA rows
 * at a pitch of 64 doubles in shared memory) whenever it keeps the occupancy, 0 = run-time pitches */
void cv_debug_set_fwd_ldc(int on);
/* forward tile kernel, balanced split with a remainder: 1 (default) = only the state groups that own one state less
 * fetch the emission rows (they are the ones that wait at the step barrier), 0 = every warp fetches a share */
void cv_debug_set_em_light(int on);
/* backtrace of the tile path: 1 (default) = four lanes per sequence (a whole history row in flight per step, no load
 * that depends on the decoded state) for batches of up to ~1300 sequences per SM, 2 = for every batch size,
 * 0 = always one thread per sequence */
void cv_debug_set_bt_split(int on);
/* streamed host path: 1 (default) = large batches with automatic chunking are cut 10 / 25 / 25 / 20 / 12 / 8 % and the long
 * sequences of the last chunk are ordered with the chunk before it, 0 = equal chunks, 2 = the uneven cut for every
 * streamed call (tests) */
void cv_debug_set_uneven_chunks(int on);
/* forward tile kernel with the f32 pre-filter (csrc/decode_prefilter.cuh) for models whose entries are all <= 0:
 * 1 = on, 0 = the plain f64 tile kernel */
void cv_debug_set_prefilter(int on);
/* row blocks per group of the large-K kernel (0 = automatic: as many as the delta history fits) */
void cv_debug_set_large_group_rb(long long rb);
/* constrained solver: 1 = the K sibling leaves of the last component are evaluated by one batched launch, 0 = node by node */
void cv_debug_set_cp_leaf_batch(int on);

/* Parity hooks for the CP path: after cv_cp_solve, copy out the final delta[N*K] / psi[N*K] state and the per-node
 * upper bounds (first `cap` nodes). */
int cv_debug_cp_last_state(cv_hmm *h, double *delta_out, uint64_t *psi_out);
int cv_debug_cp_last_ub(cv_hmm *h, double *ub_out, uint64_t cap, uint64_t *n_out);

/* Parity hook for the bound sum of solve_r (cp.rs:103-116): ((0.0 + v[0]) + v[1]) + ... of n host values,
 * mode 0 = one-thread loop, mode 1 = the parallel exact-order kernel; both must agree bit for bit. */
int cv_debug_ordered_sum(const double *values, int64_t n, int mode, double *out);

/* FP64 issue-rate probe used as the ALU roofline denominator: runs `iters` dependent-free DADD (mode 0),
 * DADD+DSETP pairs (mode 1) or the decode inner loop body (mode >= 2) on every SM and returns FP64 instructions
 * per second.  Mode 25: independent DFMA chains (the Baum-Welch cell), returns FMAs per second. */
int cv_debug_probe_fp64(int device, int mode, int iters, double *ops_per_s_out, double *ms_out);

#ifdef __cplusplus
}
#endif
#endif /* CV_B200_DEBUG_H */
