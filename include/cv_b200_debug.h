/*
 * cv_b200_debug.h -- test / bench hooks of libcv_b200.so.  NOT part of the drop-in boundary (cv_b200.h is):
 * a Rust binding of the reference's interface never needs anything declared here.  tests/, tools/ and bench.py
 * use these to force reachable launch paths, to dump solver state for parity checks and to measure the FP64 issue peak
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

/* number of chunks a batch is cut into (chunks overlap on two internal streams); -1 = automatic */
void cv_debug_set_chunks(int n);
/* batches of at most b sequences (K <= 64) use the warp-per-sequence kernel; -1 = default (8192), 0 = always the
 * tile kernel.  Exact mode only: the f32 mode always sends batches of <= 8192 sequences to that (f64) kernel. */
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
/* row blocks per group of the large-K kernel (0 = automatic: as many as the delta history fits) */
void cv_debug_set_large_group_rb(long long rb);
/* constrained solver: 1 = the K sibling leaves of the last component are evaluated by one batched launch, 0 = node by node */
void cv_debug_set_cp_leaf_batch(int on);
/* cv_loglik_batch / cv_posterior_batch: cut the batch into chunks of n sequences (0 = automatic: chunks whose history
 * and device outputs fit half the free device memory) */
void cv_debug_set_fb_chunk_seqs(int64_t n);
/* cv_decode_batch_kbest: cut the batch into chunks of n sequences (0 = automatic: chunks whose backpointers, inputs
 * and device outputs fit half the free device memory) */
void cv_debug_set_kbest_chunk_seqs(int64_t n);
/* exact decode, K <= 64, of a model of log-probabilities (every finite entry of logA / logB <= 0, |x| <= 2^64): 1 (default) =
 * f32 forward pass, backtrace that certifies every backpointer against the f64 recurrence, exact f64 re-decode of the
 * sequences it cannot certify; 0 = the f64 forward pass for every model */
void cv_debug_set_certified(int on);
/* scale of the certified backtrace's error bound: 1 (default) = the derived bound, 0 = certify every decision (the
 * f32 path is taken as it is -- NOT exact), INFINITY = certify none (every sequence goes to the f64 fallback) */
void cv_debug_set_cert_tolerance(double scale);
/* sequences the last decode call on h re-decoded in f64 after the certified backtrace; -1 = that call did not take
 * the certified path */
int64_t cv_debug_last_flagged(const cv_hmm *h);
/* route of the certified decode's f64 re-decode: 0 (default) = automatic, 1 = every flagged sequence on the tile path,
 * 2 = every one on the warp-per-sequence kernel, 3 = the n_chain longest on the warp-per-sequence kernel beside the
 * tile path, which takes the rest (n_chain is clipped to [0, flagged]) */
void cv_debug_set_fallback(int route, long long n_chain);
/* of the sequences cv_debug_last_flagged counts, the ones the warp-per-sequence kernel decoded; the rest went to the
 * tile path */
int64_t cv_debug_last_fallback_chain(const cv_hmm *h);

/* Parity hooks for the CP path: after cv_cp_solve, copy out the final delta[N*K] / psi[N*K] state and the per-node
 * upper bounds (first `cap` nodes). */
int cv_debug_cp_last_state(cv_hmm *h, double *delta_out, uint64_t *psi_out);
int cv_debug_cp_last_ub(cv_hmm *h, double *ub_out, uint64_t cap, uint64_t *n_out);

/* Launch paths the last cv_cp_solve / cv_cp_solve_dist on h took: an OR of the CV_CP_PATH_* bits below, cleared on
 * entry and set by the host at each launch site.  Tests assert them so that a case cannot drift off the path it is
 * meant to cover when a selection rule changes. */
uint32_t cv_debug_cp_last_paths(const cv_hmm *h);
#define CV_CP_PATH_SWEEP_1_2_16   (1u << 0)   /* warp-per-segment sweep, K <= 8, two segments per warp */
#define CV_CP_PATH_SWEEP_1_4_16   (1u << 1)   /* K = 9..16, two segments per warp */
#define CV_CP_PATH_SWEEP_1_6      (1u << 2)   /* K = 17..24 */
#define CV_CP_PATH_SWEEP_1_8      (1u << 3)   /* K = 25..32 */
#define CV_CP_PATH_SWEEP_2_0      (1u << 4)   /* K = 33..64, two states per lane, logA column from shared memory */
#define CV_CP_PATH_SWEEP_GENERIC  (1u << 5)   /* K > 64 */
#define CV_CP_PATH_SWEEP_FW_1_2   (1u << 6)   /* CV_CP_FULLWARP: K <= 8, one segment per warp */
#define CV_CP_PATH_SWEEP_FW_1_4   (1u << 7)   /* CV_CP_FULLWARP: K = 9..16, one segment per warp */
#define CV_CP_PATH_BT_IN_SMEM     (1u << 8)   /* logB^T staged in shared memory by the warp-per-segment sweep */
#define CV_CP_PATH_BTR_ROWS_GMEM  (1u << 9)   /* backtrack maps / fill walk psi in global memory (K too large to stage) */
#define CV_CP_PATH_BTR_CHAIN_GMEM (1u << 10)  /* backtrack entry chain walked by one thread from global memory */
#define CV_CP_PATH_SUM_LOOP       (1u << 11)  /* bound sum: one-thread loop */
#define CV_CP_PATH_SUM_BLOCKS     (1u << 12)  /* bound sum: block-structured exact-order kernels */
#define CV_CP_PATH_SUM_PREFIX     (1u << 13)  /* bound sum: block-structured, block prefixes from their own kernel */
#define CV_CP_PATH_SUM_ONE_CTA    (1u << 14)  /* bound sum: single-CTA binade scan */
#define CV_CP_PATH_LEAF_BATCH     (1u << 15)  /* the siblings of the last component evaluated as one batch */
#define CV_CP_PATH_BOUND_COPY     (1u << 16)  /* CV_CP_HOSTPOLL=0: a node's bound copied back and the stream synchronised */

/* Parity hook for the bound sum of solve_r (cp.rs:103-116): ((0.0 + v[0]) + v[1]) + ... of n host values,
 * mode 0 = one-thread loop, mode 1 = the parallel exact-order kernel; both must agree bit for bit. */
int cv_debug_ordered_sum(const double *values, int64_t n, int mode, double *out);

/* FP64 issue-rate probe used as the ALU roofline denominator: runs `iters` dependent-free DADD (mode 0) or
 * DADD+DSETP pairs (mode 1) on every SM and returns FP64 instructions per second.  Mode 25: independent DFMA chains
 * (the Baum-Welch cell), returns FMAs per second.  Any other mode is CV_ERR_ARG. */
int cv_debug_probe_fp64(int device, int mode, int iters, double *ops_per_s_out, double *ms_out);

#ifdef __cplusplus
}
#endif
#endif /* CV_B200_DEBUG_H */
