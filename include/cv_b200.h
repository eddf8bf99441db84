/*
 * cv_b200.h -- C ABI of the B200-native consistent-viterbi hot path.
 *
 * The reference (AlexandreDubray/consistent-viterbi) is one Rust binary with no
 * FFI seam; this header is the seam a maintainer would bind from Rust (see
 * INTEGRATION.md for the `extern "C"` block + build.rs).  Every entry point
 * cites the reference interface it replaces.  Plain pointers and sizes only.
 *
 * Conventions
 *   - All probabilities are log10, zero probability = -inf, exactly as the
 *     reference stores them (src/hmm/hmm.rs:192-205).
 *   - logA  [K*K]  row-major, logA[from*K + to]   (hmm.rs:12-13, a[[from,to]])
 *     logB  [K*M]  state-major, logB[state*M + o] (hmm.rs:14-15, b[state][obs]);
 *                  o = the D-dimensional observation flattened row-major over
 *                  bdims, M = prod(bdims)
 *     logPi [K]                                   (hmm.rs:16-17)
 *   - Every function returns CV_OK or a non-zero status; where the reference
 *     would panic (unwrap/assert/index) the status says which panic.  The text
 *     of the last error of the calling thread is cv_last_error().
 *   - There is NO CPU fallback: without a CUDA device every compute entry point
 *     returns CV_ERR_CUDA.
 */
#ifndef CV_B200_H
#define CV_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CV_OK          0
#define CV_ERR_EMPTY   1  /* reference panics: empty sequence / empty super-sequence      */
#define CV_ERR_NAN     2  /* reference panics: argmax().unwrap() on NaN (model has NaN/+inf) */
#define CV_ERR_ARG     3  /* bad argument; observation >= M or comp id >= ncomp (index panic) */
#define CV_ERR_ASSERT  4  /* reference assert!(obj > self.best_obj) fires (cp.rs:87)        */
#define CV_ERR_CUDA    5  /* CUDA runtime error / no device                                */
#define CV_ERR_OOM     6  /* device or host allocation failed                              */
#define CV_ERR_UNSUPPORTED 7 /* shape outside what the kernels cover (see DESIGN.md)        */

typedef struct cv_hmm cv_hmm;   /* device-resident model + its workspaces, one device */

/* ---- model ---------------------------------------------------------------
 * Replaces: struct HMM<D>{a,b,pi} (hmm.rs:10-18) as loaded by HMM::from_json
 * (hmm.rs:242-245).  Uploads the model to `device` (-1 = current device),
 * builds the padded/transposed device layouts the kernels read.  NaN or +inf
 * entries are rejected with CV_ERR_NAN (the reference would panic later inside
 * argmax).  A finite entry with |x| > 2^900 is rejected with CV_ERR_UNSUPPORTED:
 * with |x| <= 2^900 no sum of fewer than 2^63 entries reaches 2^1024, so no
 * finite sum a kernel forms (decode, CP, CFN) overflows to +-inf and every -inf
 * means an impossible event, as the backtraces rely on.  Real log10
 * probabilities are >= -324, far inside the bound. */
int  cv_hmm_create(int K, int D, const uint64_t *bdims, const double *logA,
                   const double *logB, const double *logPi, int device,
                   cv_hmm **out);
void cv_hmm_destroy(cv_hmm *h);
int  cv_hmm_nstates(const cv_hmm *h);          /* HMM::nstates (hmm.rs:207-209) */
int64_t cv_hmm_nobs(const cv_hmm *h);          /* M = prod(bdims)               */

/* ---- plain Viterbi, batched ------------------------------------------------
 * Replaces: B calls of viterbi::decode(sequence, hmm) -> Array1<usize>
 * (src/viterbi_solver/viterbi.rs:5-32), association order (delta + a) + b,
 * pi and the first observation ignored, lowest-index argmax.
 *   obs_flat[N]   flattened observations of all sequences back to back
 *   seq_off[B+1]  offsets into obs_flat / path_out (seq_off[0] = 0)
 *   path_out[N]   decoded state of every element
 *   score_out[B]  delta[T-1][end_state] of every sequence (may be NULL)
 * HOST pointers (pinned memory gives full PCIe speed; see cv_host_alloc).
 * An empty sequence returns CV_ERR_EMPTY (reference: usize underflow panic). */
int cv_decode_batch(cv_hmm *h, const uint32_t *obs_flat, const int64_t *seq_off,
                    int64_t B, uint32_t *path_out, double *score_out);

/* ---- k-best (list) Viterbi, batched ------------------------------------------
 * The k highest-scoring state paths of every sequence under the recurrence of cv_decode_batch (pi and o_0 ignored,
 * every fl one binary64 add).  The score of a path s_0 .. s_{T-1} is the left-to-right rounded sum
 *   v_0 = 0,  v_t = fl(fl(v_{t-1} + a[s_{t-1}][s_t]) + b[s_t][o_t]),  score = v_{T-1}.
 * The list at (t, i) holds at most k entries, each a value and a backpointer (j, r).  At t = 0 every state has one
 * entry, value 0.0.  For t >= 1 the candidates are every entry (j, r) of row t-1, with c = fl(L[t-1][j][r] + a[j][i]):
 *   - b[i][o_t] > -inf: the first min(k, #candidates) candidates in the order (c descending, j ascending, r ascending),
 *     compared with IEEE > (-0.0 and +0.0 tie); each entry's value is fl(c + b[i][o_t]);
 *   - b[i][o_t] = -inf: the first min(k, #candidates) candidates in (j ascending, r ascending) order, every value -inf
 *     (the psi = 0 rule of the plain decode).
 * Ranks 0 .. k-1 of a sequence are the first k entries (i, r) of row T-1 in the order (value descending, i ascending,
 * r ascending), each backtraced through the stored (j, r).  Hence:
 *   - rank 0 is cv_decode_batch's path and score, byte for byte (fl(x + a) is monotone, so (j, r > 0) never beats
 *     (j, 0)), including sequences whose every path is -inf and exact ties;
 *   - every score is its path's rounded sum, scores do not increase with rank, the paths are pairwise distinct, and
 *     the multiset of the scores is the top k of the scores of all K^T paths;
 *   - a sequence has min(k, K^T) paths; a rank at or beyond that count is "no path": score -inf and every path
 *     element 0xFFFFFFFF.
 *   path_out[k*N]   rank-major: plane r (path_out + r*N) is laid out as cv_decode_batch's path_out
 *   score_out[k*B]  rank-major: plane r (score_out + r*B) as cv_decode_batch's score_out (may be NULL)
 * A sequence's outputs do not depend on the batch it is in, its place there or how the call cuts the batch into
 * chunks; two calls with the same inputs return the same bytes.  Any model cv_hmm_create accepts.
 *   B = 0: CV_OK, nothing written   CV_ERR_ARG NULL h / obs_flat / seq_off / path_out, seq_off[0] != 0, an observation
 *   >= M or k < 1 (checked on the host before any launch)   CV_ERR_EMPTY an empty sequence   CV_ERR_UNSUPPORTED K > 64
 *   or k > 32   CV_ERR_CUDA no device.  HOST pointers, as for cv_decode_batch. */
int cv_decode_batch_kbest(cv_hmm *h, const uint32_t *obs_flat, const int64_t *seq_off, int64_t B, int k,
                          uint32_t *path_out /* [k*N] */, double *score_out /* [k*B], may be NULL */);

/* Same call with narrow HOST formats: u16 observations (needs M <= 65536) and u8 states (needs K <= 256; implemented
 * for K <= 64).  A third of the bytes cross PCIe (POS shape: 216 MB -> 75 MB per million sentences); the kernels read
 * and write the narrow types directly.  cv_decode_batch stays the reference-shaped entry. */
int cv_decode_batch_u16u8(cv_hmm *h, const uint16_t *obs_flat, const int64_t *seq_off,
                          int64_t B, uint8_t *path_out, double *score_out);

/* OPTIONAL f32 mode -- not the parity path.  The same recurrence with the model rounded to f32 once and every add an
 * IEEE binary32 add; the returned path is the exact optimum of that f32 recurrence (first-maximum backpointers),
 * score_out[b] its f32 score widened to double (the sign of a zero score is unspecified).  The path can differ from
 * the f64 path where candidates are within f32 rounding of each other.  For models whose entries are all <= 0 the
 * score of a sequence of T steps is within about 2T * 2^-24 relative of the f64 score of cv_decode_batch (measured on
 * random models, K = 45: 4.8e-7 at T = 80, 1.9e-6 at T = 2000, 9.5e-6 at T = 20000).  About 3-4x the throughput of the
 * exact mode (packed FADD2 / 3-input FMNMX3).  K <= 64; a model with a finite entry |x| > 2^64 is CV_ERR_UNSUPPORTED
 * (f32 sums could reach FLT_MAX).  A call of <= 8192 sequences is decoded by the exact f64 warp-per-sequence kernel,
 * a larger call in f32 throughout.  HOST pointers / DEVICE pointers as for cv_decode_batch(_dev). */
int cv_decode_batch_f32(cv_hmm *h, const uint32_t *obs_flat, const int64_t *seq_off,
                        int64_t B, uint32_t *path_out, double *score_out);
int cv_decode_batch_dev_f32(cv_hmm *h, const uint32_t *d_obs_flat, const int64_t *d_seq_off,
                            int64_t B, int64_t N, int64_t max_len, uint32_t *d_path_out,
                            double *d_score_out, void *stream, int sync_status);

/* Same call, and the device copies of the results are left in the caller's DEVICE buffers d_path_keep[N] /
 * d_score_keep[B] as well (e.g. rows of an all-gather buffer: a multi-GPU caller decodes its slice from host memory
 * and runs the device-side collective without uploading the paths again).  The device buffers are complete when the
 * call returns. */
int cv_decode_batch_keep(cv_hmm *h, const uint32_t *obs_flat, const int64_t *seq_off,
                         int64_t B, uint32_t *path_out, double *score_out,
                         uint32_t *d_path_keep, double *d_score_keep);

/* Same, with every buffer already resident on the model's device; enqueued on
 * `stream` (a cudaStream_t, NULL = default stream) without host sync, except
 * that the status word is read back when `sync_status` != 0.
 * N = d_seq_off[B]; max_len = an upper bound on the sequence lengths (sizes the workspace, and the ordering of the
 * batch by length only looks at the bits such a length can have), <= 0 = not known (one extra synchronisation reads it
 * back).  A sequence longer than a positive max_len is CV_ERR_ARG.
 * K <= 64, more than 8192 sequences, a model of log-probabilities (every finite logA / logB entry <= 0, |x| <= 2^64):
 * the call also waits once for `stream` -- the exact result comes from an f32 forward pass whose backpointers are
 * certified against the f64 recurrence, and the host reads back how many sequences need an f64 re-decode. */
int cv_decode_batch_dev(cv_hmm *h, const uint32_t *d_obs_flat, const int64_t *d_seq_off,
                        int64_t B, int64_t N, int64_t max_len, uint32_t *d_path_out,
                        double *d_score_out, void *stream, int sync_status);

/* cv_decode_batch_dev with u8 states in d_path_out[N] (K <= 64): a quarter of the bytes for a following all-gather of
 * the decoded paths across GPUs. */
int cv_decode_batch_dev_u8(cv_hmm *h, const uint32_t *d_obs_flat, const int64_t *d_seq_off,
                           int64_t B, int64_t N, int64_t max_len, uint8_t *d_path_out,
                           double *d_score_out, void *stream, int sync_status);

/* ---- constrained decode ----------------------------------------------------
 * Replaces: CPSolver::new(&hmm, &super_seq) + Solver::solve + get_solution +
 * get_objective + get_explored_nodes (src/viterbi_solver/cp.rs:20-152,
 * src/viterbi_solver.rs:11-16), association order delta + (a + b), argmax on
 * delta + a, clamp = row reset to {-inf.., 0.0 at the chosen state}.
 *   obs[N]          flattened observation of each super-sequence element, in the
 *                   (reordered) order SuperSequence holds them
 *   is_seq_start[N] 1 iff MetaElements.t == 0 (viterbi_solver/utils.rs:11)
 *   comp[N]         constraint_component of ACTIVE elements, -1 otherwise
 *                   (is_constrained(), viterbi_solver/utils.rs:44-46)
 *   ncomp           SuperSequence::number_constraints() (utils.rs:200-202)
 *   max_nodes       0 = unlimited (reference); else stop opening nodes once
 *                   explored == max_nodes
 *   sol_out[N]      get_solution()      obj_out  get_objective()
 *   explored_out    get_explored_nodes() steps_out forward sweep steps executed
 * HOST pointers.  Any K that fits the kernels' shared memory (K <= ~3000); K <= 64 takes the tuned kernels. */
int cv_cp_solve(cv_hmm *h, const uint32_t *obs, const uint8_t *is_seq_start,
                const int32_t *comp, int64_t N, int32_t ncomp, uint64_t max_nodes,
                uint64_t *sol_out, double *obj_out, uint64_t *explored_out,
                uint64_t *steps_out);

/* ---- constrained decode sharded over the GPUs of one NVSwitch box ------------
 * One process per GPU.  The super-sequence is cut at positions of component 0 (no sweep of cp.rs:47-60 crosses
 * such a position, cp.rs:48), every rank sweeps its own rows; per B&B node the ranks exchange the bound terms
 * of cp.rs:103-116 by storing them into each other's term lists over NVLink (CUDA-IPC peer mappings, one flag
 * per rank), then every rank runs the same exact-order sum and takes the same decision.  Results are
 * bit-identical to cv_cp_solve on every rank.  When component 0 has fewer than nranks-1 usable positions every
 * rank solves the whole problem itself (replicas).
 *   cv_cp_dist_create   allocates this rank's exchange buffer (capacity: super-sequences of up to cap_N elements
 *                       with up to cap_terms clamped positions) and returns its CV_IPC_HANDLE_BYTES-byte IPC handle
 *   cv_cp_dist_connect  all_handles = the nranks handles in rank order (the host exchanges them: MPI,
 *                       torch.distributed, a file -- any transport)
 *   cv_cp_solve_dist    collective: every rank calls it with the same arguments; all ranks return the full result
 * A rank that fails leaves its peers waiting for at most a few seconds before they fail with CV_ERR_CUDA. */
#define CV_IPC_HANDLE_BYTES 64
typedef struct cv_cp_dist cv_cp_dist;
int  cv_cp_dist_create(cv_hmm *h, int rank, int nranks, int64_t cap_N, int64_t cap_terms,
                       void *handle_out, cv_cp_dist **out);
int  cv_cp_dist_connect(cv_cp_dist *d, const void *all_handles);
void cv_cp_dist_destroy(cv_cp_dist *d);
int  cv_cp_solve_dist(cv_cp_dist *d, const uint32_t *obs, const uint8_t *is_seq_start,
                      const int32_t *comp, int64_t N, int32_t ncomp, uint64_t max_nodes,
                      uint64_t *sol_out, double *obj_out, uint64_t *explored_out,
                      uint64_t *steps_out);
/* the row cuts cv_cp_solve_dist uses: cuts_out[nranks + 1], rank r owns rows [cuts[r], cuts[r+1]); when the
 * problem cannot be cut, cuts = {0, N, N, ...} (replicas).  Pure host code, no device needed. */
int  cv_cp_plan_cuts(const int32_t *comp, int64_t N, int nranks, int64_t *cuts_out);

/* ---- CFN cost tables -------------------------------------------------------------
 * Replaces the numeric part of write_cfn(hmm, super_seq, ..) (src/viterbi_solver/cfn.rs:82-167): the boundaries
 * between constraint components, the K*K clamped longest_path runs (cfn.rs:11-35) of every consecutive boundary
 * pair accumulated into the k*k cost tables with the reference's `== 0.0 => assign, else +=` rule, the unary
 * start / end costs (cfn.rs:37-80), the lower bound and the -inf -> lower_bound patch.  Arithmetic order
 * (max_j (row[j] + tr_j)) + emit.  obs / is_seq_start / comp as for cv_cp_solve; k = number_constraints().
 *   cost_tables[k*k*K*K]  [c1][c2][n1][n2]     unary[k*K]     lower_bound_out, nboundaries_out, device_ms_out may be NULL
 * No constrained element => CV_ERR_EMPTY (the reference unwraps None).  K <= 64.  The .cfn text file itself
 * (cfn.rs:169-205) is host formatting of these arrays and is left to the caller.  HOST pointers. */
int cv_cfn_tables(cv_hmm *h, const uint32_t *obs, const uint8_t *is_seq_start, const int32_t *comp,
                  int64_t N, int32_t k, double *cost_tables, double *unary, double *lower_bound_out,
                  int64_t *nboundaries_out, double *device_ms_out);

/* ---- supervised maximum-likelihood estimation --------------------------------
 * Replaces: HMM::maximum_likelihood_estimation(&mut self, sequences, tags) followed by HMM::log
 * (src/hmm/hmm.rs:30-62,192-205).  a [K*K], b [K*M], pi [K] hold the model the reference would call it on --
 * HMM::new's random model (hmm.rs:22-28), or zeros for a plain count-based estimate -- as PROBABILITIES on entry;
 * on exit they hold what the reference holds after log(): ln(x)/ln(10), -inf for 0.  The events are counted on
 * the device; given the same initial model the result is the reference's bit for bit (each entry is its initial
 * value with `+= 1.0` applied count times, then the reference's divisions).  tags < 0 = None.
 *   CV_ERR_EMPTY  an empty sequence (tag[0] / len()-1 panics)   CV_ERR_ARG  a None tag, tag >= K, observation >= M
 * count_ms_out (may be NULL): device time of the counting kernels.  HOST pointers. */
int cv_mle(int K, int D, const uint64_t *bdims, double *a, double *b, double *pi,
           const uint32_t *obs_flat, const int32_t *tags_flat, const int64_t *seq_off,
           int64_t B, int device, double *count_ms_out);

/* ---- unsupervised training: Baum-Welch (EM) ------------------------------------
 * The counterpart of HMM::train (hmm.rs:69-190).  The semantics below are defined by this library (textbook
 * Baum-Welch over multiple observation sequences, Rabiner 1989); they are not a restatement of hmm.rs, whose random
 * start makes bit parity impossible anyway.  One iteration from model theta (probabilities p = 10^log10 entry):
 *   P(O) = sum over paths of pi[s0] b[s0][o0] prod_{t>=1} a[s_{t-1}][s_t] b[s_t][o_t]   (unlike cv_decode_batch,
 *          pi and the first observation count)
 *   gamma_t(i) = P(s_t = i | O), xi_t(i,j) = P(s_{t-1} = i, s_t = j | O), summed over the contributing sequences:
 *   pi'[i]   = sum gamma_0(i) / (number of contributing sequences)
 *   a'[i][j] = sum_{t=1..T-1} xi_t(i,j) / sum_{t=0..T-2} gamma_t(i)
 *   b'[j][m] = sum_{t: o_t = m} gamma_t(j) / sum_t gamma_t(j)
 * A zero denominator gives a zero row; a zero is written as -inf, anything else as ln(x)/ln(10).  An entry that is
 * -inf on entry stays -inf.  A sequence with P(O) = 0 under the current model (also: whose scaled forward sum
 * underflows) is not a contributing sequence: it adds nothing and is counted in *skipped_out (of the last iteration).
 * loglik_out[k] = log10 P(O | theta_k) summed over the contributing sequences, theta_k = the model BEFORE update k.
 * Runs n_iter iterations, or stops after iteration k >= 1 (its update kept) when tol > 0 and
 * loglik[k] - loglik[k-1] < tol * |loglik[k-1]|; *iters_out = iterations run.
 *   logA, logB, logPi  log10 in, log10 out, in place (layouts as above)
 *   obs_flat[N], seq_off[B+1] as for cv_decode_batch; device -1 = current device; device_ms_out may be NULL
 * Two calls with the same inputs on the same GPU return the same bytes.  K <= 64.
 *   CV_ERR_EMPTY an empty sequence   CV_ERR_ARG observation >= M, n_iter < 1, B < 1, bad sizes   CV_ERR_NAN NaN or
 *   +inf in the model   CV_ERR_UNSUPPORTED K > 64   CV_ERR_CUDA no device.  HOST pointers. */
int cv_baum_welch(int K, int D, const uint64_t *bdims, double *logA, double *logB, double *logPi,
                  const uint32_t *obs_flat, const int64_t *seq_off, int64_t B,
                  int n_iter, double tol, int device,
                  double *loglik_out /* [n_iter] */, int *iters_out,
                  int64_t *skipped_out /* last iteration */, double *device_ms_out /* may be NULL */);

/* ---- forward-backward inference: log-likelihood, posterior marginals, posterior decoding --------
 * The model is the handle's log10 entries read as probabilities 10^x; as in cv_baum_welch (and unlike
 * cv_decode_batch) pi and the first observation count.  For sequence b with positions x = seq_off[b] + t:
 *   loglik_out[b]  = log10 P(O_b), P(O) as defined at cv_baum_welch
 *   post_out[x*K + i] = gamma_t(i) = P(s_t = i | O_b)        (row x = position x, in the caller's order)
 *   path_out[x]    = the lowest i at which row x of the posterior reaches its maximum (maximum posterior marginal)
 *   pmax_out[x]    = that maximum
 * path and pmax are taken from the same values post_out receives, so a call with post_out = NULL returns the same
 * path.  Any output of cv_posterior_batch may be NULL; cv_loglik_batch needs loglik_out.
 * A sequence with P(O) = 0 (also: whose scaled forward sum underflows, the rule by which cv_baum_welch skips a
 * sequence) gets loglik -inf, posterior rows of 0.0, path 0 and pmax 0.0; the other sequences are unaffected.
 * A sequence's outputs are the same bytes whatever batch it is in, wherever it is in that batch and however the call
 * cuts the batch into chunks: nothing is reduced across sequences.  Two calls with the same inputs return the same
 * bytes, and the loglik_out of cv_posterior_batch is the same bytes as that of cv_loglik_batch.
 * Probabilities 10^x must not overflow: a model with a finite entry x > 64 is CV_ERR_UNSUPPORTED.  With every entry
 * <= x the scaled forward rows sum to < K 10^(2x), the scaled backward vectors stay < 10^x and the normaliser
 * Z_t = sum_i r_t(i) beta_t(i) < K 10^(3x); at x = 64, K = 64 these are < 1e130 and < 1e194.  Models of
 * log-probabilities (entries <= 0) are never refused.
 *   B = 0: CV_OK, nothing written   CV_ERR_EMPTY an empty sequence   CV_ERR_ARG NULL model / obs_flat / seq_off
 *   (/ loglik_out for cv_loglik_batch), observation >= M (checked on the host before any launch)
 *   CV_ERR_UNSUPPORTED K > 64 or an entry beyond the bound above.  HOST pointers, as for cv_decode_batch. */
int cv_loglik_batch(cv_hmm *h, const uint32_t *obs_flat, const int64_t *seq_off, int64_t B,
                    double *loglik_out /* [B] */);
int cv_posterior_batch(cv_hmm *h, const uint32_t *obs_flat, const int64_t *seq_off, int64_t B,
                       uint32_t *path_out /* [N] may be NULL */, double *pmax_out /* [N] may be NULL */,
                       double *post_out /* [N*K] may be NULL */, double *loglik_out /* [B] may be NULL */);

/* ---- plumbing --------------------------------------------------------------*/
const char *cv_last_error(void);
/* kernels launched by this library in this process (bench.py "gpu_launches") */
uint64_t cv_launch_count(void);
/* device time (ms, CUDA events on the library's stream) of the forward kernel(s)
 * of the most recent cv_decode_batch / cv_decode_batch_dev / cv_cp_solve call
 * when timing was enabled with cv_set_timing(1). */
void   cv_set_timing(int on);
double cv_last_kernel_ms(const cv_hmm *h);     /* forward (dominant) kernel */
double cv_last_backtrace_ms(const cv_hmm *h);  /* end-state + backtrace kernel */
/* pinned host memory helpers */
void *cv_host_alloc(uint64_t bytes);
void  cv_host_free(void *p);
/* Test / bench hooks (launch-shape overrides, parity dumps, the FP64 issue-rate probe) are declared in
 * cv_b200_debug.h; nothing a caller of this header needs. */

#ifdef __cplusplus
}
#endif
#endif /* CV_B200_H */
