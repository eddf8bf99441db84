// cv_internal.cuh -- what the translation units of libcv_b200.so share: the model handle, device buffers, error
// reporting and the tuning block.  Not part of the ABI (include/cv_b200.h is; include/cv_b200_debug.h declares the
// test / bench hooks).
#pragma once

#include "../../include/cv_b200.h"
#include "../../include/cv_b200_debug.h"

#include <cuda_runtime.h>

#include "common.cuh"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>
#include <vector>

namespace cvb {

// ---- errors, counters --------------------------------------------------------------------------------------------
int fail(int code, const char *fmt, ...);          // records the calling thread's error text, returns `code`
extern std::atomic<uint64_t> g_launches;           // kernels launched by this library (cv_launch_count)
extern std::atomic<int> g_timing;                  // cv_set_timing

#define CUDA_TRY(expr)                                                                         \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            int _c = (_e == cudaErrorMemoryAllocation) ? CV_ERR_OOM : CV_ERR_CUDA;             \
            return ::cvb::fail(_c, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
        }                                                                                      \
    } while (0)

int check_device(int device);

// ---- tuning block ---------------------------------------------------------------------------------------------------
// Defaults are what the library ships with.  The environment is read ONCE, when the library is loaded (never on a
// launch path); tests and bench.py change single fields through include/cv_b200_debug.h.
struct Tuning {
    int chunks = -1;               // chunks a host batch is cut into, -1 = automatic             (cv_debug_set_chunks, CV_CHUNKS)
    long long chain_max_b = -1;    // batches up to this size use the warp-per-sequence kernel, -1 = 8192
    int bt_concurrent = 1;         // backtrace next to the forward kernel                        (CV_BT_CONCURRENT)
    int streamed = 1;              // host copies streamed past one launch                        (CV_STREAMED)
    int balanced_split = 1;        // forward tile kernel: state groups of near-equal size, no padded states (CV_BALANCED)
    int fwd_ldc = 1;               // forward tile kernel with compile-time row pitches (tiles of 64, logA pitch 64) when it costs no occupancy (CV_FWD_LDC)
    int em_light = 1;              // uneven balanced split: only the lighter state groups fetch the emission rows (CV_EM_LIGHT)
    int bt_split = 1;              // backtrace with four lanes per sequence (backtrace_split_kernel) where it applies (CV_BT_SPLIT)
    int uneven_chunks = 1;         // streamed host path, automatic chunking: 10/25/25/20/12/8 % with the last chunk's long sequences promoted (CV_UNEVEN_CHUNKS)
    int long_pct = 0;              // long-sequence split: limit in % of the tile-steps per resident CTA, 0 = automatic (70 / 45) (CV_LONG_PCT)
    int long_split = 1;            // very long sequences of a short batch go to the warp-per-sequence kernel (CV_LONG_SPLIT)
    int debug = 0;                 // print launch shapes                                         (CV_DEBUG)
    int bt_prof = 0, e2e_prof = 0; // print pipeline timelines                                    (CV_BT_PROF, CV_E2E_PROF)
    long long large_group_rb = 0;  // row blocks per group of the large-K kernel, 0 = automatic    (CV_LARGE_GROUP_RB)
    long long fb_chunk_seqs = 0;   // sequences per chunk of cv_loglik_batch / cv_posterior_batch, 0 = automatic (cv_debug_set_fb_chunk_seqs)
    long long kbest_chunk_seqs = 0; // sequences per chunk of cv_decode_batch_kbest, 0 = automatic (cv_debug_set_kbest_chunk_seqs)
    int cp_fullwarp = 0, cp_prof = 0, cp_sum = -1, cp_hostpoll = 1, cp_leaf_batch = 1;   // constrained solver (CV_CP_*)
    int certified = 1;             // eligible models: f32 forward pass + certified backtrace + exact fallback (cv_debug_set_certified)
    double cert_tol = 1.0;         // scale of the certified backtrace's error bound (cv_debug_set_cert_tolerance)
    int fb_route = 0;              // certified fallback: 0 = automatic, 1 = tiles, 2 = warp kernel, 3 = the fb_chain longest on the warp kernel (cv_debug_set_fallback)
    long long fb_chain = 0;
};
extern Tuning g_tune;

// ---- device buffer that only grows ---------------------------------------------------------------------------------
struct DevBuf {
    void *p = nullptr;
    size_t bytes = 0;
    int ensure(size_t need)
    {
        if (need <= bytes) return CV_OK;
        if (p) cudaFree(p);
        p = nullptr; bytes = 0;
        size_t want = need + need / 8;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            cudaGetLastError();
            e = cudaMalloc(&p, need);
            want = need;
        }
        if (e != cudaSuccess) { p = nullptr; return fail(CV_ERR_OOM, "cudaMalloc(%zu) failed: %s", need, cudaGetErrorString(e)); }
        bytes = want;
        return CV_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
};

// ---- fixed layouts: the words of a decode workspace's misc buffer and the handle's pinned host block -----------------
constexpr int STREAM_MAX_CHUNKS = 16;   // chunks of the streamed host path (cv_api.cu, decode_streamed)

// u32 words of cv_hmm::DecodeWs::misc (MISC_BYTES, zeroed before the keys kernel of every chunk)
enum MiscWord : int {
    MISC_COUNTER = 0,         // tile counter of the forward / warp-per-sequence kernel; words 0-1: the large-K item counter (u64)
    MISC_LONG_COUNTER = 8,    // tile counter of the long-sequence split's warp-per-sequence kernel
    MISC_LONG_COUNT = 9,      // sequences the long-sequence split moved (LongSplit::n_long)
    MISC_CERT = 10,           // [4] certified backtrace: flagged sequences, their longest length, their elements (u64)
    MISC_CERT_COUNTER = 14,   // tile counter of certified_fallback's warp-per-sequence kernel
    MISC_STATUS = 16,         // device status (int)
    MISC_MAX_LEN = 17,        // longest length, found by the streamed path's keys kernel
    MISC_ARRIVED = 32,        // streamed path: chunks whose observations have arrived
    MISC_CHUNK_DONE = 33,     // streamed path: [STREAM_MAX_CHUNKS] finished sequences per chunk
};
constexpr size_t MISC_BYTES = 256;
static_assert(MISC_CERT % 2 == 0, "the certified element count at MISC_CERT + 2 is a u64");
static_assert(MISC_MAX_LEN == MISC_STATUS + 1, "decode_streamed reads the status and the longest length in one copy");
static_assert(sizeof(unsigned int) * (MISC_CHUNK_DONE + STREAM_MAX_CHUNKS) <= MISC_BYTES, "chunk_done lies inside misc");

// byte offsets into cv_hmm::pinned_status (PIN_BYTES of pinned host memory)
enum PinnedAt : size_t {
    PIN_CP_BOUND = 8,     // double[3] constrained solver: a node's bound, the peer-timeout flag, the node's sequence number
    PIN_STATUS = 32,      // int[2] decode status words of the two workspace sets (decode_streamed: status, longest length)
    PIN_CERT = 64,        // u32[4] the MISC_CERT words (certified_fallback)
    PIN_LEAF_UB = 1024,   // double[K] leaf-batch bounds of the constrained solver, K <= SMALL_K_MAX
    PIN_BYTES = 2048,
};
static_assert(PIN_CP_BOUND + 3 * sizeof(double) <= PIN_STATUS && PIN_STATUS + 2 * sizeof(int) <= PIN_CERT &&
              PIN_CERT + 4 * sizeof(unsigned int) <= PIN_LEAF_UB && PIN_LEAF_UB + SMALL_K_MAX * sizeof(double) <= PIN_BYTES,
              "the pinned words do not overlap");

}  // namespace cvb

// ---- model handle (opaque in the ABI) ------------------------------------------------------------------------------
struct cv_hmm {
    int device = 0, K = 0, Kp = 0, G = 0, D = 0, num_sms = 0;
    int64_t M = 1;
    // device model
    double *dA = nullptr;    // [K][Kp]   small-K layout (Kp = 8*ceil(K/8)), pad = -inf
    double *dBT = nullptr;   // [M][Kp]
    double *dPi = nullptr;   // [Kp]
    // slot-permuted copies for the balanced state split of the forward tile kernel (K % 8 != 0), else null
    double *dAb = nullptr, *dBTb = nullptr;
    // f32 mode (decode_f32.cuh): rn32(logA) natural [K][Kp] and slot-permuted [K][Kp], rn32(logB^T) slot-permuted [M][Kp]
    float *dA32n = nullptr, *dA32f = nullptr, *dBT32 = nullptr;
    bool f32_range_ok = false;                // every finite model entry has |x| <= 2^64 (cv_hmm_create)
    // the exact decode may run the f32 forward pass and certify it (decode_small.cuh, certified backtrace): K <= 64,
    // f32_range_ok and every finite entry of logA / logB <= 0
    bool cert_ok = false;
    int64_t last_flagged = -1;                // sequences the last decode call re-decoded in f64; -1: not certified
    int64_t last_fb_chain = 0;                // of those, the ones the warp-per-sequence kernel decoded (the rest: tiles)
    // large-K layout
    int Kl = 0;              // K padded to a multiple of LARGE_BN
    double *dAl = nullptr;   // [Kl][Kl]
    double *dATl = nullptr;  // [Kl][Kl] transposed (lazy-psi backtrace)
    double *dBTl = nullptr;  // [M][Kl]
    // forward-backward (fb_host.inl): probabilities (10^x, -inf -> 0) in the layouts of bw_prep_kernel, built on the
    // first cv_loglik_batch / cv_posterior_batch call
    double *fbA = nullptr;   // [K][Kp]
    double *fbAT = nullptr;  // [K][Kp] transposed
    double *fbBT = nullptr;  // [M][Kp]
    double *fbPi = nullptr;  // [Kp]
    // host copy (control logic of the CP solver, range check of the forward-backward calls)
    std::vector<double> hA, hB, hPi;
    // workspaces
    cvb::DevBuf obs, seq_off, path, score;   // device copies of the host-API buffers
    // decode workspaces: two sets so that consecutive chunks of a batch overlap (forward of chunk k+1 with the
    // backtrace / copies of chunk k) on two internal streams
    struct DecodeWs {
        cvb::DevBuf order, keys_in, keys_out, vals_in, cub_tmp, hist, tmax, base, misc, lg_arr, lg_start, lg_done, delta_g;
        cvb::DevBuf is_long, long_list, long_psi;          // long-sequence split of the tile path (cv_api.cu)
        cvb::DevBuf cert_list;                             // sequences the certified backtrace could not certify
        cudaStream_t st = nullptr;
        cudaEvent_t done = nullptr;
        cudaStream_t st_bt = nullptr;                      // concurrent backtrace (launch_decode_small)
        cudaEvent_t ev_pre = nullptr, ev_bt = nullptr;
        unsigned int *word(cvb::MiscWord i) const { return (unsigned int *)misc.p + i; }
        int *status() const { return (int *)word(cvb::MISC_STATUS); }
    } ws[2];
    cudaEvent_t ev_fork = nullptr;
    cudaStream_t st_long = nullptr;                        // warp-per-sequence kernel for the long sequences of a tile launch
    cudaEvent_t ev_long_dep = nullptr, ev_long_done = nullptr, ev_all_in = nullptr;
    cvb::DevBuf cpb[24];     // constrained-solver state (kept after cv_cp_solve for the parity hooks)
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;
    double last_ms = 0.0, last_bt_ms = 0.0;   // forward kernel / backtrace kernel
    // CP debug state
    int64_t cp_N = 0;
    std::vector<double> cp_ub;
    uint32_t cp_paths = 0;                    // CV_CP_PATH_* bits of the last solve (cv_debug_cp_last_paths)
    void *pinned_status = nullptr;            // cvb::PIN_BYTES, laid out as cvb::PinnedAt
    template <class T> T *pinned(cvb::PinnedAt at) const { return (T *)((char *)pinned_status + at); }
};
