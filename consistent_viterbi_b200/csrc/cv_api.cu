// cv_api.cu -- C ABI (include/cv_b200.h) over the sm_100a kernels.
//
// Host side of the drop-in boundary: model upload, workspace management, launch
// logic and the branch-and-bound control loop of the constrained solver.  No
// CPU compute fallback exists anywhere in this file: if CUDA is unavailable the
// entry points return CV_ERR_CUDA.
#include "cv_internal.cuh"

#include <chrono>

#include <cub/cub.cuh>

#include "common.cuh"
#include "decode_small.cuh"
#include "decode_f32.cuh"
#include "decode_chain.cuh"
#include "decode_large.cuh"

using namespace cvb;

// ---------------------------------------------------------------------------
// errors, counters, tuning block
// ---------------------------------------------------------------------------
static thread_local std::string g_err;
std::atomic<uint64_t> cvb::g_launches{0};
std::atomic<int> cvb::g_timing{0};

int cvb::fail(int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

// The environment is read once, here, when the library is loaded.
static Tuning tuning_from_env()
{
    Tuning t;
    auto geti = [](const char *name, int dflt) { const char *e = getenv(name); return e ? atoi(e) : dflt; };
    t.chunks = geti("CV_CHUNKS", t.chunks);
    t.bt_concurrent = geti("CV_BT_CONCURRENT", t.bt_concurrent);
    t.streamed = geti("CV_STREAMED", t.streamed);
    t.balanced_split = geti("CV_BALANCED", t.balanced_split);
    t.fwd_ldc = geti("CV_FWD_LDC", t.fwd_ldc);
    t.em_light = geti("CV_EM_LIGHT", t.em_light);
    t.bt_split = geti("CV_BT_SPLIT", t.bt_split);
    t.uneven_chunks = geti("CV_UNEVEN_CHUNKS", t.uneven_chunks);
    t.long_split = geti("CV_LONG_SPLIT", t.long_split);
    t.long_pct = geti("CV_LONG_PCT", t.long_pct);
    t.debug = getenv("CV_DEBUG") != nullptr;
    t.bt_prof = getenv("CV_BT_PROF") != nullptr;
    t.e2e_prof = getenv("CV_E2E_PROF") != nullptr;
    if (const char *e = getenv("CV_LARGE_GROUP_RB")) t.large_group_rb = atoll(e);
    t.cp_fullwarp = getenv("CV_CP_FULLWARP") != nullptr;
    t.cp_prof = getenv("CV_CP_PROF") != nullptr;
    t.cp_sum = geti("CV_CP_SUM", t.cp_sum);
    t.cp_hostpoll = geti("CV_CP_HOSTPOLL", t.cp_hostpoll);
    t.cp_leaf_batch = geti("CV_CP_LEAF_BATCH", t.cp_leaf_batch);
    return t;
}
Tuning cvb::g_tune = tuning_from_env();

extern "C" const char *cv_last_error(void) { return g_err.c_str(); }
extern "C" uint64_t cv_launch_count(void) { return g_launches.load(); }
extern "C" void cv_set_timing(int on) { g_timing.store(on); }

int cvb::check_device(int device)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(CV_ERR_CUDA, "no CUDA device available (%s); this library has no CPU fallback",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    }
    if (device >= n) return fail(CV_ERR_ARG, "device %d out of range (%d devices)", device, n);
    return CV_OK;
}

__global__ void build_layouts_kernel(const double *A, const double *Bm, const double *pi, int K, int64_t M, int Kp,
                                     int rowsA, double *Ap, double *BT, double *Pip)
{
    const int64_t n1 = (int64_t)rowsA * Kp, n2 = M * Kp;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n1 + n2 + Kp; e += stride) {
        if (e < n1) {
            int j = (int)(e / Kp), i = (int)(e % Kp);
            Ap[e] = (i < K && j < K) ? A[(int64_t)j * K + i] : neg_inf();
        } else if (e < n1 + n2) {
            int64_t r = e - n1;
            int64_t o = r / Kp; int i = (int)(r % Kp);
            BT[r] = i < K ? Bm[(int64_t)i * M + o] : neg_inf();
        } else {
            int i = (int)(e - n1 - n2);
            Pip[i] = i < K ? pi[i] : neg_inf();
        }
    }
}

extern "C" void cv_hmm_destroy(cv_hmm *h);

// Slot-permuted copies for the balanced state split: column slot 8g + q of row r <- column (state) first(g) + q of the
// natural layout when q < count(g), else -inf; first(g) = g * base + min(g, rem), count(g) = base + (g < rem).
__global__ void permute_slots_kernel(const double *in, double *out, int64_t rows, int Kp, int base, int rem)
{
    const int64_t n = rows * Kp, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride) {
        const int64_t r = e / Kp; const int c = (int)(e % Kp), g = c >> 3, q = c & 7;
        const int first = g * base + min(g, rem), cnt = base + (g < rem ? 1 : 0);
        out[e] = q < cnt ? in[r * Kp + first + q] : neg_inf();
    }
}

__global__ void transpose_kernel(const double *in, double *out, int n)
{
    __shared__ double tile[32][33];
    const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += 8)
        if (by + r < n && bx + threadIdx.x < n) tile[r][threadIdx.x] = in[(size_t)(by + r) * n + bx + threadIdx.x];
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += 8)
        if (bx + r < n && by + threadIdx.x < n) out[(size_t)(bx + r) * n + by + threadIdx.x] = tile[threadIdx.x][r];
}

// f32 copies for the optional f32 mode (decode_f32.cuh): out[r][c] = rn32(in[r][state(c)]) with the slot permutation of
// the balanced split (base = 0: identity), -inf padding.
__global__ void build_f32_kernel(const double *in, float *out, int64_t rows, int K, int Kp, int base, int rem)
{
    const int64_t n = rows * Kp, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride) {
        const int64_t r = e / Kp; const int c = (int)(e % Kp), g = c >> 3, q = c & 7;
        int st = c;
        if (base) { const int first = g * base + min(g, rem), cnt = base + (g < rem ? 1 : 0); st = q < cnt ? first + q : -1; }
        out[e] = (st >= 0 && st < K) ? __double2float_rn(in[r * Kp + st]) : __int_as_float(0xff800000);
    }
}

extern "C" int cv_hmm_create(int K, int D, const uint64_t *bdims, const double *logA, const double *logB,
                             const double *logPi, int device, cv_hmm **out)
{
    if (!out) return fail(CV_ERR_ARG, "out is NULL");
    *out = nullptr;
    if (K <= 0 || K > 65535) return fail(CV_ERR_ARG, "K=%d out of range [1,65535]", K);
    if (D <= 0 || !bdims || !logA || !logB || !logPi) return fail(CV_ERR_ARG, "NULL/empty model argument");
    int64_t M = 1;
    for (int d = 0; d < D; d++) {
        if (bdims[d] == 0) return fail(CV_ERR_ARG, "bdims[%d] == 0", d);
        M *= (int64_t)bdims[d];
    }
    // NaN / +inf would make the reference's argmax().unwrap() panic (or poison every sum): reject.
    auto bad = [](const double *v, int64_t n) {
        for (int64_t i = 0; i < n; i++) if (std::isnan(v[i]) || v[i] == std::numeric_limits<double>::infinity()) return true;
        return false;
    };
    if (bad(logA, (int64_t)K * K) || bad(logB, (int64_t)K * M) || bad(logPi, K))
        return fail(CV_ERR_NAN, "model contains NaN or +inf");
    // Finite entries beyond 2^900 are refused (cv_b200.h): below it no sum of fewer than 2^63 entries can overflow, so
    // every kernel's -inf means "impossible" exactly as in the reference.  The f32 mode has the same guarantee below 2^64.
    auto beyond = [](const double *v, int64_t n, double lim) {
        for (int64_t i = 0; i < n; i++) if (std::isfinite(v[i]) && std::fabs(v[i]) > lim) return true;
        return false;
    };
    auto model_beyond = [&](double lim) { return beyond(logA, (int64_t)K * K, lim) || beyond(logB, (int64_t)K * M, lim) || beyond(logPi, K, lim); };
    if (model_beyond(0x1p900)) return fail(CV_ERR_UNSUPPORTED, "model entry with |x| > 2^900 (sums could overflow)");
    const bool f32_range_ok = !model_beyond(0x1p64);
    auto nonpositive = [](const double *v, int64_t n) {
        for (int64_t i = 0; i < n; i++) if (std::isfinite(v[i]) && v[i] > 0.0) return false;
        return true;
    };
    // log-probabilities (every finite entry <= 0, -0.0 included) within the f32 range: the exact decode may certify an
    // f32 forward pass (decode_small.cuh, certified backtrace); any other model keeps the f64 forward pass
    const bool cert_ok = K <= SMALL_K_MAX && f32_range_ok && nonpositive(logA, (int64_t)K * K) && nonpositive(logB, (int64_t)K * M);
    if (device < 0) {
        int rc = check_device(0);
        if (rc) return rc;
        CUDA_TRY(cudaGetDevice(&device));
    }
    int rc = check_device(device);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(device));

    cv_hmm *h = new cv_hmm();
    struct Guard { cv_hmm *h; ~Guard() { if (h) cv_hmm_destroy(h); } } guard{h};   // released on every early return
    h->device = device; h->K = K; h->D = D; h->M = M;
    h->f32_range_ok = f32_range_ok;
    h->cert_ok = cert_ok;
    // state groups of the forward tile kernel: G = ceil(K/8) warps of TQ = 8 target states, Kp = 8 G
    h->G = (K + TQ - 1) / TQ;
    h->Kp = h->G * TQ;
    h->hA.assign(logA, logA + (size_t)K * K);
    h->hB.assign(logB, logB + (size_t)K * M);
    h->hPi.assign(logPi, logPi + K);
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    h->num_sms = prop.multiProcessorCount;
    CUDA_TRY(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreate(&h->ev0));
    CUDA_TRY(cudaEventCreate(&h->ev1));
    CUDA_TRY(cudaEventCreate(&h->ev2));
    CUDA_TRY(cudaMallocHost(&h->pinned_status, PIN_BYTES));     // laid out as PinnedAt (cv_internal.cuh)
    CUDA_TRY(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    CUDA_TRY(cudaStreamCreateWithFlags(&h->st_long, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&h->ev_long_dep, cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&h->ev_long_done, cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&h->ev_all_in, cudaEventDisableTiming));
    for (auto &w : h->ws) {
        CUDA_TRY(cudaStreamCreateWithFlags(&w.st, cudaStreamNonBlocking));
        CUDA_TRY(cudaEventCreateWithFlags(&w.done, cudaEventDisableTiming));
        CUDA_TRY(cudaStreamCreateWithFlags(&w.st_bt, cudaStreamNonBlocking));
        CUDA_TRY(cudaEventCreateWithFlags(&w.ev_pre, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&w.ev_bt, cudaEventDisableTiming));
    }

    const int Kp = (K <= SMALL_K_MAX) ? h->Kp : ((K + LARGE_BN - 1) / LARGE_BN) * LARGE_BN;
    if (K > SMALL_K_MAX) { h->Kl = Kp; }
    double *tA = nullptr, *tB = nullptr, *tPi = nullptr;
    double *pA = nullptr, *pBT = nullptr, *pPi = nullptr;
    // staging + layout buffers are freed on every early return (the layout buffers are handed to the handle at the end)
    struct Staging { double **p[6]; ~Staging() { for (double **q : p) if (*q) { cudaFree(*q); *q = nullptr; } } } staging{{&tA, &tB, &tPi, &pA, &pBT, &pPi}};
    CUDA_TRY(cudaMalloc(&tA, sizeof(double) * (size_t)K * K));
    CUDA_TRY(cudaMalloc(&tB, sizeof(double) * (size_t)K * M));
    CUDA_TRY(cudaMalloc(&tPi, sizeof(double) * (size_t)K));
    CUDA_TRY(cudaMemcpy(tA, logA, sizeof(double) * (size_t)K * K, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(tB, logB, sizeof(double) * (size_t)K * M, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(tPi, logPi, sizeof(double) * (size_t)K, cudaMemcpyHostToDevice));
    const int rowsA = (K <= SMALL_K_MAX) ? K : Kp;   // the large-K TMA ring reads whole 16-row chunks
    CUDA_TRY(cudaMalloc(&pA, sizeof(double) * (size_t)rowsA * Kp));
    CUDA_TRY(cudaMalloc(&pBT, sizeof(double) * (size_t)M * Kp));
    CUDA_TRY(cudaMalloc(&pPi, sizeof(double) * (size_t)Kp));
    build_layouts_kernel<<<std::max(1, h->num_sms) * 4, 256>>>(tA, tB, tPi, K, M, Kp, rowsA, pA, pBT, pPi);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaDeviceSynchronize());
    if (K <= SMALL_K_MAX) { h->dA = pA; h->dBT = pBT; h->dPi = pPi; }
    else { h->dAl = pA; h->dBTl = pBT; h->dPi = pPi; }
    pA = pBT = pPi = nullptr;                      // owned by the handle now (cv_hmm_destroy)
    if (K <= SMALL_K_MAX && K % 8 != 0 && K / h->G >= 5) {
        // balanced state split of the forward tile kernel: no padded target states (K = 45: 8,8,8,7,7,7 instead of 5 x 8 + 5)
        CUDA_TRY(cudaMalloc(&h->dAb, sizeof(double) * (size_t)K * Kp));
        CUDA_TRY(cudaMalloc(&h->dBTb, sizeof(double) * (size_t)M * Kp));
        permute_slots_kernel<<<std::max(1, h->num_sms) * 4, 256>>>(h->dA, h->dAb, K, Kp, K / h->G, K % h->G);
        permute_slots_kernel<<<std::max(1, h->num_sms) * 4, 256>>>(h->dBT, h->dBTb, M, Kp, K / h->G, K % h->G);
        g_launches += 2;
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaDeviceSynchronize());
    }
    if (K <= SMALL_K_MAX) {
        // optional f32 mode (cv_decode_batch_f32): f32 copies of the model
        const bool bal = h->dAb != nullptr;
        const int base = bal ? K / h->G : 0, rem = bal ? K % h->G : 0;
        CUDA_TRY(cudaMalloc(&h->dA32n, sizeof(float) * (size_t)K * Kp));
        CUDA_TRY(cudaMalloc(&h->dA32f, sizeof(float) * (size_t)K * Kp));
        CUDA_TRY(cudaMalloc(&h->dBT32, sizeof(float) * (size_t)M * Kp));
        build_f32_kernel<<<32, 256>>>(h->dA, h->dA32n, K, K, Kp, 0, 0);
        build_f32_kernel<<<32, 256>>>(h->dA, h->dA32f, K, K, Kp, base, rem);
        build_f32_kernel<<<std::max(1, h->num_sms) * 4, 256>>>(h->dBT, h->dBT32, M, K, Kp, base, rem);
        g_launches += 3;
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaDeviceSynchronize());
    }
    if (K > SMALL_K_MAX) {
        CUDA_TRY(cudaMalloc(&h->dATl, sizeof(double) * (size_t)Kp * Kp));
        transpose_kernel<<<dim3((Kp + 31) / 32, (Kp + 31) / 32), dim3(32, 8)>>>(h->dAl, h->dATl, Kp);
        g_launches++;
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaDeviceSynchronize());
    }
    guard.h = nullptr;
    *out = h;
    return CV_OK;
}

extern "C" void cv_hmm_destroy(cv_hmm *h)
{
    if (!h) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    for (double *p : {h->dA, h->dBT, h->dPi, h->dAl, h->dBTl, h->dATl, h->dAb, h->dBTb, h->fbA, h->fbAT, h->fbBT, h->fbPi}) if (p) cudaFree(p);
    for (float *p : {h->dA32n, h->dA32f, h->dBT32}) if (p) cudaFree(p);
    for (DevBuf *b : {&h->obs, &h->seq_off, &h->path, &h->score}) b->release();
    for (auto &w : h->ws) {
        for (DevBuf *b : {&w.order, &w.keys_in, &w.keys_out, &w.vals_in, &w.cub_tmp, &w.hist, &w.tmax, &w.base, &w.misc,
                          &w.lg_arr, &w.lg_start, &w.lg_done, &w.delta_g, &w.is_long, &w.long_list, &w.long_psi, &w.cert_list})
            b->release();
        if (w.st) cudaStreamDestroy(w.st);
        if (w.done) cudaEventDestroy(w.done);
        if (w.st_bt) cudaStreamDestroy(w.st_bt);
        if (w.ev_pre) cudaEventDestroy(w.ev_pre);
        if (w.ev_bt) cudaEventDestroy(w.ev_bt);
    }
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->st_long) cudaStreamDestroy(h->st_long);
    for (cudaEvent_t e : {h->ev_long_dep, h->ev_long_done, h->ev_all_in}) if (e) cudaEventDestroy(e);
    for (auto &b : h->cpb) b.release();
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->ev2) cudaEventDestroy(h->ev2);
    if (h->stream) cudaStreamDestroy(h->stream);
    if (h->pinned_status) cudaFreeHost(h->pinned_status);
    delete h;
}

extern "C" int cv_hmm_nstates(const cv_hmm *h) { return h ? h->K : 0; }
extern "C" int64_t cv_hmm_nobs(const cv_hmm *h) { return h ? h->M : 0; }
extern "C" double cv_last_kernel_ms(const cv_hmm *h) { return h ? h->last_ms : 0.0; }
extern "C" double cv_last_backtrace_ms(const cv_hmm *h) { return h ? h->last_bt_ms : 0.0; }

extern "C" void *cv_host_alloc(uint64_t bytes)
{
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
extern "C" void cv_host_free(void *p) { if (p) cudaFreeHost(p); }

// ---------------------------------------------------------------------------
// batched plain Viterbi
// ---------------------------------------------------------------------------
typedef cv_hmm::DecodeWs DecodeWs;

// Options of one decode call.  Each public decode entry point builds one and passes it down, so that a function's
// signature shows which precision and which formats it serves.
struct DecodeCall {
    bool f32;              // cv_decode_batch_f32 / cv_decode_batch_dev_f32
    int64_t B;             // the call's batch size: the f32 mode picks its kernel once per call (chain_batch)
    int obs16, path8;      // narrow formats: u16 observations (cv_decode_batch_u16u8), u8 states (and cv_decode_batch_dev_u8)
    bool timing;           // cv_set_timing, read once when the call starts
    size_t obs_bytes() const { return obs16 ? 2 : 4; }     // per element of the caller's host buffers
    size_t path_bytes() const { return path8 ? 1 : 4; }
};
static DecodeCall decode_call(int64_t B, bool f32 = false, int obs16 = 0, int path8 = 0)
{
    return DecodeCall{f32, B, obs16, path8, g_timing.load() != 0};
}

// Long-sequence split (launch_decode_small): the tile kernel runs a tile in lock step for as many steps as its longest
// sequence has, ~8 us per step, so in a SHORT batch (a slice of a sharded batch) a handful of very long sequences
// are the critical path of the whole launch.  Sequences longer than `lstar` are taken out of the tiles: they get
// sort key 0 (they sit in a tile of the shortest sequences as inactive slots), are flagged in is_long[] and
// appended to long_list, and the warp-per-sequence kernel decodes them next to the tile kernel (0.3-0.5 us per
// step).  lstar = 0: no split.  At most cap_long sequences are moved (the rest stay in the tiles: still correct).
struct LongSplit {
    uint32_t lstar, cap_long;
    uint8_t *is_long;            // [B], zeroed by the host
    uint32_t *long_list;         // [cap_long]
    unsigned int *n_long;        // appended so far (may exceed cap_long)
};
__device__ __forceinline__ bool take_long(const LongSplit &ls, int64_t b, int64_t len)
{
    if (ls.lstar == 0 || len <= (int64_t)ls.lstar) return false;
    const unsigned int idx = atomicAdd(ls.n_long, 1u);
    if (idx >= ls.cap_long) return false;
    ls.long_list[idx] = (uint32_t)b;
    ls.is_long[b] = 1;
    return true;
}

// max_len > 0: the caller's bound on the lengths -- the sort then looks only at the bits a length can have, so a longer
// sequence must be an error (CV_ERR_ARG), not a mis-sorted batch
__global__ void seq_len_keys_kernel(const int64_t *seq_off, int64_t B, uint32_t *keys, uint32_t *vals, int *status, const LongSplit ls,
                                    int64_t max_len)
{
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int64_t len = seq_off[b + 1] - seq_off[b];
    if (len <= 0) *status = CV_ERR_EMPTY;          // reference: sequence.len()-1 underflow panic
    else if (max_len > 0 && len > max_len) *status = CV_ERR_ARG;
    const bool lng = take_long(ls, b, len);
    keys[b] = lng ? 0u : (uint32_t)(len < 0 ? 0 : (len > 0xffffffffLL ? 0xffffffffLL : len));
    vals[b] = (uint32_t)b;
}

// bits of the sort key that a length <= max_len can set
static int key_bits(int64_t max_len)
{
    int b = 1;
    while (b < 32 && (max_len >> b) != 0) b++;
    return b;
}

// stable descending radix sort of (keys_in, vals_in) on the key bits [0, end_bit): keys_out, order
static int sort_desc(DecodeWs &w, int64_t n, int end_bit, cudaStream_t st)
{
    size_t tmp_bytes = 0;
    CUDA_TRY(cub::DeviceRadixSort::SortPairsDescending(nullptr, tmp_bytes, (uint32_t *)w.keys_in.p, (uint32_t *)w.keys_out.p,
                                                       (uint32_t *)w.vals_in.p, (uint32_t *)w.order.p, (int)n, 0, end_bit, st));
    if (int rc = w.cub_tmp.ensure(tmp_bytes)) return rc;
    CUDA_TRY(cub::DeviceRadixSort::SortPairsDescending(w.cub_tmp.p, tmp_bytes, (uint32_t *)w.keys_in.p, (uint32_t *)w.keys_out.p,
                                                       (uint32_t *)w.vals_in.p, (uint32_t *)w.order.p, (int)n, 0, end_bit, st));
    return CV_OK;
}

// max_len <= 0 (not supplied): the longest length of the sorted batch is read back (one sync)
static int read_max_len(const DecodeWs &w, int64_t &max_len, cudaStream_t st)
{
    if (max_len > 0) return CV_OK;
    uint32_t L = 0;
    CUDA_TRY(cudaMemcpyAsync(&L, w.keys_out.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    max_len = L;
    return CV_OK;
}

// the buffers of workspace set w that ordering B sequences needs
static int ensure_order_ws(DecodeWs &w, int64_t B)
{
    for (DevBuf *b : {&w.order, &w.keys_in, &w.keys_out, &w.vals_in})
        if (int rc = b->ensure(sizeof(uint32_t) * (size_t)B)) return rc;
    return w.misc.ensure(MISC_BYTES);
}

// Lengths of the sequences [b0, b1) from the host's offsets: their longest one, CV_ERR_ARG for offsets that are not
// monotone, CV_ERR_EMPTY for an empty sequence (reference: usize underflow panic).
static int scan_lengths(const int64_t *seq_off, int64_t b0, int64_t b1, int64_t &max_len)
{
    max_len = 0;
    for (int64_t b = b0; b < b1; b++) {
        const int64_t len = seq_off[b + 1] - seq_off[b];
        if (len < 0) return fail(CV_ERR_ARG, "seq_off not monotone at %lld", (long long)b);
        if (len == 0) return fail(CV_ERR_EMPTY, "sequence %lld is empty (reference: usize underflow panic)", (long long)b);
        max_len = std::max(max_len, len);
    }
    return CV_OK;
}

// longest length of every tile of NS sequences (lengths are sorted descending)
__global__ void tile_tmax_kernel(const uint32_t *sorted_len, int ntiles, int NS, long long *tmax)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < ntiles) tmax[t] = (long long)sorted_len[(size_t)t * NS];
}

// ---- streamed host path: keys = (chunk descending-coded, length) so that one descending sort orders the batch by
// chunk (ascending) and, inside a chunk, by length (longest first); lengths must fit 24 bits
// key = ordering group << shift | length.  promote_len > 0: the sequences of the chunks behind promote_to that are longer
// than this are ordered with chunk promote_to (all observations have long arrived when that group is reached): every
// group starts with its longest tiles, and a late, small group must not start tiles that outlast everything else.
struct ChunkBounds { int nch; int shift; int promote_len, promote_to; int64_t cb[STREAM_MAX_CHUNKS + 2]; };

__global__ void seq_chunk_keys_kernel(const int64_t *seq_off, int64_t B, const ChunkBounds cbs, uint32_t *keys, uint32_t *vals,
                                      int *status, unsigned int *max_len, const LongSplit ls)
{
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int64_t len = seq_off[b + 1] - seq_off[b];
    if (len == 0) atomicMax(status, CV_ERR_EMPTY);            // reference: sequence.len()-1 underflow panic
    if (len < 0) atomicMax(status, CV_ERR_ARG);               // offsets not monotone
    const uint32_t l = (uint32_t)(len < 0 ? 0 : (len > 0xffffffLL ? 0xffffffLL : len));
    if (len > 0xffffffLL) atomicMax(status, CV_ERR_UNSUPPORTED);
    atomicMax(max_len, l);
    int c = 0;
    while (c + 1 < cbs.nch && b >= cbs.cb[c + 1]) c++;
    if (cbs.promote_len > 0 && c > cbs.promote_to && len > (int64_t)cbs.promote_len) c = cbs.promote_to;
    keys[b] = ((uint32_t)(cbs.nch - 1 - c) << cbs.shift) | (take_long(ls, b, len) ? 0u : l);
    vals[b] = (uint32_t)b;
}

// per tile of NS sorted sequences: the longest length and the last chunk it takes sequences from
// promote_to >= 0: tiles of that ordering group may hold sequences of any later chunk (ChunkBounds::promote_len)
__global__ void tile_meta_kernel(const uint32_t *sorted_keys, int ntiles, int NS, int64_t B, int nch, int shift, int promote_to, long long *tmax, int *tchunk)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ntiles) return;
    uint32_t lmax = 0; int cmax = 0;
    for (int s = 0; s < NS; s++) {
        const int64_t r = (int64_t)t * NS + s;
        if (r >= B) break;
        const uint32_t k = sorted_keys[r];
        lmax = max(lmax, k & ((1u << shift) - 1u));
        cmax = max(cmax, nch - 1 - (int)(k >> shift));
    }
    if (promote_to >= 0 && cmax == promote_to) cmax = nch - 1;
    tmax[t] = (long long)lmax; tchunk[t] = cmax;
}

// what launch_decode_small needs to know about the streamed host path
struct StreamedIO {
    ChunkBounds cbs;
    unsigned int *d_arrived;        // chunks whose observations have arrived
    unsigned int *d_chunk_done;     // [nch] finished sequences per chunk
    cudaEvent_t all_in;             // recorded on the copy stream behind the last chunk of observations
};

// Threshold of the long-sequence split (see LongSplit): a tile should not run longer than ~70 % of the tile-steps an
// average resident CTA executes in this launch; never below 64 steps; 0 = no split (nothing is that long).
// Batches above the four-lane backtrace's range (launch_decode_small) are backtraced by one thread per sequence at
// 6-9 us per step -- about as long again as the sequence's forward pass in a tile -- so there the limit is 45 %: at
// 250 k sentences (a rank of a 4-GPU run) the slice holding a 191-step sentence ended 0.18 ms after the others.
static uint32_t long_threshold(const cv_hmm *h, const DecodeCall &call, int64_t B, int64_t N, int64_t max_len)
{
    if (!g_tune.long_split || max_len <= 0 || h->K > SMALL_K_MAX || call.f32) return 0;   // (the warp-per-sequence kernel is f64)
    const int64_t per_cta = (N / 64) / std::max<int64_t>(1, (int64_t)h->num_sms * 2);
    const int pct = g_tune.long_pct > 0 ? g_tune.long_pct : (g_tune.bt_split && B <= (int64_t)1300 * h->num_sms) ? 70 : 45;
    const int64_t l = std::max<int64_t>(64, per_cta * pct / 100);
    return l >= max_len ? 0u : (uint32_t)std::min<int64_t>(l, 0xffffff);
}
constexpr uint32_t LONG_CAP = 4096;

// binds the split's buffers for one launch (workspace set w) and zeroes the flags; ls.lstar = 0 when there is no split
static int long_split_setup(cv_hmm *h, const DecodeCall &call, DecodeWs &w, int64_t B, int64_t N, int64_t max_len,
                            cudaStream_t st, LongSplit &ls)
{
    ls = LongSplit{0u, 0u, nullptr, nullptr, nullptr};
    const uint32_t lstar = long_threshold(h, call, B, N, max_len);
    if (!lstar) return CV_OK;
    int rc;
    const size_t row = (size_t)max_len * h->Kp;
    const uint32_t cap = (uint32_t)std::max<size_t>(1, std::min<size_t>(LONG_CAP, ((size_t)512 << 20) / std::max<size_t>(row, 1)));
    if ((rc = w.is_long.ensure((size_t)B))) return rc;
    if ((rc = w.long_list.ensure(sizeof(uint32_t) * cap))) return rc;
    if ((rc = w.long_psi.ensure(row * cap + 64))) return rc;
    CUDA_TRY(cudaMemsetAsync(w.is_long.p, 0, (size_t)B, st));
    ls.lstar = lstar; ls.cap_long = cap;
    ls.is_long = (uint8_t *)w.is_long.p; ls.long_list = (uint32_t *)w.long_list.p;
    ls.n_long = w.word(MISC_LONG_COUNT);                     // misc is zeroed by the caller before the keys kernel
    return CV_OK;
}

#include "decode_large_host.inl"

// cuStreamWaitValue32 / cuStreamWriteValue32 through the runtime's driver entry-point lookup (no link-time dependency
// on libcuda): a stream waits until a word in device memory reaches a value / writes a word once everything before it
// in the stream is done.  nullptr when unavailable.
typedef int (*StreamValue32Fn)(cudaStream_t, unsigned long long, unsigned int, unsigned int);
static StreamValue32Fn driver_value32(const char *name)
{
    void *f = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint(name, &f, cudaEnableDefault, &qr) != cudaSuccess || qr != cudaDriverEntryPointSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return (StreamValue32Fn)f;
}
static StreamValue32Fn stream_wait_value32() { static const StreamValue32Fn fn = driver_value32("cuStreamWaitValue32"); return fn; }
static StreamValue32Fn stream_write_value32() { static const StreamValue32Fn fn = driver_value32("cuStreamWriteValue32"); return fn; }

// the warp-per-sequence kernel with the instantiation that fits K (register-resident logA column for K <= 32)
static int launch_chain_kernel(const cv_hmm *h, const DecodeChainParams &p, int grid, cudaStream_t st)
{
    const size_t smem = (size_t)h->K * h->Kp * 8 + (p.bt_in_smem ? (size_t)h->M * h->Kp * 8 : 0) +
                        (size_t)DC_WARPS * (16 * h->Kp + 32 * h->Kp + 128);
    auto go = [&](auto kern) -> int {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<grid, 32 * DC_WARPS, smem, st>>>(p);
        return CV_OK;
    };
    // every model has Kp = 8 G (cv_hmm_create), so K <= 32 always fits the register-resident column of 4 KQ = Kp
    int rc;
    switch (h->G) {
        case 1: rc = go(decode_chain_kernel<1, 2>); break;
        case 2: rc = go(decode_chain_kernel<1, 4>); break;
        case 3: rc = go(decode_chain_kernel<1, 6>); break;
        case 4: rc = go(decode_chain_kernel<1, 8>); break;
        default: rc = go(decode_chain_kernel<2, 0>);
    }
    if (rc) return rc;
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return CV_OK;
}

// Residency budget of a forward kernel that a backtrace kernel runs beside (launch_decode_small, concurrent mode): the
// most forward CTAs per SM, at most occ, that leave room on the SM for at least one backtrace CTA (bt, bt_threads,
// bt_smem) -- registers, shared memory with the per-CTA reservation, threads and CTA slots, from the device's
// per-SM limits and the kernels' attributes.  The block scheduler puts as many forward CTAs on an SM as its resources
// allow, so a grid of n CTAs per SM alone does not keep the room free: when n < occ, fwd_smem is padded to the
// smallest size at which n + 1 forward CTAs no longer fit on an SM.  Returns n (fwd_smem updated), or 0 when not even
// one forward CTA leaves room (fwd_smem unchanged; the backtrace then waits for forward CTAs to exit).
static int residency_budget(int dev, void (*fwd)(DecodeSmallParams), int fwd_threads, size_t &fwd_smem,
                            void (*bt)(DecodeSmallParams), int bt_threads, size_t bt_smem, int occ)
{
    int regs_sm = 0, smem_sm = 0, resv = 0, threads_sm = 0, ctas_sm = 0;
    cudaFuncAttributes af, ab;
    if (cudaDeviceGetAttribute(&regs_sm, cudaDevAttrMaxRegistersPerMultiprocessor, dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&resv, cudaDevAttrReservedSharedMemoryPerBlock, dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&threads_sm, cudaDevAttrMaxThreadsPerMultiProcessor, dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&ctas_sm, cudaDevAttrMaxBlocksPerMultiprocessor, dev) != cudaSuccess ||
        cudaFuncGetAttributes(&af, fwd) != cudaSuccess || cudaFuncGetAttributes(&ab, bt) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    // registers are allocated per warp in units of 256, shared memory per CTA in units of 128 bytes
    auto regs_cta = [](const cudaFuncAttributes &a, int threads) -> int64_t {
        return (int64_t)((threads + 31) / 32) * ((a.numRegs * 32 + 255) / 256 * 256);
    };
    auto smem_cta = [&](const cudaFuncAttributes &a, size_t dyn) -> int64_t {
        return (int64_t)((a.sharedSizeBytes + dyn + 127) / 128 * 128) + resv;
    };
    const int64_t rf = regs_cta(af, fwd_threads), rb = regs_cta(ab, bt_threads), sb = smem_cta(ab, bt_smem);
    for (int n = occ; n >= 1; n--) {
        if (n * rf + rb > regs_sm || n * fwd_threads + bt_threads > threads_sm || n + 1 > ctas_sm) continue;
        int64_t sf = smem_cta(af, fwd_smem);
        if (n < occ) sf = std::max(sf, ((int64_t)smem_sm / (n + 1) + 1 + 127) / 128 * 128);
        if (n * sf + sb > smem_sm) continue;
        fwd_smem = (size_t)(sf - resv - (int64_t)af.sharedSizeBytes);
        return n;
    }
    return 0;
}

// Parameters of the warp-per-sequence kernel over the sequences order[0, B) with workspace set w: backpointer rows in
// psi, tile counter in the misc word `counter`.  B_dev: the number of sequences is read on the device (at most B), and
// the rows of list entry r start at row r * psi_stride.  sio: finished sequences are counted per chunk (streamed path).
static DecodeChainParams chain_params(const cv_hmm *h, const DecodeCall &call, const DecodeWs &w, const uint32_t *d_obs,
                                      const int64_t *d_off, uint32_t *d_path, double *d_score, const uint32_t *order,
                                      void *psi, MiscWord counter, int64_t B, const unsigned int *B_dev = nullptr,
                                      int64_t psi_stride = 0, const StreamedIO *sio = nullptr)
{
    DecodeChainParams q;
    q.A = h->dA; q.BT = h->dBT; q.obs = d_obs; q.seq_off = d_off; q.order = order;
    q.psi = (uint8_t *)psi; q.path = d_path; q.score = d_score; q.counter = w.word(counter); q.status = w.status();
    q.M = h->M; q.B = B; q.K = h->K; q.Kp = h->Kp;
    q.bt_in_smem = ((size_t)h->M * h->Kp * 8 <= CHAIN_BT_SMEM_MAX) ? 1 : 0;
    q.obs16 = call.obs16; q.path8 = call.path8;
    q.B_dev = B_dev; q.psi_stride = psi_stride;
    q.chunk_done = sio ? sio->d_chunk_done : nullptr; q.nch = sio ? sio->cbs.nch : 0;
    if (sio) for (int c = 0; c <= sio->cbs.nch; c++) q.cb[c] = sio->cbs.cb[c];
    return q;
}

// The tile path of workspace set w: forward kernel over tiles of 64 sequences ordered longest first (w.order from rank
// `first` on), then the backtrace.  The tile counter and the status are w's misc words.
static int launch_decode_small(cv_hmm *h, const DecodeCall &call, DecodeWs &w, const uint32_t *d_obs, const int64_t *d_off,
                               int64_t B, int64_t N, uint32_t *d_path, double *d_score, int64_t max_len, cudaStream_t st,
                               bool cert, const StreamedIO *sio = nullptr, const LongSplit *ls = nullptr, int64_t first = 0)
{
    const int G = h->G;
    const uint32_t *d_order = (const uint32_t *)w.order.p + first, *d_sorted_len = (const uint32_t *)w.keys_out.p + first;
    // optional f32 mode (decode_f32.cuh): its own forward kernel, f32 history, f32 backtrace.  cert: the same forward
    // kernel and history, then the certified backtrace (decode_small.cuh) -- the exact decode of an eligible model
    const bool f32 = call.f32 || cert;
    // tiles of NS = 64 sequences (TP = 2 per lane), one warp per state group
    const int NS = 32 * TP, threads = 32 * G;
    size_t smem = f32 ? decode_f32_smem_bytes(h->K, h->Kp) : decode_small_smem_bytes(h->K, h->Kp, NS);
    const int64_t ntiles64 = (B + NS - 1) / NS;
    if (ntiles64 > 0x7fffffffLL) return fail(CV_ERR_UNSUPPORTED, "batch too large");
    const int ntiles = (int)ntiles64;
    int rc;
    if ((rc = read_max_len(w, max_len, st))) return rc;
    // history slabs: sum over tiles of NS * Tmax(tile) <= N + NS * max_len because lengths are sorted (per chunk, plus
    // the tiles that straddle two chunks, on the streamed path)
    // Streamed path: tiles are ordered by (chunk, length).  Inside a chunk the staircase bound above holds (one
    // NS * max_len term per chunk); a tile that straddles two chunks takes its length from either and adds up to
    // NS * max_len of its own, and there are at most nch - 1 of those: 2 * nch - 1 terms in all.  The forward kernel
    // also checks every tile against hist_cap_rows and reports CV_ERR_UNSUPPORTED instead of storing past the end.
    const size_t stairs = sio ? 2 * (size_t)sio->cbs.nch - 1 : 1;
    const size_t hist_rows = (size_t)N + (size_t)NS * (size_t)max_len * stairs;     // in units of K doubles
    const size_t hist_elems = hist_rows * (size_t)h->K;
    if ((rc = w.hist.ensure(hist_elems * (f32 ? sizeof(float) : sizeof(double))))) return rc;
    if ((rc = w.tmax.ensure(sizeof(long long) * (size_t)ntiles))) return rc;
    if ((rc = w.base.ensure(sizeof(long long) * (size_t)ntiles))) return rc;
    if (sio) {
        if ((rc = w.delta_g.ensure(sizeof(int) * (size_t)ntiles + 64))) return rc;     // tile -> chunk (buffer unused for K <= 64)
        tile_meta_kernel<<<(ntiles + 127) / 128, 128, 0, st>>>(d_sorted_len, ntiles, NS, B, sio->cbs.nch, sio->cbs.shift, sio->cbs.promote_len > 0 ? sio->cbs.promote_to : -1, (long long *)w.tmax.p, (int *)w.delta_g.p);
    } else {
        tile_tmax_kernel<<<(ntiles + 255) / 256, 256, 0, st>>>(d_sorted_len, ntiles, NS, (long long *)w.tmax.p);
    }
    g_launches++;
    size_t tmp_bytes = 0;
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, (long long *)w.tmax.p, (long long *)w.base.p, ntiles, st));
    if ((rc = w.cub_tmp.ensure(tmp_bytes))) return rc;
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(w.cub_tmp.p, tmp_bytes, (long long *)w.tmax.p, (long long *)w.base.p, ntiles, st));

    DecodeSmallParams p;
    p.A = h->dA; p.BT = h->dBT; p.obs = d_obs; p.seq_off = d_off; p.order = d_order;
    p.At = h->dA; p.BTt = h->dBT; p.nq_base = p.nq_rem = 0;
    p.obs16 = call.obs16; p.path8 = call.path8; p.em_light = g_tune.em_light;
    p.is_long = (ls && ls->lstar) ? ls->is_long : nullptr;
    p.A32s = h->dA32f; p.A32n = h->dA32n; p.BT32 = h->dBT32;
    p.cert_list = cert ? (uint32_t *)w.cert_list.p : nullptr;
    p.cert_count = cert ? w.word(MISC_CERT) : nullptr;       // zeroed by the caller with the rest of misc
    p.cert_tol = g_tune.cert_tol;
    if ((f32 || g_tune.balanced_split) && h->dAb) {
        p.At = h->dAb; p.BTt = h->dBTb; p.nq_base = h->K / G; p.nq_rem = h->K % G;
    }
    p.tile_base = (const long long *)w.base.p;
    p.hist = (double *)w.hist.p; p.hist_cap_slabs = (long long)(hist_rows / (size_t)NS); p.path = d_path; p.score = d_score; p.tile_counter = w.word(MISC_COUNTER); p.status = w.status();
    p.M = h->M; p.B = B; p.K = h->K; p.Kp = h->Kp; p.G = G; p.NS = NS; p.ntiles = ntiles;
    p.tile_tmax = nullptr; p.tile_chunk = nullptr; p.arrived = nullptr; p.chunk_done = nullptr; p.nch = 0;
    if (sio) {
        p.tile_tmax = (const long long *)w.tmax.p; p.tile_chunk = (const int *)w.delta_g.p;
        p.arrived = sio->d_arrived; p.chunk_done = sio->d_chunk_done; p.nch = sio->cbs.nch;
        for (int c = 0; c <= sio->cbs.nch; c++) p.cb[c] = sio->cbs.cb[c];
    }
    // f32: the 64-register build of the forward kernel leaves room for the concurrent backtrace and hides it behind a
    // long batch's forward pass (1 M POS sentences: 7.3 -> 6.6 ms per certified step); a short batch -- a few tiles per
    // CTA, the same bound as the four-lane backtrace's -- cannot hide it and runs the faster 78-register build
    // (125 k sentences: 1.58 ms per step with it, 1.71 ms with the 64-register build).
    const bool long_batch = B > (int64_t)1300 * h->num_sms;
    void (*kern)(DecodeSmallParams) = !f32 ? decode_small_fwd_kernel<0>
                                    : long_batch ? decode_f32_fwd_kernel<4> : decode_f32_fwd_kernel<3>;
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    int occ = 1;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem));
    occ = std::max(1, occ);
    if (!f32 && g_tune.fwd_ldc) {
        // The same kernel with compile-time row pitches (tiles of 64 sequences, logA rows at a pitch of 64 doubles in
        // shared memory) -- unless the wider logA costs a resident CTA per SM.
        void (*kc)(DecodeSmallParams) = decode_small_fwd_kernel<FWD_LDC>;
        const size_t smem_c = decode_small_smem_bytes(h->K, h->Kp, NS, FWD_LDC);
        int occ_c = 0;
        if (smem_c <= 220 * 1024) {
            CUDA_TRY(cudaFuncSetAttribute(kc, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_c));
            CUDA_TRY(cudaFuncSetAttribute(kc, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
            CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_c, kc, threads, smem_c));
        }
        if (occ_c >= occ) { kern = kc; smem = smem_c; }
    }
    // Concurrent backtrace: the backtrace kernel runs next to the forward kernel on a second stream and follows
    // it tile by tile (tile_done flags).  It is released only when every forward CTA is resident (stream wait on
    // the `started` counter), so its spinning CTAs can never keep a forward CTA off an SM; it then lives on the
    // registers / shared memory the forward CTAs leave free.
    StreamValue32Fn wait32 = stream_wait_value32();
    const bool concurrent = !call.timing && g_tune.bt_concurrent && wait32 != nullptr && w.st_bt != nullptr;
    if (sio && !concurrent) return fail(CV_ERR_UNSUPPORTED, "the streamed path needs the concurrent backtrace");
    // end state + backtrace with lazy backpointers: one thread per sequence
    const size_t smem_bt = (size_t)h->K * (h->K | 1) * 8 + 16 * 8;      // + one chunk of padding behind the last row
    void (*bt_seq)(DecodeSmallParams) = cert ? backtrace_small_kernel<16, 4, float, true>
                                      : f32 ? backtrace_small_kernel<16, 4, float> : backtrace_small_kernel<16, 4>;
    void (*bt_con)(DecodeSmallParams) = cert ? backtrace_small_kernel<8, 8, float, true>
                                      : f32 ? backtrace_small_kernel<8, 8, float> : backtrace_small_kernel<8, 8>;
    // The f32 forward kernel alone fills an SM's registers (four CTAs at K = 45): make room for the backtrace
    if (f32 && concurrent) {
        if (int n = residency_budget(h->device, kern, threads, smem, bt_con, 128, smem_bt, occ)) {
            CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem));
            if (occ != n) return fail(CV_ERR_CUDA, "forward CTAs per SM: %d, budget %d", occ, n);
        }
    }
    const int grid = (int)std::min<int64_t>((int64_t)h->num_sms * occ, ntiles);
    if (g_tune.debug)
        fprintf(stderr, "[cv] decode_small: K=%d G=%d f32=%d cert=%d threads=%d smem=%zu occ=%d grid=%d tiles=%d\n",
                h->K, G, (int)f32, (int)cert, threads, smem, occ, grid, ntiles);
    p.tile_done = nullptr; p.started = nullptr;
    if (concurrent) {
        if ((rc = w.lg_done.ensure(sizeof(int) * ((size_t)ntiles + 8)))) return rc;
        CUDA_TRY(cudaMemsetAsync(w.lg_done.p, 0, sizeof(int) * ((size_t)ntiles + 8), st));
        p.tile_done = (int *)w.lg_done.p;
        p.started = (unsigned int *)w.lg_done.p + ntiles;
        CUDA_TRY(cudaEventRecord(w.ev_pre, st));
    }
    // Long-sequence split: the flagged sequences run on the warp-per-sequence kernel next to the tile kernels, on a
    // stream of its own; it is launched first so that its few CTAs are resident before the persistent forward CTAs.
    bool long_launched = false;
    if (ls && ls->lstar) {
        const DecodeChainParams q = chain_params(h, call, w, d_obs, d_off, d_path, d_score, ls->long_list, w.long_psi.p,
                                                 MISC_LONG_COUNTER, (int64_t)ls->cap_long, ls->n_long, max_len, sio);
        CUDA_TRY(cudaEventRecord(h->ev_long_dep, st));                        // keys kernel (list, count) and the offsets are done
        CUDA_TRY(cudaStreamWaitEvent(h->st_long, h->ev_long_dep, 0));
        if (sio) CUDA_TRY(cudaStreamWaitEvent(h->st_long, sio->all_in, 0));   // streamed: all observations on the device
        const int grid_l = (int)std::min<int64_t>((ls->cap_long + DC_WARPS - 1) / DC_WARPS, (int64_t)h->num_sms);
        if ((rc = launch_chain_kernel(h, q, grid_l, h->st_long))) return rc;
        CUDA_TRY(cudaEventRecord(h->ev_long_done, h->st_long));
        long_launched = true;
    }
    const bool bt_prof = g_tune.bt_prof != 0;   // prints forward / forward+backtrace times of the concurrent mode
    if (call.timing || bt_prof) CUDA_TRY(cudaEventRecord(h->ev0, st));
    kern<<<std::max(1, grid), threads, smem, st>>>(p);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    if (call.timing || bt_prof) CUDA_TRY(cudaEventRecord(h->ev1, st));
    // Four lanes per sequence (backtrace_split_kernel, f64 only) -- for batches that do
    // not fill the GPU for long (a rank's slice of a sharded batch): there the one-thread-per-sequence kernel is latency
    // bound and most of its work is still open when the forward kernel ends.  Measured, device step with the concurrent
    // backtrace, split vs. one thread per sequence: 125 k sentences 1.51 vs 1.74 ms, 250 k 2.83 vs 2.79 ms, 500 k 5.59 vs
    // 5.29 ms, 1 M 11.20 vs 10.56 ms (four times the threads re-stage logA four times as often and execute ~15 % more
    // instructions next to an issue-bound forward kernel).  bt_split = 2 forces it for every size.
    bool bt_split = g_tune.bt_split && !f32 && (g_tune.bt_split >= 2 || B <= (int64_t)1300 * h->num_sms);
    size_t smem_bt_use = smem_bt;
    if (bt_split) {
        const int JP = h->K <= 16 ? 4 : h->K <= 32 ? 8 : h->K <= 48 ? 12 : 16;
        bt_seq = bt_con = JP == 4 ? backtrace_split_kernel<4, 8> : JP == 8 ? backtrace_split_kernel<8, 8>
                        : JP == 12 ? backtrace_split_kernel<12, 8> : backtrace_split_kernel<16, 8>;
        smem_bt_use = ((size_t)(h->K + 1) * (h->K | 1) + 4 * JP) * 8;
    }
    CUDA_TRY(cudaFuncSetAttribute(bt_seq, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bt_use));
    CUDA_TRY(cudaFuncSetAttribute(bt_con, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bt_use));
    // same shared-memory carve-out as the forward kernel, or the two kernels cannot share an SM
    CUDA_TRY(cudaFuncSetAttribute(bt_con, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    const int64_t nblk = ((int64_t)ntiles * NS * (bt_split ? 4 : 1) + 127) / 128;
    if (concurrent) {
        CUDA_TRY(cudaStreamWaitEvent(w.st_bt, w.ev_pre, 0));
        if (wait32(w.st_bt, (unsigned long long)(uintptr_t)p.started, (unsigned int)std::max(1, grid), 0x0 /* GEQ */) != 0)
            return fail(CV_ERR_CUDA, "cuStreamWaitValue32 failed");
        bt_con<<<(unsigned)std::max<int64_t>(1, nblk), 128, smem_bt_use, w.st_bt>>>(p);   // blocks in tile order
        g_launches++;
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaEventRecord(w.ev_bt, w.st_bt));
        CUDA_TRY(cudaStreamWaitEvent(st, w.ev_bt, 0));
        if (long_launched) CUDA_TRY(cudaStreamWaitEvent(st, h->ev_long_done, 0));
        if (bt_prof) {
            CUDA_TRY(cudaEventRecord(h->ev2, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            float a = 0.f, b = 0.f;
            cudaEventElapsedTime(&a, h->ev0, h->ev1); cudaEventElapsedTime(&b, h->ev0, h->ev2);
            fprintf(stderr, "[cv] concurrent: forward %.3f ms, forward + backtrace %.3f ms (B = %lld)\n", a, b, (long long)B);
        }
        return CV_OK;
    }
    const int grid_bt = (int)std::max<int64_t>(1, std::min<int64_t>(nblk, (int64_t)h->num_sms * 12));
    bt_seq<<<grid_bt, 128, smem_bt_use, st>>>(p);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    if (call.timing) CUDA_TRY(cudaEventRecord(h->ev2, st));
    if (long_launched) CUDA_TRY(cudaStreamWaitEvent(st, h->ev_long_done, 0));
    return CV_OK;
}

// Batches of up to 8192 sequences with K <= 64 go to the warp-per-sequence kernel; cv_debug_set_chain_max_batch moves
// that bound for the exact mode.  The f32 mode keeps it whatever the override says, and applies it to the whole call,
// not to one chunk: cv_b200.h promises such calls the exact f64 kernel, and every larger call the f32 kernels in all
// its chunks (a forced small chunk count must not hand part of an f32 call to the f64 kernel).
constexpr int64_t CHAIN_BATCH_MAX = 8192;
static bool chain_batch(const cv_hmm *h, const DecodeCall &call, int64_t B)
{
    if (call.f32) return h->K <= SMALL_K_MAX && call.B <= CHAIN_BATCH_MAX;
    const long long bound = g_tune.chain_max_b < 0 ? CHAIN_BATCH_MAX : g_tune.chain_max_b;
    return h->K <= SMALL_K_MAX && B <= bound;
}

// sort keys of the sequences in list[0, n): length, id
__global__ void listed_len_keys_kernel(const int64_t *seq_off, const uint32_t *list, int64_t n, uint32_t *keys, uint32_t *vals)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t b = list[i];
    keys[i] = (uint32_t)(seq_off[b + 1] - seq_off[b]);
    vals[i] = b;
}

// How many of the n flagged sequences (longest lmax) certified_fallback gives the warp-per-sequence kernel.
// - Up to CHAIN_BATCH_MAX: all of them, as a batch of n would go there (chain_batch).
// - Up to two tiles per SM: the tile path is one wave of about one tile per CTA, in lock step for as many steps as its
//   longest tile, and flagged sequences are the long ones (the certificate's bound grows with the step).  The
//   FB_CHAIN_PER_SM * num_sms longest go to the warp-per-sequence kernel beside it, one warp each.  Measured on one
//   NVIDIA B200 (148 SMs), fallback with its host round trip: 1 M POS sentences (17 369 flagged) 1.34-1.46 ms on the
//   tiles alone, 0.81-0.89 ms with 296-592 on the warp kernel, 1.35 ms with 4736 and 1.36 ms with all of them (a warp
//   then decodes several sequences, at 1-2 us per step beside the tile kernel); 500 k (8494 flagged) 1.08 ms on the
//   tiles, 0.59-0.66 ms with 148-296, 0.74 ms with all of them.
// - More: the tile scheduler balances several waves of tiles, and the warp kernel beside them only takes issue slots
//   (tie-heavy model, 124 952 flagged: 1.45 ms on the tiles, 1.50 ms with 296 on the warp kernel).
constexpr int64_t FB_CHAIN_PER_SM = 2;
static int64_t fallback_chain_count(const cv_hmm *h, int64_t n, int64_t lmax)
{
    int64_t k;
    switch (g_tune.fb_route) {
        case 1: k = 0; break;
        case 2: k = n; break;
        case 3: k = g_tune.fb_chain; break;
        default:
            if (n <= CHAIN_BATCH_MAX) return n;
            if (n > (int64_t)2 * 64 * h->num_sms) return 0;
            // backpointer rows of the moved sequences: at most 512 MB
            k = std::min<int64_t>(FB_CHAIN_PER_SM * h->num_sms, ((int64_t)512 << 20) / (lmax * h->Kp));
    }
    return std::max<int64_t>(0, std::min(k, n));
}

// Exact f64 re-decode of the sequences the certified backtrace could not certify (launch_decode_small with cert): their
// paths and scores are overwritten.  This is the one host round trip of a certified call: the flagged count, their
// longest length and their elements are read back, and decide the kernels (fallback_chain_count): the warp-per-sequence
// kernel for all of them, or the flagged sequences ordered by length with the longest on the warp-per-sequence kernel
// (stream st_long) and the rest on the f64 tile path beside it.
static int certified_fallback(cv_hmm *h, const DecodeCall &call, DecodeWs &w, const uint32_t *d_obs, const int64_t *d_off,
                              uint32_t *d_path, double *d_score, cudaStream_t st)
{
    unsigned int *hc = h->pinned<unsigned int>(PIN_CERT);
    CUDA_TRY(cudaMemcpyAsync(hc, w.word(MISC_CERT), 4 * sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    const int64_t n = hc[0], lmax = hc[1];
    const int64_t nel = (int64_t)*reinterpret_cast<const unsigned long long *>(hc + 2);
    h->last_flagged = n;
    h->last_fb_chain = 0;
    if (n == 0) return CV_OK;
    const uint32_t *list = (const uint32_t *)w.cert_list.p;
    const int64_t n_chain = fallback_chain_count(h, n, lmax);
    h->last_fb_chain = n_chain;
    int rc;
    if (n_chain == n) {
        // the f32 history is no longer needed: its buffer takes the backpointer rows
        if ((rc = w.hist.ensure((size_t)n * (size_t)lmax * h->Kp + 64))) return rc;
        const DecodeChainParams q = chain_params(h, call, w, d_obs, d_off, d_path, d_score, list, w.hist.p, MISC_CERT_COUNTER,
                                                 n, w.word(MISC_CERT), lmax);
        const int grid = (int)std::min<int64_t>((n + DC_WARPS - 1) / DC_WARPS, (int64_t)h->num_sms * 8);
        return launch_chain_kernel(h, q, grid, st);
    }
    listed_len_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_off, list, n, (uint32_t *)w.keys_in.p, (uint32_t *)w.vals_in.p);
    g_launches++;
    if ((rc = sort_desc(w, n, key_bits(lmax), st))) return rc;
    CUDA_TRY(cudaMemsetAsync(w.word(MISC_COUNTER), 0, sizeof(unsigned int), st));
    if (n_chain > 0) {
        // the n_chain longest (w.order[0, n_chain)) on the warp-per-sequence kernel; its backpointer rows go to long_psi
        // because the tile path writes its history to w.hist at the same time.  Its count is read on the device: the
        // flagged count is at least n_chain.
        if ((rc = w.long_psi.ensure((size_t)n_chain * (size_t)lmax * h->Kp + 64))) return rc;
        const DecodeChainParams q = chain_params(h, call, w, d_obs, d_off, d_path, d_score, (const uint32_t *)w.order.p,
                                                 w.long_psi.p, MISC_CERT_COUNTER, n_chain, w.word(MISC_CERT), lmax);
        CUDA_TRY(cudaEventRecord(h->ev_long_dep, st));                        // the sorted order is done
        CUDA_TRY(cudaStreamWaitEvent(h->st_long, h->ev_long_dep, 0));
        const int grid = (int)std::min<int64_t>((n_chain + DC_WARPS - 1) / DC_WARPS, (int64_t)h->num_sms);
        if ((rc = launch_chain_kernel(h, q, grid, h->st_long))) return rc;
        CUDA_TRY(cudaEventRecord(h->ev_long_done, h->st_long));
    }
    DecodeCall exact = call;
    exact.timing = false;                     // the call's kernel times stay those of the certified pass
    if ((rc = launch_decode_small(h, exact, w, d_obs, d_off, n - n_chain, nel, d_path, d_score, lmax, st, false, nullptr,
                                  nullptr, n_chain)))
        return rc;
    if (n_chain > 0) CUDA_TRY(cudaStreamWaitEvent(st, h->ev_long_done, 0));
    if (g_tune.bt_prof) {
        CUDA_TRY(cudaEventRecord(h->ev2, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        float ms = 0.f;
        cudaEventElapsedTime(&ms, h->ev0, h->ev2);
        fprintf(stderr, "[cv] fallback: %lld flagged, %lld on the warp kernel, tiles + warp kernel %.3f ms\n",
                (long long)n, (long long)n_chain, ms);
    }
    return CV_OK;
}

// One chunk of sequences [0, B) of d_off (offsets are absolute into d_obs / d_path): order by length,
// forward, backtrace; everything enqueued on `st` with workspace set `w`.  can_certify: the chunk is the whole call
// (certified_fallback's host round trip is made once per call).
static int decode_chunk(cv_hmm *h, const DecodeCall &call, DecodeWs &w, const uint32_t *d_obs, const int64_t *d_off,
                        int64_t B, int64_t N, int64_t max_len, uint32_t *d_path, double *d_score, cudaStream_t st,
                        bool can_certify)
{
    int rc;
    if (B > 0x7fffffffLL) return fail(CV_ERR_UNSUPPORTED, "more than 2^31 sequences in one chunk");
    if ((rc = ensure_order_ws(w, B))) return rc;
    CUDA_TRY(cudaMemsetAsync(w.misc.p, 0, MISC_BYTES, st));
    const bool chain_all = chain_batch(h, call, B);
    LongSplit ls{0u, 0u, nullptr, nullptr, nullptr};
    if (!chain_all && (rc = long_split_setup(h, call, w, B, N, max_len, st, ls))) return rc;
    // order sequences by length, longest first (stable radix sort => deterministic)
    seq_len_keys_kernel<<<(unsigned)((B + 255) / 256), 256, 0, st>>>(d_off, B, (uint32_t *)w.keys_in.p,
                                                                    (uint32_t *)w.vals_in.p, w.status(), ls, max_len);
    g_launches++;
    // the radix sort only visits the bits a length can have (one 8-bit pass for lengths up to 255 instead of four)
    if ((rc = sort_desc(w, B, max_len > 0 ? key_bits(max_len) : 32, st))) return rc;
    if (chain_all) {
        // few sequences: one warp per sequence (latency-oriented), backpointers as u8 rows
        if ((rc = w.hist.ensure((size_t)N * h->Kp + 64))) return rc;
        const DecodeChainParams p = chain_params(h, call, w, d_obs, d_off, d_path, d_score, (const uint32_t *)w.order.p,
                                                 w.hist.p, MISC_COUNTER, B);
        const int grid = (int)std::min<int64_t>((B + DC_WARPS - 1) / DC_WARPS, (int64_t)h->num_sms * 8);
        if (call.timing) CUDA_TRY(cudaEventRecord(h->ev0, st));
        if ((rc = launch_chain_kernel(h, p, grid, st))) return rc;
        if (call.timing) { CUDA_TRY(cudaEventRecord(h->ev1, st)); CUDA_TRY(cudaEventRecord(h->ev2, st)); }
        return CV_OK;
    }
    if (h->K <= SMALL_K_MAX) {
        const bool cert = can_certify && h->cert_ok && !call.f32 && g_tune.certified;
        if (cert && (rc = w.cert_list.ensure(sizeof(uint32_t) * (size_t)B))) return rc;
        if ((rc = launch_decode_small(h, call, w, d_obs, d_off, B, N, d_path, d_score, max_len, st, cert, nullptr, &ls))) return rc;
        if (!cert) return CV_OK;
        if ((rc = certified_fallback(h, call, w, d_obs, d_off, d_path, d_score, st))) return rc;
        if (call.timing) CUDA_TRY(cudaEventRecord(h->ev2, st));               // backtrace time = backtrace + fallback
        return CV_OK;
    }
    if (call.timing) CUDA_TRY(cudaEventRecord(h->ev0, st));
    if ((rc = launch_decode_large(h, w, d_obs, d_off, B, d_path, d_score, max_len, st))) return rc;
    if (call.timing) { CUDA_TRY(cudaEventRecord(h->ev1, st)); CUDA_TRY(cudaEventRecord(h->ev2, st)); }
    return CV_OK;
}

static int chunk_count(const cv_hmm *h, const DecodeCall &call, bool host_buffers)
{
    const int64_t B = call.B;
    if (call.timing || h->K > SMALL_K_MAX) return 1;     // kernel timing wants one launch for the whole batch
    if (g_tune.chunks > 0) return (int)std::min<int64_t>(g_tune.chunks, std::max<int64_t>(B, 1));
    // >= ~6 tiles per resident CTA per chunk keeps the dynamic tile scheduler balanced.  Host buffers: six
    // chunks so that H2D / D2H copies hide behind the kernels (measured at the POS shape: 2 chunks 16.5 ms,
    // 4: 15.4, 6: 15.3, 8: 15.7, 12: 19.2).
    // Device buffers: one launch when the backtrace can run next to the forward kernel (launch_decode_small), else two
    // chunks so that the backtrace of one overlaps the forward pass of the other.
    const int64_t per_chunk = (int64_t)h->num_sms * 2 * 6 * 64;
    const int dev_chunks = (g_tune.bt_concurrent && stream_wait_value32() != nullptr) ? 1 : 2;
    // Host buffers, streamed past one launch (decode_streamed): 4 chunks measured best (2: 14.8 ms, 3: 14.3, 4: 14.2-14.3,
    // 6: 14.4, 10: 14.8, 16: 15.0 -- every chunk restarts the longest-first tile order); one launch per chunk: 6.
    const bool can_stream = g_tune.streamed && g_tune.bt_concurrent && stream_wait_value32() != nullptr;
    // Streaming pays from ~450 k sequences: below, every chunk's restart of the longest-first tile order costs more
    // than the copies it hides (measured: 250 k sequences 4.2 ms streamed in two chunks vs 3.0 ms on the device; one
    // H2D -> decode -> D2H pass is 3.7 ms), so shorter batches go through in one piece.
    // With the tapering chunks of decode_streamed the crossover is lower: 350 k sequences 5.05 ms streamed vs 5.62 ms in
    // one piece, 250 k 4.27 vs 4.03 ms.
    if (host_buffers && can_stream) return (g_tune.uneven_chunks ? B >= (int64_t)2000 * h->num_sms : B / per_chunk >= 4) ? 4 : 1;
    return (int)std::max<int64_t>(1, std::min<int64_t>(host_buffers ? 6 : dev_chunks, B / per_chunk));
}

// The end of a call that used workspace sets [0, nws): their status words are read back behind the work on st[k], the
// kernel times are taken when the call is timed, and the first error status is reported.
static int finish_call(cv_hmm *h, const DecodeCall &call, int nws, cudaStream_t st0, cudaStream_t st1 = nullptr)
{
    const cudaStream_t st[2] = {st0, st1};
    int *hs = h->pinned<int>(PIN_STATUS);
    for (int k = 0; k < nws; k++) CUDA_TRY(cudaMemcpyAsync(hs + k, h->ws[k].status(), sizeof(int), cudaMemcpyDeviceToHost, st[k]));
    for (int k = 0; k < nws; k++) CUDA_TRY(cudaStreamSynchronize(st[k]));
    if (call.timing) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, h->ev0, h->ev1) == cudaSuccess) h->last_ms = ms; else cudaGetLastError();
        if (cudaEventElapsedTime(&ms, h->ev1, h->ev2) == cudaSuccess) h->last_bt_ms = ms; else cudaGetLastError();
    }
    for (int k = 0; k < nws; k++) {
        const int s = hs[k];
        if (s == CV_ERR_EMPTY) return fail(CV_ERR_EMPTY, "empty sequence in batch (reference: usize underflow panic)");
        if (s == CV_ERR_ARG) return fail(CV_ERR_ARG, "observation index >= M (reference: ndarray index panic)");
        if (s) return fail(s, "device status %d", s);
    }
    return CV_OK;
}

static int decode_batch_dev(cv_hmm *h, const DecodeCall &call, const uint32_t *d_obs, const int64_t *d_off, int64_t N,
                            int64_t max_len, uint32_t *d_path, double *d_score, void *stream, int sync_status)
{
    const int64_t B = call.B;
    if (!h) return fail(CV_ERR_ARG, "NULL model");
    if (B < 0 || N < 0) return fail(CV_ERR_ARG, "negative size");
    if (B == 0) return CV_OK;
    if (!d_obs || !d_off || !d_path) return fail(CV_ERR_ARG, "NULL buffer");
    CUDA_TRY(cudaSetDevice(h->device));
    h->last_flagged = -1;
    cudaStream_t user = (cudaStream_t)stream;
    const int nch = chunk_count(h, call, false);
    int rc;
    if (nch == 1) {
        if ((rc = decode_chunk(h, call, h->ws[0], d_obs, d_off, B, N, max_len, d_path, d_score, user, true))) return rc;
    } else {
        // fork: chunk k runs on internal stream k % 2 so that backtrace(k) overlaps forward(k+1)
        if (max_len <= 0) return fail(CV_ERR_ARG, "max_len is required for the chunked device path");
        CUDA_TRY(cudaEventRecord(h->ev_fork, user));
        for (int k = 0; k < 2; k++) CUDA_TRY(cudaStreamWaitEvent(h->ws[k].st, h->ev_fork, 0));
        for (int k = 0; k < nch; k++) {
            const int64_t b0 = B * k / nch, b1 = B * (k + 1) / nch;
            DecodeWs &w = h->ws[k & 1];
            if ((rc = decode_chunk(h, call, w, d_obs, d_off + b0, b1 - b0, N, max_len, d_path,
                                   d_score ? d_score + b0 : nullptr, w.st, false)))
                return rc;
        }
        for (int k = 0; k < 2; k++) {
            CUDA_TRY(cudaEventRecord(h->ws[k].done, h->ws[k].st));
            CUDA_TRY(cudaStreamWaitEvent(user, h->ws[k].done, 0));
        }
    }
    if (!sync_status && !call.timing) return CV_OK;
    return finish_call(h, call, nch == 1 ? 1 : 2, user, user);
}

extern "C" int cv_decode_batch_dev(cv_hmm *h, const uint32_t *d_obs, const int64_t *d_off, int64_t B, int64_t N,
                                   int64_t max_len, uint32_t *d_path, double *d_score, void *stream, int sync_status)
{
    return decode_batch_dev(h, decode_call(B), d_obs, d_off, N, max_len, d_path, d_score, stream, sync_status);
}

extern "C" int cv_decode_batch_dev_u8(cv_hmm *h, const uint32_t *d_obs, const int64_t *d_off, int64_t B, int64_t N,
                                      int64_t max_len, uint8_t *d_path, double *d_score, void *stream, int sync_status)
{
    if (!h) return fail(CV_ERR_ARG, "NULL model");
    if (h->K > SMALL_K_MAX) return fail(CV_ERR_UNSUPPORTED, "u8 paths are implemented for K <= %d", SMALL_K_MAX);
    return decode_batch_dev(h, decode_call(B, false, 0, 1), d_obs, d_off, N, max_len, reinterpret_cast<uint32_t *>(d_path),
                            d_score, stream, sync_status);
}

// preconditions of the f32 entry points
static int check_f32(const cv_hmm *h)
{
    if (!h) return fail(CV_ERR_ARG, "NULL model");
    if (!h->dA32f) return fail(CV_ERR_UNSUPPORTED, "the f32 mode is implemented for K <= %d", SMALL_K_MAX);
    if (!h->f32_range_ok) return fail(CV_ERR_UNSUPPORTED, "the f32 mode needs every finite model entry within |x| <= 2^64");
    return CV_OK;
}

extern "C" int cv_decode_batch_dev_f32(cv_hmm *h, const uint32_t *d_obs, const int64_t *d_off, int64_t B, int64_t N,
                                       int64_t max_len, uint32_t *d_path, double *d_score, void *stream, int sync_status)
{
    if (int rc = check_f32(h)) return rc;
    return decode_batch_dev(h, decode_call(B, true), d_obs, d_off, N, max_len, d_path, d_score, stream, sync_status);
}

// Streamed host path (K <= 64, large batches): ONE forward + backtrace launch over the whole batch while the
// observations still arrive chunk by chunk on a copy stream (each chunk followed by a stream write of the
// `arrived` word the forward CTAs poll) and the paths / scores of a chunk leave on another copy stream as soon as
// the backtrace has counted the chunk's sequences done (stream wait on chunk_done[c]).  The batch is ordered by
// (chunk, length), so the kernels consume the chunks in arrival order.  Against one launch per chunk this
// removes the per-chunk sort / launch / ramp costs: the copies hide behind 13 ms of kernels instead of 6 x 2.3 ms.
static int decode_streamed(cv_hmm *h, const DecodeCall &call, const uint32_t *obs_flat, const int64_t *seq_off,
                           uint32_t *path_out, double *score_out, int nch, bool *handled, uint32_t *d_path, double *d_score)
{
    *handled = false;
    const int64_t B = call.B;
    const size_t ob = call.obs_bytes(), pb = call.path_bytes();
    StreamValue32Fn wait32 = stream_wait_value32(), write32 = stream_write_value32();
    if (!g_tune.streamed || !g_tune.bt_concurrent || !wait32 || !write32 || nch < 2 || nch > STREAM_MAX_CHUNKS) return CV_OK;
    if (h->K > SMALL_K_MAX || chain_batch(h, call, B) || B > 0x7fffffffLL) return CV_OK;
    const int64_t N = seq_off[B];
    DecodeWs &w = h->ws[0];
    cudaStream_t sk = w.st, s_in = h->ws[1].st, s_out = h->ws[1].st_bt;
    uint32_t *d_obs = (uint32_t *)h->obs.p;
    int64_t *d_off = (int64_t *)h->seq_off.p;
    int rc;
    if ((rc = ensure_order_ws(w, B))) return rc;
    unsigned int *d_arrived = w.word(MISC_ARRIVED), *d_chunk_done = w.word(MISC_CHUNK_DONE);
    StreamedIO sio;
    sio.cbs.nch = nch;
    // Chunk sizes.  The forward kernel cannot start before chunk 0 is on the device and the last chunk's paths leave after
    // the kernels have ended, so both should be small -- but tiles are ordered by (chunk, length): every chunk starts with
    // its longest, most ragged tiles, and a small late chunk starts them when everything else is about to end (measured
    // with plain uneven chunks: 1/8, 3/8, 3/8, 1/8 13.45 vs 13.24 ms for four equal ones; six tapering chunks end the
    // kernels 0.5 ms later than five).  The automatic choice for large batches therefore cuts 10 / 25 / 25 / 20 / 12 / 8 %
    // and orders the LONG sequences of chunks 3.. with chunk 2 (ChunkBounds::promote_len): the late groups hold short,
    // even tiles only, a chunk's copy out fits into the work ordered behind it, and 8 % of the paths are copied after
    // the kernels.  A forced chunk count (cv_debug_set_chunks) gives equal chunks.
    sio.cbs.promote_len = 0; sio.cbs.promote_to = 0;
    if ((g_tune.chunks <= 0 && nch == 4 && g_tune.uneven_chunks) || (g_tune.uneven_chunks >= 2 && B >= 100)) {     // (2: forced, for tests)
        nch = 6;
        sio.cbs.nch = nch;
        static const int pct[7] = {0, 10, 35, 60, 80, 92, 100};
        for (int k = 0; k <= nch; k++) sio.cbs.cb[k] = B * pct[k] / 100;
        // a tile of a late group should take at most a quarter of the tile-steps a resident CTA runs for the last chunk
        const int64_t steps_per_cta = (seq_off[B] - seq_off[sio.cbs.cb[nch - 1]]) / ((int64_t)64 * 2 * h->num_sms);
        sio.cbs.promote_len = (int)std::max<int64_t>(4, std::min<int64_t>(steps_per_cta / 4, 1 << 20));
        sio.cbs.promote_to = 2;
    } else {
        for (int k = 0; k <= nch; k++) sio.cbs.cb[k] = B * k / nch;
    }
    sio.d_arrived = d_arrived; sio.d_chunk_done = d_chunk_done;

    // From here on copies from / to the caller's host buffers are in flight: every return (error or not) first drains
    // the three streams, so the caller may free or reuse its buffers as soon as this function returns.
    struct Drain { cudaStream_t s[3]; ~Drain() { for (cudaStream_t x : s) cudaStreamSynchronize(x); cudaGetLastError(); } } drain{{sk, s_in, s_out}};
    // CV_E2E_PROF=1: a timeline of this call (host clock for the enqueue / wait phases, events for the device phases)
    const bool prof = g_tune.e2e_prof != 0;
    cudaEvent_t pe[6] = {};
    const auto host_t0 = std::chrono::steady_clock::now();
    auto host_ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - host_t0).count(); };
    double hm_scan = 0.0, hm_enq = 0.0;
    if (prof) { for (auto &e : pe) cudaEventCreate(&e); cudaEventRecord(pe[0], sk); }
    // offsets first (the ordering needs nothing else), then the observations chunk by chunk on the copy stream
    CUDA_TRY(cudaMemsetAsync(w.misc.p, 0, MISC_BYTES, sk));
    CUDA_TRY(cudaMemcpyAsync(d_off, seq_off, sizeof(int64_t) * (size_t)(B + 1), cudaMemcpyHostToDevice, sk));
    CUDA_TRY(cudaEventRecord(w.ev_pre, sk));
    // `arrived` is zeroed first -- and the offsets have the link to themselves: the ordering (keys, sort) waits for them,
    // and two host-to-device copies in flight share the bandwidth (offsets + keys done at 0.5 instead of 0.25 ms)
    CUDA_TRY(cudaStreamWaitEvent(s_in, w.ev_pre, 0));
    for (int k = 0; k < nch; k++) {
        const int64_t e0 = seq_off[sio.cbs.cb[k]], e1 = seq_off[sio.cbs.cb[k + 1]];
        if (e1 < e0 || e1 > N) return fail(CV_ERR_ARG, "seq_off not monotone");
        if (e1 > e0) CUDA_TRY(cudaMemcpyAsync((char *)d_obs + ob * e0, (const char *)obs_flat + ob * e0, ob * (size_t)(e1 - e0), cudaMemcpyHostToDevice, s_in));
        if (write32(s_in, (unsigned long long)(uintptr_t)d_arrived, (unsigned int)(k + 1), 0x0) != 0) return fail(CV_ERR_CUDA, "cuStreamWriteValue32 failed");
    }
    CUDA_TRY(cudaEventRecord(h->ev_all_in, s_in));
    sio.all_in = h->ev_all_in;
    // the long-sequence split needs the longest length before the keys kernel: small batches only (host scan below
    // is moved up for them); large batches have nothing that long relative to their size
    LongSplit ls{0u, 0u, nullptr, nullptr, nullptr};
    int64_t max_len_host = 0;
    if (B <= (1 << 18)) {
        if ((rc = scan_lengths(seq_off, 0, B, max_len_host))) return rc;
        if (max_len_host <= 0xffffffLL && (rc = long_split_setup(h, call, w, B, N, max_len_host, sk, ls))) return rc;
    }
    // sort key = chunk field << shift | length: 24 bits of length when the longest one is not known yet, else just the
    // bits it needs (the sort then takes one or two 8-bit passes instead of four)
    sio.cbs.shift = (max_len_host > 0 && max_len_host <= 0xffffffLL) ? key_bits(max_len_host) : 24;
    seq_chunk_keys_kernel<<<(unsigned)((B + 255) / 256), 256, 0, sk>>>(d_off, B, sio.cbs, (uint32_t *)w.keys_in.p,
                                                                      (uint32_t *)w.vals_in.p, w.status(), w.word(MISC_MAX_LEN), ls);
    g_launches++;
    // Lengths are checked and the longest one is found before the launch (the history is sized from it).  Small
    // batches (a slice of a sharded batch): on the HOST while the first copies fly -- 0.1 ms per 100 k sequences and no
    // device round trip.  Large ones: by the keys kernel, read back with one ~0.2 ms synchronisation (a single host
    // thread would need ~0.7 ms for a million offsets, which delays the launch past the arrival of chunk 0).
    int64_t max_len = max_len_host;
    if (B > (1 << 18)) {
        int *hs = h->pinned<int>(PIN_STATUS);
        CUDA_TRY(cudaMemcpyAsync(hs, w.status(), 2 * sizeof(int), cudaMemcpyDeviceToHost, sk));  // MISC_STATUS, MISC_MAX_LEN
        CUDA_TRY(cudaStreamSynchronize(sk));
        if (hs[0] == CV_ERR_EMPTY) return fail(CV_ERR_EMPTY, "empty sequence in batch (reference: usize underflow panic)");
        if (hs[0] == CV_ERR_ARG) return fail(CV_ERR_ARG, "seq_off not monotone");
        if (hs[0]) { *handled = false; return CV_OK; }                                         // e.g. a sequence longer than 2^24: chunked path
        max_len = (int64_t)(unsigned int)hs[1];
    }
    if (max_len > 0xffffffLL) { *handled = false; return CV_OK; }                              // does not fit the 24-bit sort key: chunked path
    if (prof) { hm_scan = host_ms(); cudaEventRecord(pe[1], sk); cudaEventRecord(pe[4], s_in); }

    if ((rc = sort_desc(w, B, std::min(32, sio.cbs.shift + key_bits(nch - 1)), sk))) return rc;
    if (prof) cudaEventRecord(pe[2], sk);
    if ((rc = launch_decode_small(h, call, w, d_obs, d_off, B, N, d_path, d_score, max_len, sk, false, &sio, &ls))) return rc;
    if (prof) cudaEventRecord(pe[3], sk);
    // paths / scores of chunk c leave as soon as the backtrace has counted all its sequences
    CUDA_TRY(cudaStreamWaitEvent(s_out, w.ev_pre, 0));
    for (int k = 0; k < nch; k++) {
        const int64_t b0 = sio.cbs.cb[k], b1 = sio.cbs.cb[k + 1], e0 = seq_off[b0], e1 = seq_off[b1];
        if (b1 == b0) continue;
        if (wait32(s_out, (unsigned long long)(uintptr_t)(d_chunk_done + k), (unsigned int)(b1 - b0), 0x0 /* GEQ */) != 0)
            return fail(CV_ERR_CUDA, "cuStreamWaitValue32 failed");
        CUDA_TRY(cudaMemcpyAsync((char *)path_out + pb * e0, (const char *)d_path + pb * e0, pb * (size_t)(e1 - e0), cudaMemcpyDeviceToHost, s_out));
        if (score_out) CUDA_TRY(cudaMemcpyAsync(score_out + b0, d_score + b0, sizeof(double) * (size_t)(b1 - b0), cudaMemcpyDeviceToHost, s_out));
    }
    if (prof) { hm_enq = host_ms(); cudaEventRecord(pe[5], s_out); }
    const int status = finish_call(h, call, 1, sk);
    CUDA_TRY(cudaStreamSynchronize(s_out));
    CUDA_TRY(cudaStreamSynchronize(s_in));
    if (prof) {
        const double hm_end = host_ms();
        float t[6] = {};
        for (int i = 1; i < 6; i++) cudaEventElapsedTime(&t[i], pe[0], pe[i]);
        fprintf(stderr, "[cv] streamed B=%lld nch=%d | host: lengths known %.2f, all enqueued %.2f, done %.2f ms | device (from first enqueue): "
                        "offsets+keys %.2f, sorted %.2f, forward+backtrace done %.2f, last chunk in %.2f, last copy out %.2f ms\n",
                (long long)B, nch, hm_scan, hm_enq, hm_end, t[1], t[2], t[3], t[4], t[5]);
        for (auto &e : pe) cudaEventDestroy(e);
    }
    *handled = true;
    return status;
}

static int decode_batch_host(cv_hmm *h, const DecodeCall &call, const uint32_t *obs_flat, const int64_t *seq_off,
                             uint32_t *path_out, double *score_out, uint32_t *d_path_keep = nullptr, double *d_score_keep = nullptr)
{
    const int64_t B = call.B;
    if (!h) return fail(CV_ERR_ARG, "NULL model");
    if (B < 0) return fail(CV_ERR_ARG, "negative B");
    if (B == 0) return CV_OK;
    if (!obs_flat || !seq_off || !path_out) return fail(CV_ERR_ARG, "NULL buffer");
    if (seq_off[0] != 0) return fail(CV_ERR_ARG, "seq_off[0] must be 0");
    const int64_t N = seq_off[B];
    CUDA_TRY(cudaSetDevice(h->device));
    h->last_flagged = -1;
    int rc;
    if ((rc = h->obs.ensure(sizeof(uint32_t) * (size_t)N))) return rc;
    if ((rc = h->seq_off.ensure(sizeof(int64_t) * (size_t)(B + 1)))) return rc;
    if (!d_path_keep && (rc = h->path.ensure(sizeof(uint32_t) * (size_t)N))) return rc;
    if (!d_score_keep && (rc = h->score.ensure(sizeof(double) * (size_t)B))) return rc;
    // the device copies of the results: the library's own buffers, or the caller's (cv_decode_batch_keep)
    uint32_t *d_obs = (uint32_t *)h->obs.p, *d_path = d_path_keep ? d_path_keep : (uint32_t *)h->path.p;
    int64_t *d_off = (int64_t *)h->seq_off.p;
    double *d_score = d_score_keep ? d_score_keep : (double *)h->score.p;
    const int nch = chunk_count(h, call, true);
    const size_t ob = call.obs_bytes(), pb = call.path_bytes();
    if (!call.timing) {
        bool handled = false;
        if ((rc = decode_streamed(h, call, obs_flat, seq_off, path_out, score_out, nch, &handled, d_path, d_score))) return rc;
        if (handled) return CV_OK;
    }
    // Chunk k: H2D of its observations -> order/forward/backtrace -> D2H of its paths, on stream k % 2, so the
    // copies of one chunk overlap the kernels of its neighbours.  Offsets are validated while the first copy flies.
    std::vector<int64_t> cb;                                            // chunk boundaries (sequence indices)
    for (int k = 0; k <= nch; k++) cb.push_back(B * k / nch);
    const int nck = (int)cb.size() - 1;
    const bool e2e_prof = g_tune.e2e_prof != 0;      // prints a per-chunk timeline (copy in / kernels / copy out)
    std::vector<cudaEvent_t> pev;
    auto mark = [&](cudaStream_t s_) { if (e2e_prof) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, s_); pev.push_back(e); } };
    if (e2e_prof) { cudaDeviceSynchronize(); mark(h->ws[0].st); }
    for (int k = 0; k < nck; k++) {
        const int64_t b0 = cb[k], b1 = cb[k + 1];
        int64_t max_len = 0;
        if ((rc = scan_lengths(seq_off, b0, b1, max_len))) return rc;
        DecodeWs &w = h->ws[k & 1];
        cudaStream_t st = nch == 1 ? h->stream : w.st;
        const int64_t e0 = seq_off[b0], e1 = seq_off[b1];
        CUDA_TRY(cudaMemcpyAsync(d_off + b0, seq_off + b0, sizeof(int64_t) * (size_t)(b1 - b0 + 1), cudaMemcpyHostToDevice, st));
        mark(st);
        CUDA_TRY(cudaMemcpyAsync((char *)d_obs + ob * e0, (const char *)obs_flat + ob * e0, ob * (size_t)(e1 - e0), cudaMemcpyHostToDevice, st));
        mark(st);
        if ((rc = decode_chunk(h, call, w, d_obs, d_off + b0, b1 - b0, e1 - e0, max_len, d_path, d_score + b0, st, nck == 1))) return rc;
        mark(st);
        CUDA_TRY(cudaMemcpyAsync((char *)path_out + pb * e0, (const char *)d_path + pb * e0, pb * (size_t)(e1 - e0), cudaMemcpyDeviceToHost, st));
        if (score_out)
            CUDA_TRY(cudaMemcpyAsync(score_out + b0, d_score + b0, sizeof(double) * (size_t)(b1 - b0), cudaMemcpyDeviceToHost, st));
        mark(st);
    }
    if (e2e_prof) {
        cudaDeviceSynchronize();
        for (int k = 0; k < nck; k++) {
            float t[4];
            for (int i = 0; i < 4; i++) cudaEventElapsedTime(&t[i], pev[0], pev[1 + 4 * k + i]);
            fprintf(stderr, "[cv] chunk %d (%lld seqs): in %.2f-%.2f  kernels -%.2f  out -%.2f ms\n", k, (long long)(cb[k + 1] - cb[k]), t[0], t[1], t[2], t[3]);
        }
        for (cudaEvent_t e : pev) cudaEventDestroy(e);
    }
    return nch == 1 ? finish_call(h, call, 1, h->stream) : finish_call(h, call, 2, h->ws[0].st, h->ws[1].st);
}

extern "C" int cv_decode_batch(cv_hmm *h, const uint32_t *obs_flat, const int64_t *seq_off, int64_t B,
                               uint32_t *path_out, double *score_out)
{
    return decode_batch_host(h, decode_call(B), obs_flat, seq_off, path_out, score_out);
}

extern "C" int cv_decode_batch_keep(cv_hmm *h, const uint32_t *obs_flat, const int64_t *seq_off, int64_t B,
                                    uint32_t *path_out, double *score_out, uint32_t *d_path_keep, double *d_score_keep)
{
    if (!d_path_keep || !d_score_keep) return fail(CV_ERR_ARG, "NULL device buffer");
    return decode_batch_host(h, decode_call(B), obs_flat, seq_off, path_out, score_out, d_path_keep, d_score_keep);
}

extern "C" int cv_decode_batch_f32(cv_hmm *h, const uint32_t *obs_flat, const int64_t *seq_off, int64_t B,
                                   uint32_t *path_out, double *score_out)
{
    if (int rc = check_f32(h)) return rc;
    return decode_batch_host(h, decode_call(B, true), obs_flat, seq_off, path_out, score_out);
}

extern "C" int cv_decode_batch_u16u8(cv_hmm *h, const uint16_t *obs_flat, const int64_t *seq_off, int64_t B,
                                     uint8_t *path_out, double *score_out)
{
    if (!h) return fail(CV_ERR_ARG, "NULL model");
    if (h->M > 65536) return fail(CV_ERR_UNSUPPORTED, "u16 observations need M <= 65536 (M = %lld)", (long long)h->M);
    if (h->K > 256) return fail(CV_ERR_UNSUPPORTED, "u8 paths need K <= 256 (K = %d)", h->K);
    if (h->K > SMALL_K_MAX) return fail(CV_ERR_UNSUPPORTED, "the narrow host formats are implemented for K <= %d", SMALL_K_MAX);
    return decode_batch_host(h, decode_call(B, false, 1, 1), reinterpret_cast<const uint32_t *>(obs_flat), seq_off,
                             reinterpret_cast<uint32_t *>(path_out), score_out);
}
