// cv_debug.cu -- test / bench hooks of include/cv_b200_debug.h: tuning setters and the FP64 issue-rate probe that
// bench.py uses as the roofline denominator.  Nothing here is on a product path.
#include "cv_internal.cuh"

#include "common.cuh"
#include "probe.cuh"

using namespace cvb;

extern "C" void cv_debug_set_chunks(int n) { g_tune.chunks = n; }
extern "C" void cv_debug_set_chain_max_batch(long long b) { g_tune.chain_max_b = b; }
extern "C" void cv_debug_set_pipeline(int bt_concurrent, int streamed)
{
    if (bt_concurrent >= 0) g_tune.bt_concurrent = bt_concurrent;
    if (streamed >= 0) g_tune.streamed = streamed;
}
extern "C" void cv_debug_set_balanced_split(int on) { g_tune.balanced_split = on; }
extern "C" void cv_debug_set_fwd_ldc(int on) { g_tune.fwd_ldc = on; }
extern "C" void cv_debug_set_em_light(int on) { g_tune.em_light = on; }
extern "C" void cv_debug_set_bt_split(int on) { g_tune.bt_split = on; }
extern "C" void cv_debug_set_uneven_chunks(int on) { g_tune.uneven_chunks = on; }
extern "C" void cv_debug_set_large_group_rb(long long rb) { g_tune.large_group_rb = rb; }
extern "C" void cv_debug_set_cp_leaf_batch(int on) { g_tune.cp_leaf_batch = on; }
extern "C" void cv_debug_set_fb_chunk_seqs(int64_t n) { g_tune.fb_chunk_seqs = n; }
extern "C" void cv_debug_set_kbest_chunk_seqs(int64_t n) { g_tune.kbest_chunk_seqs = n; }
extern "C" void cv_debug_set_certified(int on) { g_tune.certified = on; }
extern "C" void cv_debug_set_cert_tolerance(double scale) { g_tune.cert_tol = scale; }
extern "C" int64_t cv_debug_last_flagged(const cv_hmm *h) { return h ? h->last_flagged : -1; }
extern "C" void cv_debug_set_fallback(int route, long long n_chain) { g_tune.fb_route = route; g_tune.fb_chain = n_chain; }
extern "C" int64_t cv_debug_last_fallback_chain(const cv_hmm *h) { return h ? h->last_fb_chain : 0; }

// ---------------------------------------------------------------------------
// FP64 probe
// ---------------------------------------------------------------------------
extern "C" int cv_debug_probe_fp64(int device, int mode, int iters, double *ops_per_s_out, double *ms_out)
{
    int rc = check_device(device < 0 ? 0 : device);
    if (rc) return rc;
    if (device >= 0) CUDA_TRY(cudaSetDevice(device));
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
    if (mode != 0 && mode != 1 && mode != 25) return fail(CV_ERR_ARG, "unknown probe mode %d", mode);
    const int threads = 384;
    const int blocks = prop.multiProcessorCount;
    double *d_out = nullptr;
    CUDA_TRY(cudaMalloc(&d_out, sizeof(double) * (size_t)threads * blocks));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    double fp64_ops = 0.0;
    for (int rep = 0; rep < 2; rep++) {   // rep 0 = warm-up
        CUDA_TRY(cudaEventRecord(e0));
        if (mode == 0) {
            probe_fp64_kernel<0><<<blocks, threads>>>(d_out, iters, 1.0);
            fp64_ops = 16.0 * iters * threads * blocks;
        } else if (mode == 1) {
            probe_fp64_kernel<1><<<blocks, threads>>>(d_out, iters, 1.0);
            fp64_ops = 32.0 * iters * threads * blocks;
        } else {
            probe_fp64_kernel<2><<<blocks, threads>>>(d_out, iters, 1.0);   // independent DFMA chains (Baum-Welch cell)
            fp64_ops = 16.0 * iters * threads * blocks;                      // FMAs
        }
        g_launches++;
        CUDA_TRY(cudaEventRecord(e1));
        CUDA_TRY(cudaEventSynchronize(e1));
        CUDA_TRY(cudaGetLastError());
    }
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
    if (ops_per_s_out) *ops_per_s_out = fp64_ops / (ms * 1e-3);
    if (ms_out) *ms_out = ms;
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d_out);
    return CV_OK;
}

