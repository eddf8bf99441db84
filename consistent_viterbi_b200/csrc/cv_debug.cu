// cv_debug.cu -- test / bench hooks of include/cv_b200_debug.h: tuning setters and the FP64 issue-rate probe that
// bench.py uses as the roofline denominator.  Nothing here is on a product path.
#include "cv_internal.cuh"

#include "common.cuh"
#include "probe.cuh"

using namespace cvb;

extern "C" void cv_debug_set_small_config(int cfg) { g_tune.small_cfg = cfg; }
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
extern "C" void cv_debug_set_prefilter(int on) { g_tune.prefilter = on; }
extern "C" void cv_debug_set_large_group_rb(long long rb) { g_tune.large_group_rb = rb; }
extern "C" void cv_debug_set_cp_leaf_batch(int on) { g_tune.cp_leaf_batch = on; }

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
    const int threads = g_tune.probe_threads;
    const int blocks = prop.multiProcessorCount;
    double *d_out = nullptr;
    CUDA_TRY(cudaMalloc(&d_out, sizeof(double) * (size_t)threads * blocks));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    const int K = 45;
    const size_t smem = (size_t)K * 48 * 8 + (size_t)K * ((threads / 32 + 5) / 6) * 64 * 8;
    double fp64_ops = 0.0;
    for (int rep = 0; rep < 2; rep++) {   // rep 0 = warm-up
        CUDA_TRY(cudaEventRecord(e0));
        if (mode == 0) {
            probe_fp64_kernel<0><<<blocks, threads>>>(d_out, iters, 1.0);
            fp64_ops = 16.0 * iters * threads * blocks;
        } else if (mode == 1) {
            probe_fp64_kernel<1><<<blocks, threads>>>(d_out, iters, 1.0);
            fp64_ops = 32.0 * iters * threads * blocks;
        } else if (mode == 25) {
            probe_fp64_kernel<2><<<blocks, threads>>>(d_out, iters, 1.0);   // independent DFMA chains (Baum-Welch cell)
            fp64_ops = 16.0 * iters * threads * blocks;                      // FMAs
        } else {
            auto launch = [&](auto kern) -> cudaError_t {
                cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                if (e != cudaSuccess) return e;
                kern<<<blocks, threads, smem>>>(d_out, K, iters, 0, 1.0);
                return cudaSuccess;
            };
            auto launch_val = [&](auto kern) -> cudaError_t {
                cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                if (e != cudaSuccess) return e;
                kern<<<blocks, threads, smem>>>(d_out, K, iters, 1.0);
                return cudaSuccess;
            };
            cudaError_t e = cudaSuccess;
            switch (mode) {
                case 2: e = launch(probe_tile_kernel<0>); break;
                case 3: e = launch(probe_tile_kernel<1>); break;
                case 4: e = launch(probe_tile_kernel<2>); break;
                case 5: e = launch(probe_tile_kernel<3>); break;
                case 6: e = launch_val(probe_tile_val_kernel<2>); break;
                case 20: e = launch_val(probe_tile_val_kernel<3>); break;
                case 21: e = launch_val(probe_tile_val_kernel<4>); break;
                case 22: e = launch_val(probe_tile_val_kernel<5>); break;
                case 23: e = launch_val(probe_tile_val_kernel<9>); break;
                case 24: e = launch_val(probe_tile_val_kernel<0>); break;
                case 7: probe_mix_kernel<1, 1><<<blocks, threads>>>(d_out, iters, 1.0); break;
                case 8: probe_mix_kernel<1, 2><<<blocks, threads>>>(d_out, iters, 1.0); break;
                case 9: probe_mix_kernel<0, 3><<<blocks, threads>>>(d_out, iters, 1.0); break;
                case 10: probe_mix_kernel<1, 0><<<blocks, threads>>>(d_out, iters, 1.0); break;
                case 17: probe_tile_val_reg_kernel<<<blocks, threads>>>(d_out, K, iters, 1.0); break;
                case 18: probe_tile_val_var_kernel<1><<<blocks, threads>>>(d_out, K, iters, 1.0); break;
                case 19: probe_tile_val_var_kernel<2><<<blocks, threads>>>(d_out, K, iters, 1.0); break;
                case 14: probe_mix_alu_kernel<1, 1><<<blocks, threads>>>(d_out, iters, 1.0); break;
                case 15: probe_mix_alu_kernel<1, 2><<<blocks, threads>>>(d_out, iters, 1.0); break;
                case 16: probe_mix_alu_kernel<0, 2><<<blocks, threads>>>(d_out, iters, 1.0); break;
                case 11: case 12: case 13: {
                    long long *d_cyc = nullptr, h_cyc = 0;
                    CUDA_TRY(cudaMalloc(&d_cyc, sizeof(long long)));
                    if (mode == 11) probe_latency_kernel<0><<<1, 32>>>(d_out, iters, 1.0, d_cyc);
                    else if (mode == 12) probe_latency_kernel<1><<<1, 32>>>(d_out, iters, 1.0, d_cyc);
                    else probe_latency_kernel<2><<<1, 32>>>(d_out, iters, 1.0, d_cyc);
                    CUDA_TRY(cudaMemcpy(&h_cyc, d_cyc, sizeof(long long), cudaMemcpyDeviceToHost));
                    cudaFree(d_cyc);
                    if (ms_out) *ms_out = (double)h_cyc / (16.0 * iters);      // cycles per dependent op
                    if (ops_per_s_out) *ops_per_s_out = (double)h_cyc / (16.0 * iters);
                    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d_out);
                    g_launches++;
                    return CV_OK;
                }
                default: return fail(CV_ERR_ARG, "unknown probe mode %d", mode);
            }
            CUDA_TRY(e);
            fp64_ops = 2.0 * 16.0 * K * (double)iters * threads * blocks;   // DADD + DSETP per cell
            if (mode >= 7) fp64_ops = 8.0 * (double)iters * threads * blocks;   // DADD count (8 chains) per iteration
            if (mode >= 17) fp64_ops = 2.0 * 16.0 * K * (double)iters * threads * blocks;
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

