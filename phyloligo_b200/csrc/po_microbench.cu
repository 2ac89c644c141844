// Pipe-peak microbenchmarks used as roofline denominators for the CUDA-core
// distance kernels (MEASURED_PEAKS.json holds only HBM and bf16 tensor peaks).
//   kind 0: dependent-chain-free FFMA throughput, TFLOP/s (2 flop per FFMA)
//   kind 1: MUFU.LG2 throughput, 1e12 op/s
//   kind 2: POPC throughput, 1e12 op/s
//   kind 3: MUFU.RCP throughput (rcp.approx.ftz.f32, the t-SNE repulsion's reciprocal), 1e12 op/s
//   kind 4: grid-barrier latency, microseconds per grid.sync() of the linkage kernels' grid (po_linkage.cu)
#include "po_common.cuh"

namespace po {

template <int KIND>
__global__ void __launch_bounds__(256) pipe_peak_kernel(float* sink, int iters) {
    float a[8];
    unsigned u[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        a[i] = 1.0f + 0.001f * (float)(threadIdx.x + i);
        u[i] = 0x9E3779B9u * (threadIdx.x + i + 1);
    }
    const float m = 0.999999f, c = 1e-7f;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int rep = 0; rep < 8; ++rep) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                if (KIND == 0) a[i] = fmaf(a[i], m, c);
                if (KIND == 1) asm volatile("lg2.approx.f32 %0, %0;" : "+f"(a[i]));
                if (KIND == 2) u[i] = __popc(u[i]) + u[i];
                if (KIND == 3) {  // the add keeps ptxas from folding rcp(rcp(x)) = x; the FP32 pipe has 8x the MUFU rate
                    asm volatile("rcp.approx.ftz.f32 %0, %0;" : "+f"(a[i]));
                    a[i] += c;
                }
            }
        }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += a[i] + (float)u[i];
    if (s == 123.456f) sink[0] = s;
}

}  // namespace po

extern "C" int po_microbench(int kind, double* result) {
    using namespace po;
    if (kind < 0 || kind > 4 || !result) {
        set_error("po_microbench: bad arguments");
        return PO_ERR_ARG;
    }
    if (kind == 4) return barrier_latency_us(result);
    int dev = 0, sms = 0;
    PO_CUDA_CHECK(cudaGetDevice(&dev));
    PO_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    float* sink = nullptr;
    PO_CUDA_CHECK(cudaMalloc(&sink, 4));
    const int iters = (kind == 0) ? 4096 : 1024;
    const int blocks = sms * 8;
    cudaEvent_t e0, e1;
    PO_CUDA_CHECK(cudaEventCreate(&e0));
    PO_CUDA_CHECK(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0, 0);
        if (kind == 0) pipe_peak_kernel<0><<<blocks, 256>>>(sink, iters);
        if (kind == 1) pipe_peak_kernel<1><<<blocks, 256>>>(sink, iters);
        if (kind == 2) pipe_peak_kernel<2><<<blocks, 256>>>(sink, iters);
        if (kind == 3) pipe_peak_kernel<3><<<blocks, 256>>>(sink, iters);
        cudaEventRecord(e1, 0);
        PO_CUDA_CHECK(cudaEventSynchronize(e1));
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        const double ops = (double)blocks * 256.0 * (double)iters * 64.0;
        const double rate = ops / (ms * 1e-3) / 1e12 * (kind == 0 ? 2.0 : 1.0);
        if (rep > 0 && rate > best) best = rate;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    *result = best;
    return PO_OK;
}
