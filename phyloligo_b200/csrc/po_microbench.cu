// Pipe-peak microbenchmarks used as roofline denominators for the CUDA-core
// distance kernels (MEASURED_PEAKS.json holds only HBM and bf16 tensor peaks).
//   kind 0: dependent-chain-free FFMA throughput, TFLOP/s (2 flop per FFMA)
//   kind 1: MUFU.LG2 throughput, 1e12 op/s
//   kind 2: POPC throughput, 1e12 op/s
//   kind 3: MUFU.RCP throughput (rcp.approx.ftz.f32, the t-SNE repulsion's reciprocal), 1e12 op/s
//   kind 4: grid-barrier latency, microseconds per grid.sync() of the linkage kernels' grid (po_linkage.cu)
// Operand-bandwidth kinds (DESIGN.md section 4.3): which packed-f32x2 forms the FP32 pipe of po_jsd.cu's
// chunk loops sustains at its full rate, counted in warp-instructions per SM per clock (the SM clock is
// measured inside the kernel, clock64 against %globaltimer).  64 independent chains per thread:
//   kind 5:  FFMA2, three register pairs, different ones in every chain (6 register reads per lane)
//   kind 6:  FFMA2, two register pairs + an immediate (4 reads)
//   kind 7:  FFMA2, three register pairs, multiplier and addend shared by all chains (.reuse hits)
//   kind 8:  FFMA2, two register pairs, the multiplier shared by all chains, + an immediate
//   kind 9:  FFMA2, a scalar-broadcast .F32 multiplier + an immediate (3 reads)
//   kind 10: FADD2, a scalar-broadcast .F32 operand + a register pair (3 reads)
//   kind 11: FMUL2 x*x, the same register pair in both slots
//   kind 12: the V0 recipe of po_jsd.cu (FADD2, FADD2-negate with the broadcast row value, 2 MUFU.RCP,
//            3 FMUL2, 4 Horner FFMA2, the accumulating FFMA2): packed FP32 instructions per SM per clock
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

typedef unsigned long long u64;
__device__ __forceinline__ u64 ub_pk2(float lo, float hi) {
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ u64 ub_fma2(u64 a, u64 b, u64 c) {
    u64 r;
    asm volatile("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ u64 ub_add2(u64 a, u64 b) {
    u64 r;
    asm volatile("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ u64 ub_sub2(u64 a, u64 b) {
    u64 r;
    asm volatile("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ u64 ub_mul2(u64 a, u64 b) {
    u64 r;
    asm volatile("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ float ub_rcp(float x) {
    float y;
    asm volatile("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// t[0..1]: clock64 and %globaltimer (ns) at the start and end of CTA 0, for the SM clock of the run
template <int KIND>
__global__ void __launch_bounds__(256) operand_kernel(float* sink, long long* t, int iters) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        long long g;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
        t[0] = clock64();
        t[1] = g;
    }
    constexpr int C = 8;  // chains per rep; 8 reps per iteration
    u64 a[C], m[C], c[C];
    float sc[C];
#pragma unroll
    for (int i = 0; i < C; ++i) {
        const float f = 1.0f + 1e-3f * (float)(threadIdx.x + i);
        a[i] = ub_pk2(f, f + 0.5f);
        // operands from the thread index, so that ptxas cannot fold them into immediates or uniform registers
        m[i] = ub_pk2(0.999f - 1e-6f * (float)(threadIdx.x + i), 0.998f - 1e-9f * (float)threadIdx.x);
        c[i] = ub_pk2(1e-7f * (float)(threadIdx.x + i + 1), 2e-7f * (float)(threadIdx.x + 1));
        sc[i] = 0.999f - 1e-5f * (float)(threadIdx.x & (i + 1));
    }
    const u64 M = ub_pk2(0.999f - 1e-6f * (float)(threadIdx.x & 7), 0.998f), Cc = ub_pk2(1e-7f * (float)(threadIdx.x & 3), 2e-7f);
    const u64 imm = ub_pk2(1e-7f, 1e-7f);
    const u64 h4 = ub_pk2(3.614963273e-02f, 3.614963273e-02f), h3 = ub_pk2(3.220779540e-02f, 3.220779540e-02f);
    const u64 h2 = ub_pk2(6.700734910e-02f, 6.700734910e-02f), h1 = ub_pk2(1.666553656e-01f, 1.666553656e-01f);
    const u64 h0 = ub_pk2(1.000000059e+00f, 1.000000059e+00f);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int rep = 0; rep < 8; ++rep) {
#pragma unroll
            for (int i = 0; i < C; ++i) {
                if (KIND == 5) a[i] = ub_fma2(a[i], m[i], c[i]);
                if (KIND == 6) a[i] = ub_fma2(a[i], m[i], imm);
                if (KIND == 7) a[i] = ub_fma2(a[i], M, Cc);
                if (KIND == 8) a[i] = ub_fma2(a[i], M, imm);
                if (KIND == 9) a[i] = ub_fma2(a[i], ub_pk2(sc[i], sc[i]), imm);
                if (KIND == 10) a[i] = ub_add2(ub_pk2(sc[i], sc[i]), a[i]);
                if (KIND == 11) a[i] = ub_mul2(a[i], a[i]);
                if (KIND == 12) {
                    // one packed term pair of the V0 loop: row value sc[i] against the pair a[i]
                    const u64 sa = ub_pk2(sc[i], sc[i]);
                    const u64 s2 = ub_add2(sa, a[i]);
                    const u64 d2 = ub_sub2(sa, a[i]);
                    float s0, s1;
                    asm("mov.b64 {%0, %1}, %2;" : "=f"(s0), "=f"(s1) : "l"(s2));
                    const u64 x = ub_mul2(d2, ub_pk2(ub_rcp(s0), ub_rcp(s1)));
                    const u64 u = ub_mul2(x, x);
                    u64 G = ub_fma2(h4, u, h3);
                    G = ub_fma2(G, u, h2);
                    G = ub_fma2(G, u, h1);
                    G = ub_fma2(G, u, h0);
                    a[i] = ub_fma2(ub_mul2(d2, x), G, a[i]);
                }
            }
        }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < C; ++i) {
        float lo, hi;
        asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a[i]));
        s += lo + hi;
    }
    if (s == 123.456f) sink[0] = s;
    __syncthreads();
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        long long g;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g));
        t[2] = clock64();
        t[3] = g;
    }
}

// kinds 5..12: warp-instructions (kind 12: packed FP32 instructions) per SM per clock
static int operand_rate(int kind, double* result) {
    int dev = 0, sms = 0;
    PO_CUDA_CHECK(cudaGetDevice(&dev));
    PO_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    float* sink = nullptr;
    long long* t = nullptr;
    PO_CUDA_CHECK(cudaMalloc(&sink, 4));
    PO_CUDA_CHECK(cudaMalloc(&t, 4 * sizeof(long long)));
    const int iters = (kind == 12) ? 512 : 4096;
    const int blocks = sms * 8;
    cudaEvent_t e0, e1;
    PO_CUDA_CHECK(cudaEventCreate(&e0));
    PO_CUDA_CHECK(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0, 0);
        switch (kind) {
            case 5: operand_kernel<5><<<blocks, 256>>>(sink, t, iters); break;
            case 6: operand_kernel<6><<<blocks, 256>>>(sink, t, iters); break;
            case 7: operand_kernel<7><<<blocks, 256>>>(sink, t, iters); break;
            case 8: operand_kernel<8><<<blocks, 256>>>(sink, t, iters); break;
            case 9: operand_kernel<9><<<blocks, 256>>>(sink, t, iters); break;
            case 10: operand_kernel<10><<<blocks, 256>>>(sink, t, iters); break;
            case 11: operand_kernel<11><<<blocks, 256>>>(sink, t, iters); break;
            default: operand_kernel<12><<<blocks, 256>>>(sink, t, iters); break;
        }
        cudaEventRecord(e1, 0);
        PO_CUDA_CHECK(cudaEventSynchronize(e1));
        PO_LAUNCH_CHECK("operand_kernel");
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        long long h[4];
        PO_CUDA_CHECK(cudaMemcpy(h, t, sizeof(h), cudaMemcpyDeviceToHost));
        const double ghz = (double)(h[2] - h[0]) / (double)(h[3] - h[1]);  // cycles per ns of CTA 0
        const double per_unit = (kind == 12) ? 10.0 : 1.0;
        const double warp_inst = (double)blocks * (256 / 32) * (double)iters * 64.0 * per_unit;
        const double rate = warp_inst / (ms * 1e6 * ghz) / (double)sms;
        if (rep > 0 && rate > best) best = rate;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    cudaFree(t);
    *result = best;
    return PO_OK;
}

}  // namespace po

extern "C" int po_microbench(int kind, double* result) {
    using namespace po;
    if (kind < 0 || kind > 12 || !result) {
        set_error("po_microbench: bad arguments");
        return PO_ERR_ARG;
    }
    if (kind == 4) return barrier_latency_us(result);
    if (kind >= 5) return operand_rate(kind, result);
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
