// Euclidean distance tiles on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.
//
// Replaces euclidean_distances_loc / euclidean_distances_h5py -> sklearn
// euclidean_distances (reference bin/phyloligo.py:200-202, 238-246: the Gram form
// ||x||^2 + ||y||^2 - 2 x.y, clamped at 0, square root, exact 0 on the diagonal) and
// phylodist.Eucl (core/phylodist.py:36-41) for profile dimensions >= 256.
//
// Numerics.  The Gram form cancels, so the operands are conditioned first:
//   * centring: x' = x - mean profile (a Euclidean distance is translation invariant);
//     ||x'|| is then of the order of the distances themselves instead of ~1/sqrt(D);
//   * x' * 2^14 is split into two float16 values hi + lo (22 significant bits); the tensor
//     cores form hi.hi in one float32 accumulator in TMEM and hi.lo + lo.hi in a second one
//     (the dropped lo.lo term is 2^-22 relative) and the epilogue adds them.  The order of the
//     two cross MMAs is mirrored below the diagonal and diagonal groups copy their lower half
//     from their upper half, so (r, c) and (c, r) are the same float32 sums and the matrix is
//     bitwise symmetric whichever tile computes an entry;
//   * the row norms are float64 sums over the very same hi + lo values, and the epilogue
//     evaluates n_a + n_b - 2 dot in float64.
//   * entries whose Gram form cancels by more than 2^8 (n_a + n_b > 256 d^2: near-duplicate
//     profiles; 2^3 with the e4m3 cross terms below) are recomputed exactly as sum (a-b)^2 by the
//     warp that owns them, from a float32 copy of the profiles kept next to the operand blocks.
//   * cross terms in e4m3 (from 1024 dimensions up; PO_EUCL_CROSS=f16 keeps them in float16): hi.lo + lo.hi is 2^-11
//     of the dot product, so three mantissa bits are enough for it -- both factors are stored a
//     second time as e4m3 (power-of-two scales from the largest |x'| of the matrix) and the two cross
//     MMAs run as kind::f8f6f4 with K = 32, i.e. at half the cost of their float16 form: 2 MMA units per
//     16 dimensions instead of 3.  Error against float64: ~2e-6 relative for ordinary pairs (float16
//     cross terms: ~2e-8), below 4e-5 at the recomputation threshold; the stated tolerance is 1e-4.
// Measured error against a float64 evaluation is ~1e-8 relative for ordinary pairs and below
// 5e-5 at the cancellation threshold; the stated tolerance of this path is 1e-4
// (BASELINE.json north_star).  PO_EUCL_EXACT=1 (or dim < 256) selects
// the exact CUDA-core kernel of po_distance.cu instead.
//
// Layout.  po_prepare_profiles writes, for every group of 128 profiles and every block of
// 64 dimensions, the hi block and the lo block (16 KB each) in the canonical no-swizzle
// K-major UMMA shared-memory layout: 8x16-byte core matrices, 128 B apart along the rows
// and 2 KB apart along K.  A CTA of 16 warps computes one tile (Eucl: 128 x 256, two column
// groups sharing the row operand; SC: 128 x 128): one thread streams the operand blocks of a K
// stage with cp.async.bulk into a shared-memory ring, one thread issues the tcgen05.mma
// (128x128x16, kind::f16) of the stage and commits them to the stage's "empty" barrier, and after
// the last commit all warps read the accumulators with tcgen05.ld, finish the distances and
// store the tile (and its mirror) with coalesced stores.
#include <cuda_fp16.h>
#include <cuda_fp8.h>
#include <stdlib.h>
#include "po_common.cuh"
#include "po_rank.cuh"

namespace po {

constexpr int GT = 128;                 // tile edge (M = N = 128)
constexpr int GK = 64;                  // K elements per block (4 MMAs of K = 16)
constexpr int GBLOCK_BYTES = GT * GK * 2;     // one operand block: 16 KB
constexpr int GRASTER = 16;             // 128-column groups per rasterisation chunk
constexpr float GSCALE = 16384.0f;      // 2^14
constexpr double GUNSCALE = 1.0 / (16384.0 * 16384.0);

bool eucl_use_gram(int metric, int64_t dim) {
    if (metric != PO_EUCL_GRAM) return false;
    const char* e = getenv("PO_EUCL_EXACT");
    if (e && e[0] == '1') return false;
    return dim >= 256;
}
int64_t gram_ldk(int64_t dim) { return (dim + GK - 1) / GK * GK; }
constexpr int GSUM_SLICES = 256;  // row slices of the two-stage (order-fixed, reproducible) column sums
// operand blocks, then the float64 column sums used for centring, then a float32 copy of the
// profiles (row pitch ldk) for the exact recomputation of cancelling entries, then the
// per-slice partial column sums
int64_t gram_prepared_bytes(int64_t n, int64_t dim) {
    const int64_t npad = (n + GT - 1) / GT * GT;
    const int64_t ldk = gram_ldk(dim);
    return npad * ldk * 4 + ldk * 8 + n * ldk * 4 + (int64_t)GSUM_SLICES * ldk * 8 + 64;  // + absmax / e4m3 scales
}
// e4m3 cross terms from 1024 dimensions up, float16 cross terms below (or everywhere with PO_EUCL_CROSS=f16);
// read at prepare AND at launch.  The e4m3 rounding of the cross terms is bounded by ~3e-5 C relative on a
// distance (C = cancellation factor, entries with C > 8 are recomputed exactly) and averages out over the
// dimensions: measured 6.5e-7 at 4096 dimensions but 2e-5 on short-contig 256-dimension profiles, too close
// to the stated 1e-4 -- and at 256 dimensions the kernel is bound by its epilogue, not by the MMAs.
static bool eucl_cross8(int64_t dim) {
    const char* e = getenv("PO_EUCL_CROSS");
    if (e && e[0] == 'f' && e[1] == '1' && e[2] == '6') return false;
    return dim >= 1024;
}

// Spearman on the same kernel.  1 - rho is a Gram form as well: with r' = 2 rank - (dim + 1) (integer,
// centred; average ranks for ties -- the scipy.stats.spearmanr step of phylodist.SC, reference
// core/phylodist.py:82-85), rho = r'_a . r'_b / sqrt(|r'_a|^2 |r'_b|^2).  r' is split into two
// integer digits r' = 64 h + l, l in [-32, 31], both exact in float16; the tensor cores form
// h.h', h.l', l.h' and l.l' in four TMEM accumulators.  Every product and every partial sum
// is an integer below 2^24 for dim <= 4096, so the float32 accumulators are exact and the epilogue
// rebuilds the integer dot product 4096 hh + 64 (hl + lh) + ll: the result is bit for bit that of the
// CUDA-core kernel (po_distance.cu, K_SC).  PO_SC_CUDA_CORES=1 selects that kernel instead.
bool sc_use_gram(int metric, int64_t dim) {
    if (metric != PO_SC) return false;
    const char* e = getenv("PO_SC_CUDA_CORES");
    if (e && e[0] == '1') return false;
    return dim >= 64 && dim <= 4096;
}
// Digits as int8 for kind::i8 MMAs (default: r' = 128 h + l, l in [-64, 63], |h| <= 32; int32 accumulators,
// exact by construction, K = 32 per MMA: half the tensor time of the float16 digits) or as float16
// (PO_SC_DIGITS=f16: r' = 64 h + l).  Read at prepare AND at launch.
static bool sc_digits8() {
    const char* e = getenv("PO_SC_DIGITS");
    return !(e && e[0] == 'f' && e[1] == '1' && e[2] == '6');
}
int64_t sc_gram_prepared_bytes(int64_t n, int64_t dim) {
    const int64_t npad = (n + GT - 1) / GT * GT;
    return npad * gram_ldk(dim) * 4;  // the int8 digits use the first half
}

// ---------------------------------------------------------------------------------------------
// operand preparation
// ---------------------------------------------------------------------------------------------
// Column sums in two stages with a fixed summation order (no atomics): the result must be
// bit-reproducible, every rank of a multi-GPU run prepares the same operands.
template <typename T>
__global__ void __launch_bounds__(256) gram_colsum_kernel(const T* __restrict__ X, int64_t n, int64_t dim, int64_t ldx,
                                                          double* __restrict__ partial, int64_t ldk) {
    const int64_t col = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (col >= dim) return;
    const int64_t rows_per = (n + GSUM_SLICES - 1) / GSUM_SLICES;
    const int64_t r0 = (int64_t)blockIdx.y * rows_per, r1 = min(n, r0 + rows_per);
    double s = 0.0;
    for (int64_t r = r0; r < r1; ++r) s += (double)X[r * ldx + col];
    partial[(int64_t)blockIdx.y * ldk + col] = s;
}
__global__ void __launch_bounds__(256) gram_colsum_final_kernel(const double* __restrict__ partial, int64_t dim,
                                                                int64_t ldk, double* __restrict__ sums) {
    const int64_t col = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (col >= ldk) return;
    double s = 0.0;
    if (col < dim)
        for (int y = 0; y < GSUM_SLICES; ++y) s += partial[(int64_t)y * ldk + col];
    sums[col] = s;
}

// largest |x - mean| * 2^14 of the matrix (a maximum: order independent, reproducible)
template <typename T>
__global__ void __launch_bounds__(256) gram_absmax_kernel(const T* __restrict__ X, int64_t n, int64_t dim, int64_t ldx,
                                                          const double* __restrict__ sums, unsigned* __restrict__ absmax_bits) {
    const double inv_n = 1.0 / (double)n;
    float m = 0.f;
    const int64_t total = n * dim;
    for (int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x; e < total; e += (int64_t)gridDim.x * 256) {
        const int64_t r = e / dim, k = e - r * dim;
        m = fmaxf(m, fabsf(((float)X[r * ldx + k] - (float)(sums[k] * inv_n)) * GSCALE));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(absmax_bits, __float_as_uint(m));
}
// scales[1] = alpha (hi -> e4m3: the largest value lands in [128, 256)), [2] = beta = 2^11 alpha (lo), [3] = 1 / (alpha beta)
__global__ void gram_scales_kernel(float* scales) {
    const float amax = __uint_as_float(reinterpret_cast<const unsigned*>(scales)[0]);
    int e = 0;
    float alpha = 1.f;
    if (amax > 0.f && amax < 3.0e38f) {
        frexpf(amax, &e);  // amax = m 2^e, m in [0.5, 1)
        alpha = ldexpf(1.f, 8 - e);
    }
    scales[1] = alpha;
    scales[2] = alpha * 2048.f;
    scales[3] = 1.f / (alpha * alpha * 2048.f);
}

// One CTA per group of 128 profiles; the K blocks are walked in order so that a row's squared
// norm is accumulated in a fixed order (reproducible, no atomics).  CROSS8: per 64-dimension block the
// float16 hi plane (16 KB), then hi and lo as e4m3 (8 KB each; core matrices of 8 rows x 16 elements).
template <typename T, bool CROSS8>
__global__ void __launch_bounds__(256) gram_blocks_kernel(const T* __restrict__ X, int64_t n, int64_t dim, int64_t ldx,
                                                          const double* __restrict__ sums, unsigned char* __restrict__ P,
                                                          int nkb, double* __restrict__ aux, float* __restrict__ X32,
                                                          const float* __restrict__ scales) {
    const float alpha = CROSS8 ? scales[1] : 1.f, beta = CROSS8 ? scales[2] : 1.f;
    const int64_t grp = blockIdx.x;
    const double inv_n = 1.0 / (double)n;
    double nrm[4] = {0.0, 0.0, 0.0, 0.0};
    for (int kb = 0; kb < nkb; ++kb) {
        unsigned char* blk_hi = P + ((size_t)grp * nkb + kb) * 2 * GBLOCK_BYTES;
        unsigned char* blk_lo = blk_hi + GBLOCK_BYTES;
        // thread -> (row, chunk of 8 dimensions): 128 rows x 8 chunks = 1024 items, 4 per thread
#pragma unroll
        for (int it = 0; it < 4; ++it) {
            const int item = threadIdx.x + 256 * it;
            const int row = item >> 3, chunk = item & 7;
            const int64_t r = grp * GT + row;
            __half hi[8], lo[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                const int64_t k = (int64_t)kb * GK + chunk * 8 + e;
                float v = 0.f, x = 0.f;
                if (r < n && k < dim) {
                    x = (float)X[r * ldx + k];
                    v = (x - (float)(sums[k] * inv_n)) * GSCALE;
                }
                if (r < n) X32[r * ((int64_t)nkb * GK) + k] = x;
                hi[e] = __float2half_rn(v);
                lo[e] = __float2half_rn(v - __half2float(hi[e]));
                const double q = (double)__half2float(hi[e]) + (double)__half2float(lo[e]);
                nrm[it] += q * q;
            }
            const size_t off = ((size_t)chunk * 16 + (row >> 3)) * 128 + (row & 7) * 16;
            *reinterpret_cast<uint4*>(blk_hi + off) = *reinterpret_cast<const uint4*>(hi);
            if (!CROSS8) {
                *reinterpret_cast<uint4*>(blk_lo + off) = *reinterpret_cast<const uint4*>(lo);
            } else {
                unsigned char h8[8], l8[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    h8[e] = (unsigned char)__nv_cvt_float_to_fp8(__half2float(hi[e]) * alpha, __NV_SATFINITE, __NV_E4M3);
                    l8[e] = (unsigned char)__nv_cvt_float_to_fp8(__half2float(lo[e]) * beta, __NV_SATFINITE, __NV_E4M3);
                }
                // 16-element core-matrix rows: two of this thread's 8-dimension chunks per row
                const size_t off8 = ((size_t)(chunk >> 1) * 16 + (row >> 3)) * 128 + (row & 7) * 16 + (chunk & 1) * 8;
                *reinterpret_cast<uint2*>(blk_lo + off8) = *reinterpret_cast<const uint2*>(h8);                   // hi as e4m3
                *reinterpret_cast<uint2*>(blk_lo + GBLOCK_BYTES / 2 + off8) = *reinterpret_cast<const uint2*>(l8);  // lo as e4m3
            }
        }
    }
#pragma unroll
    for (int it = 0; it < 4; ++it) {
        // the 8 chunks of a row sit in 8 consecutive threads
        double v = nrm[it];
        v += __shfl_xor_sync(0xFFFFFFFFu, v, 1);
        v += __shfl_xor_sync(0xFFFFFFFFu, v, 2);
        v += __shfl_xor_sync(0xFFFFFFFFu, v, 4);
        const int item = threadIdx.x + 256 * it;
        const int64_t r = grp * GT + (item >> 3);
        if ((item & 7) == 0 && r < n) aux[r] = v;
    }
}

template <typename T>
static int launch_gram_prepare_t(const void* d_X, int64_t n, int64_t dim, int64_t ldx, void* d_P, double* d_aux,
                                 cudaStream_t stream) {
    const int64_t ldk = gram_ldk(dim);
    const int64_t npad = (n + GT - 1) / GT * GT;
    const int nkb = (int)(ldk / GK);
    unsigned char* P = reinterpret_cast<unsigned char*>(d_P);
    double* sums = reinterpret_cast<double*>(P + npad * ldk * 4);
    float* X32 = reinterpret_cast<float*>(P + npad * ldk * 4 + ldk * 8);
    double* partial = reinterpret_cast<double*>(P + npad * ldk * 4 + ldk * 8 + n * ldk * 4);
    dim3 g1((unsigned)((dim + 255) / 256), GSUM_SLICES, 1);
    gram_colsum_kernel<T><<<g1, 256, 0, stream>>>(reinterpret_cast<const T*>(d_X), n, dim, ldx, partial, ldk);
    count_launch(2);
    PO_LAUNCH_CHECK("gram_colsum_kernel");
    gram_colsum_final_kernel<<<(unsigned)((ldk + 255) / 256), 256, 0, stream>>>(partial, dim, ldk, sums);
    count_launch(2);
    PO_LAUNCH_CHECK("gram_colsum_final_kernel");
    float* scales = reinterpret_cast<float*>(P + npad * ldk * 4 + ldk * 8 + n * ldk * 4 + (int64_t)GSUM_SLICES * ldk * 8);
    if (eucl_cross8(dim)) {
        PO_CUDA_CHECK(cudaMemsetAsync(scales, 0, 64, stream));
        gram_absmax_kernel<T><<<1184, 256, 0, stream>>>(reinterpret_cast<const T*>(d_X), n, dim, ldx, sums,
                                                        reinterpret_cast<unsigned*>(scales));
        gram_scales_kernel<<<1, 1, 0, stream>>>(scales);
        gram_blocks_kernel<T, true><<<(unsigned)(npad / GT), 256, 0, stream>>>(reinterpret_cast<const T*>(d_X), n, dim, ldx, sums,
                                                                             P, nkb, d_aux, X32, scales);
    } else {
        gram_blocks_kernel<T, false><<<(unsigned)(npad / GT), 256, 0, stream>>>(reinterpret_cast<const T*>(d_X), n, dim, ldx, sums,
                                                                              P, nkb, d_aux, X32, scales);
    }
    count_launch(2);
    PO_LAUNCH_CHECK("gram_blocks_kernel");
    return PO_OK;
}

int launch_gram_prepare(const void* d_X, int dtype, int64_t n, int64_t dim, int64_t ldx, void* d_P, double* d_aux,
                        cudaStream_t stream) {
    if (!d_aux) {
        set_error("Eucl (tensor-core path) needs d_aux");
        return PO_ERR_ARG;
    }
    if (dtype == PO_F32) return launch_gram_prepare_t<float>(d_X, n, dim, ldx, d_P, d_aux, stream);
    return launch_gram_prepare_t<double>(d_X, n, dim, ldx, d_P, d_aux, stream);
}

// SC operands: one CTA per profile ranks it (O(dim^2) comparisons out of shared memory, as
// prepare_rank_kernel of po_prepare.cu) and scatters the two float16 digits of every centred doubled
// rank into the hi / lo operand blocks.  The block region is zeroed first (padding rows and dimensions).
template <typename T, bool DIGITS8>
__global__ void __launch_bounds__(256) sc_blocks_kernel(const T* __restrict__ X, int64_t n, int64_t dim, int64_t ldx,
                                                        unsigned char* __restrict__ P, int nkb, int dpad,
                                                        double* __restrict__ aux) {
    extern __shared__ __align__(8) unsigned char g_rank_smem[];
    __shared__ unsigned long long s_ss;
    const int64_t row = blockIdx.x;
    if (threadIdx.x == 0) s_ss = 0ull;
    const int64_t grp = row / GT;
    const int rr = (int)(row % GT);
    unsigned long long ss = rank_transform_row<T>(X + row * ldx, (int)dim, dpad, g_rank_smem, [&](int e, int val) {
        if (DIGITS8) {
            // a 64-dimension block is [h int8 8 KB | l int8 8 KB]; core matrices of 8 rows x 16 elements
            const int lo = ((val + 64) & 127) - 64;  // [-64, 63]
            const int hi = (val - lo) / 128;         // exact, |hi| <= 32
            const int kb = e / GK, kk = e % GK;
            unsigned char* blk = P + ((size_t)grp * nkb + kb) * GBLOCK_BYTES;
            const size_t off = ((size_t)(kk >> 4) * 16 + (rr >> 3)) * 128 + (rr & 7) * 16 + (kk & 15);
            blk[off] = (unsigned char)(signed char)hi;
            blk[GBLOCK_BYTES / 2 + off] = (unsigned char)(signed char)lo;
            return;
        }
        const int lo = ((val + 32) & 63) - 32;     // [-32, 31]
        const int hi = (val - lo) / 64;            // exact
        const int kb = e / GK, kk = e % GK;
        unsigned char* blk_hi = P + ((size_t)grp * nkb + kb) * 2 * GBLOCK_BYTES;
        const size_t off = ((size_t)(kk >> 3) * 16 + (rr >> 3)) * 128 + (rr & 7) * 16 + (kk & 7) * 2;
        *reinterpret_cast<__half*>(blk_hi + off) = __int2half_rn(hi);
        *reinterpret_cast<__half*>(blk_hi + GBLOCK_BYTES + off) = __int2half_rn(lo);
    });
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xFFFFFFFFu, ss, o);
    if ((threadIdx.x & 31) == 0 && ss) atomicAdd(&s_ss, ss);
    __syncthreads();
    if (threadIdx.x == 0) aux[row] = (double)s_ss;
}

int launch_sc_gram_prepare(const void* d_X, int dtype, int64_t n, int64_t dim, int64_t ldx, void* d_P, double* d_aux,
                           cudaStream_t stream) {
    if (!d_aux) {
        set_error("SC needs d_aux");
        return PO_ERR_ARG;
    }
    const int nkb = (int)(gram_ldk(dim) / GK);
    PO_CUDA_CHECK(cudaMemsetAsync(d_P, 0, (size_t)sc_gram_prepared_bytes(n, dim), stream));
    const size_t sm = rank_smem_bytes(dim);
    const int dpad = (int)rank_pad(dim);
#define PO_SC_PREP(TT, D8)                                                                                              \
    do {                                                                                                                \
        PO_CUDA_CHECK(cudaFuncSetAttribute(sc_blocks_kernel<TT, D8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm)); \
        sc_blocks_kernel<TT, D8><<<(unsigned)n, 256, sm, stream>>>(reinterpret_cast<const TT*>(d_X), n, dim, ldx,         \
                                                                   reinterpret_cast<unsigned char*>(d_P), nkb, dpad, d_aux); \
    } while (0)
    const bool d8 = sc_digits8();
    if (dtype == PO_F32) {
        if (d8) PO_SC_PREP(float, true);
        else PO_SC_PREP(float, false);
    } else {
        if (d8) PO_SC_PREP(double, true);
        else PO_SC_PREP(double, false);
    }
#undef PO_SC_PREP
    count_launch(2);
    PO_LAUNCH_CHECK("sc_blocks_kernel");
    return PO_OK;
}

// ---------------------------------------------------------------------------------------------
// tile kernel
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned g_smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void g_mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void g_mbar_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// bounded wait: a protocol error traps instead of hanging the device
__device__ __forceinline__ void g_mbar_wait(unsigned bar, unsigned parity) {
    unsigned done = 0;
    for (unsigned spin = 0; spin < (1u << 26); ++spin) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity)
            : "memory");
        if (done) return;
    }
    __trap();
}
__device__ __forceinline__ void g_bulk_g2s(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
// no-swizzle K-major operand descriptor: core matrices 128 B apart along M/N (SBO), 2 KB apart along K (LBO)
__device__ __forceinline__ uint64_t g_smem_desc(unsigned saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFFu);         // start address
    d |= (uint64_t)((2048u >> 4) & 0x3FFFu) << 16;   // leading byte offset (K direction)
    d |= (uint64_t)((128u >> 4) & 0x3FFFu) << 32;    // stride byte offset (M/N direction)
    d |= (uint64_t)1 << 46;                          // descriptor version (Blackwell)
    return d;                                        // layout type 0: no swizzle
}
__device__ __forceinline__ void g_mma_f16(unsigned tmem_d, uint64_t adesc, uint64_t bdesc, unsigned idesc, unsigned accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void g_mma_f8(unsigned tmem_d, uint64_t adesc, uint64_t bdesc, unsigned idesc, unsigned accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void g_mma_i8(unsigned tmem_d, uint64_t adesc, uint64_t bdesc, unsigned idesc, unsigned accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void g_mma_commit(unsigned bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void g_tmem_ld16(unsigned taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr));
}
__device__ __forceinline__ void g_tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

enum GramMode { GM_EUCL = 0, GM_SC = 1, GM_EUCL8 = 2, GM_SC8 = 3 };  // GM_EUCL8: e4m3 cross terms; GM_SC8: int8 digits
__host__ __device__ constexpr bool gm_is_sc(int mode) { return mode == GM_SC || mode == GM_SC8; }

struct GramParams {
    const unsigned char* P;  // operand blocks [n/128 groups][nkb][hi | lo][16 KB]
    const float* X32;        // float32 copy of the profiles, row pitch nkb * 64
    const double* aux;       // squared norms of the scaled, centred rows
    const float* scales;     // GM_EUCL8: [3] = 1 / (alpha beta), the scale of the e4m3 cross accumulator
    int nkb;
    int64_t n;
    int64_t row0, row1, col0, col1;
    int64_t tile_row0, tile_col0;
    int64_t tiles_r, tiles_c;  // tile grid; CTAs walk it in column chunks of GRASTER tiles (L2 reuse)
    void* out;
    int64_t ld_out, out_row0, out_col0;
    void* mir;
    int64_t ld_mir, mir_row0, mir_col0;
    unsigned flags;
};


// Tile geometry per mode.
// Eucl: a CTA of 8 warps computes one 128 x 128 tile with two accumulators -- hi.hi and hi.lo + lo.hi --
// in 256 TMEM columns, 32-wide K stages (32 KB) in a 3-deep ring: 97 KB of shared memory, so that TWO
// CTAs are resident per SM.  While one CTA drains its accumulators (tcgen05.ld, float64 epilogue,
// stores), the other one's MMAs keep the tensor pipe busy, and when both are in their main loops the
// pipe interleaves their MMAs, which also hides the bubble between two dependent MMAs into one
// accumulator (the cross terms).  (Round 1 ran one CTA of 16 warps per SM on 128 x 256 tiles: the
// tensor pipe idled through every epilogue, ncu: pipe 56 % active, 14 of 16 warps parked at a barrier.)
// SC: 128 x 128, four exact integer accumulators (hh, hl, lh, ll) = all 512 TMEM columns, 64-wide
// stages (64 KB) in a 3-deep ring, one CTA of 16 warps per SM.
template <int MODE> struct GramCfg;
#ifndef GRAM_EUCL_STAGES
#define GRAM_EUCL_STAGES 3
#endif
#ifndef GRAM_EUCL_KS
#define GRAM_EUCL_KS 32
#endif
template <> struct GramCfg<GM_EUCL> {
    static constexpr int NB = 1, KS = GRAM_EUCL_KS, STAGES = GRAM_EUCL_STAGES, GROUP_COLS = 256, TMEM_COLS = 256;
    static constexpr int THREADS = 256, CTAS = 2, ELEM_BYTES = 2;
};
template <> struct GramCfg<GM_EUCL8> : GramCfg<GM_EUCL> {};
template <> struct GramCfg<GM_SC8> {  // 128-wide stages of int8 digits: A [h 16 KB | l 16 KB], B the same: 64 KB
    static constexpr int NB = 1, KS = 128, STAGES = 3, GROUP_COLS = 384, TMEM_COLS = 512;
    static constexpr int THREADS = 512, CTAS = 1, ELEM_BYTES = 1;
};
template <> struct GramCfg<GM_SC> {
    static constexpr int NB = 1, KS = 64, STAGES = 3, GROUP_COLS = 384, TMEM_COLS = 512;
    static constexpr int THREADS = 512, CTAS = 1, ELEM_BYTES = 2;
};

// Epilogue of one 128 x 128 group of a tile, by all warps of the CTA.  Warp w owns TMEM lanes
// 32 (w & 3) .. +31 (the rows a warp may read) and the columns (128 / NCQ) (w >> 2) .. of the group,
// NCQ = warps / 4, which it walks in blocks of 32 (two tcgen05.ld chunks of 16).  Mirrored entries are
// stored straight from the registers (lanes = consecutive rows = consecutive addresses of the
// mirrored row); the direct entries go through a per-warp 32 x 33 shared-memory transpose so that a
// warp stores 128 contiguous bytes of one output row per instruction.  The operand ring is free by
// now.  INTERIOR groups carry no per-entry bounds tests.
//
// Eucl, diagonal group (row_base == col_base): with the cross terms hi.lo and lo.hi sharing one
// accumulator, (r, c) and (c, r) of the same group see their products in a different order.  The
// entries on and right of the diagonal are authoritative: the thread that holds (r, c), c > r, also
// stores it at (c, r) of the same group -- the mirror store of an off-diagonal group, aimed at the
// group itself -- and the computed values left of the diagonal are dropped, whatever the flags, so
// that a block row computed on its own equals the rows of the symmetric run bit for bit.  Groups
// wholly below the diagonal get the same effect from the MMA issue order (see the kernel).
// MO (PO_FLAG_MIRROR_ONLY): only the mirror stores; the kernel never calls a diagonal group's epilogue with it.
template <typename OUT_T, int MODE, bool INTERIOR, bool DIAG, bool MO>
__device__ __forceinline__ void gram_epilogue(const GramParams& p, unsigned tmem, int64_t row_base, int64_t col_base,
                                              const double* s_nb, unsigned char* gsmem) {
    constexpr int NCQ = GramCfg<MODE>::THREADS / 128;  // column slices of the group (warps per lane quarter)
    constexpr int WCOLS = GT / NCQ;                    // columns per warp
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int lq = warp & 3, cq = warp >> 2;
    const int r = lq * 32 + lane;  // tile row == TMEM lane
    const int64_t grow = row_base + r;
    const bool row_ok = INTERIOR || (grow >= p.row0 && grow < p.row1);
    const double na = (INTERIOR || grow < p.n) ? p.aux[grow] : 0.0;
    const bool do_mirror = DIAG || ((p.flags & PO_FLAG_MIRROR) && row_base + GT <= col_base);
    const int64_t ldx32 = (int64_t)p.nkb * GK;
    const float cross_scale = (MODE == GM_EUCL8) ? p.scales[3] : 1.f;
    const double cancel_limit = (MODE == GM_EUCL8) ? 8.0 : 256.0;
    OUT_T* tbuf = reinterpret_cast<OUT_T*>(gsmem) + (size_t)warp * (32 * 33) + (size_t)lane * 33;
    const OUT_T* wb = reinterpret_cast<const OUT_T*>(gsmem) + (size_t)warp * (32 * 33);
    // where the transposed entries go: the mirror buffer, or (diagonal group) the group itself.
    // mir_col0 = address of the mirrored entry (c, r) of this thread's row r and group column 0.
    OUT_T* const mbase = DIAG ? reinterpret_cast<OUT_T*>(p.out) : reinterpret_cast<OUT_T*>(p.mir);
    const int64_t m_ld = DIAG ? p.ld_out : p.ld_mir;
    OUT_T* mir_col0 = mbase + (col_base - (DIAG ? p.out_row0 : p.mir_row0)) * m_ld + (grow - (DIAG ? p.out_col0 : p.mir_col0));
    // a diagonal group's transposed entry (c, r) lies in ROW c, COLUMN r of the requested block
    const bool mcol_ok = !DIAG || (grow >= p.col0 && grow < p.col1);
#pragma unroll 1
    for (int blk = 0; blk < WCOLS / 32; ++blk) {
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
            const int c0 = cq * WCOLS + blk * 32 + half * 16;
            uint32_t vh[16], vx[16], vy[16], vz[16];
            const unsigned ta = tmem + ((unsigned)(lq * 32) << 16) + (unsigned)c0;
            g_tmem_ld16(ta, vh);
            g_tmem_ld16(ta + GT, vx);
            if (gm_is_sc(MODE)) g_tmem_ld16(ta + 2 * GT, vy);
            if (MODE == GM_SC) g_tmem_ld16(ta + 3 * GT, vz);
            g_tmem_wait_ld();
            OUT_T val[16];
            unsigned cancel = 0u;  // columns of this chunk whose Gram form cancelled too much
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const double nb = s_nb[c0 + j];
                if (gm_is_sc(MODE)) {
                    // exact integer dot product of the centred doubled ranks, then 1 - rho as K_SC does
                    const long long t = (MODE == GM_SC8)
                        ? 16384ll * (long long)(int)vh[j] + 128ll * (long long)(int)vx[j] + (long long)(int)vy[j]  // hh, hl + lh, ll (int32)
                        : 4096ll * (long long)__uint_as_float(vh[j]) +
                              64ll * ((long long)__uint_as_float(vx[j]) + (long long)__uint_as_float(vy[j])) +
                              (long long)__uint_as_float(vz[j]);
                    const double den = sqrt(na * nb);
                    const double v = (den == 0.0) ? __longlong_as_double(0x7FF8000000000000ll)  // scipy: NaN for a constant row
                                                  : 1.0 - (double)t / den;
                    val[j] = (OUT_T)v;
                    continue;
                }
                const float dot = fmaf(__uint_as_float(vx[j]), cross_scale, __uint_as_float(vh[j]));
                const double nsum = na + nb;
                double d2 = nsum - 2.0 * (double)dot;
                const bool on_diag = DIAG && r == c0 + j;
                // a diagonal group recomputes for its entries right of the diagonal: the others are copies
                const bool inside = DIAG ? (c0 + j > r && grow < p.n && col_base + c0 + j < p.n)
                                         : (INTERIOR || (row_ok && col_base + c0 + j >= p.col0 && col_base + c0 + j < p.col1));
                if (inside && d2 * cancel_limit < nsum) cancel |= 1u << j;
                d2 = (d2 > 0.0 ? d2 : 0.0) * GUNSCALE;
                if (sizeof(OUT_T) == 8) val[j] = (OUT_T)sqrt(d2);
                else val[j] = (OUT_T)sqrtf((float)d2);
                if (on_diag) val[j] = (OUT_T)0;  // sklearn forces an exact zero diagonal
            }
            // exact recomputation, one entry at a time, by the whole warp
            unsigned lanes = !gm_is_sc(MODE) ? __ballot_sync(0xFFFFFFFFu, cancel != 0u) : 0u;
            while (lanes) {
                const int l = __ffs(lanes) - 1;
                lanes &= lanes - 1;
                unsigned m = __shfl_sync(0xFFFFFFFFu, cancel, l);
                const int64_t er = row_base + lq * 32 + l;
                while (m) {
                    const int j = __ffs(m) - 1;
                    m &= m - 1;
                    const float* xa = p.X32 + er * ldx32;
                    const float* xb = p.X32 + (col_base + c0 + j) * ldx32;
                    double acc = 0.0;
                    for (int64_t k0 = 0; k0 < ldx32; k0 += 1024) {  // float32 partial sums of <= 32 terms per lane
                        float part = 0.f;
                        const int64_t k1 = min(ldx32, k0 + 1024);
                        for (int64_t k = k0 + lane; k < k1; k += 32) {
                            const float d = xa[k] - xb[k];
                            part = fmaf(d, d, part);
                        }
                        acc += (double)part;
                    }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, o);
                    if (lane == l) {
#pragma unroll
                        for (int jj = 0; jj < 16; ++jj)
                            if (jj == j) val[jj] = (sizeof(OUT_T) == 8) ? (OUT_T)sqrt(acc) : (OUT_T)sqrtf((float)acc);
                    }
                }
            }
            if (do_mirror) {
                OUT_T* mp = mir_col0 + (int64_t)c0 * m_ld;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    bool ok;
                    if (DIAG) ok = c0 + j > r && mcol_ok && col_base + c0 + j >= p.row0 && col_base + c0 + j < p.row1;
                    else ok = INTERIOR || (row_ok && col_base + c0 + j >= p.col0 && col_base + c0 + j < p.col1);
                    if (ok) *mp = val[j];
                    mp += m_ld;
                }
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) tbuf[half * 16 + j] = val[j];
        }
        __syncwarp();
        if (!MO) {
            const int c = cq * WCOLS + blk * 32 + lane;  // column of the group this lane stores
            const int64_t gcol = col_base + c;
            const bool col_ok = INTERIOR || (gcol >= p.col0 && gcol < p.col1);
            const int64_t gr0 = row_base + lq * 32;
            OUT_T* op = reinterpret_cast<OUT_T*>(p.out) + (gr0 - p.out_row0) * p.ld_out + (gcol - p.out_col0);
#pragma unroll 8
            for (int rr = 0; rr < 32; ++rr) {
                const OUT_T v = wb[rr * 33 + lane];
                bool ok = INTERIOR || (col_ok && gr0 + rr >= p.row0 && gr0 + rr < p.row1);
                if (DIAG) ok = ok && c >= lq * 32 + rr;  // on and right of the diagonal only
                if (ok) *op = v;
                op += p.ld_out;
            }
        }
        __syncwarp();  // the staging block is rewritten by the next 32 columns
    }
}

template <typename OUT_T, int MODE, bool MO>
__global__ void __launch_bounds__(GramCfg<MODE>::THREADS, GramCfg<MODE>::CTAS) gram_tile_kernel(const GramParams p) {
    using Cfg = GramCfg<MODE>;
    constexpr int NB = Cfg::NB, KS = Cfg::KS, NSTAGE = Cfg::STAGES;
    constexpr int SUB_BYTES = GT * KS * Cfg::ELEM_BYTES;  // one operand (hi or lo) of one 128-profile group per stage
    constexpr int STAGE_BYTES = (1 + NB) * 2 * SUB_BYTES;  // A hi, A lo, then B hi, B lo per group
    constexpr int TILE_N = NB * GT;
    extern __shared__ __align__(1024) unsigned char gsmem[];
    __shared__ __align__(8) unsigned long long bars[2 * NSTAGE + 1];
    __shared__ uint32_t s_tmem;
    __shared__ double s_nb[TILE_N];  // the tile columns' row constants (squared norms / rank sums)
    // rasterisation: chunks of GRASTER tile columns, all tile rows inside a chunk, so that the
    // chunk's column operands (GRASTER x 2 MB at 4096 dimensions) stay in L2 while the rows stream
    constexpr int RASTER = GRASTER / NB;  // the chunk stays GRASTER groups (2048 profiles) wide
    const int64_t per_chunk = p.tiles_r * RASTER;
    const int64_t chunk = (int64_t)blockIdx.x / per_chunk;
    const int64_t rem = (int64_t)blockIdx.x - chunk * per_chunk;
    const int64_t gw = min((int64_t)RASTER, p.tiles_c - chunk * RASTER);
    const int64_t row_base = p.tile_row0 + (rem / gw) * GT;
    const int64_t col_base = p.tile_col0 + (chunk * RASTER + rem % gw) * TILE_N;
    const int64_t npad = (p.n + GT - 1) / GT * GT;
    // which 128-column groups of the tile have anything to do
    bool act[NB];
    bool any = false;
#pragma unroll
    for (int g = 0; g < NB; ++g) {
        const int64_t cb = col_base + (int64_t)g * GT;
        act[g] = cb < npad && cb < p.col1 && cb + GT > p.col0 && !((p.flags & PO_FLAG_SKIP_LOWER) && cb + GT <= row_base);
        any = any || act[g];
    }
    if (!any) return;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const unsigned smem0 = g_smem_u32(gsmem);
    const unsigned full0 = g_smem_u32(&bars[0]), empty0 = g_smem_u32(&bars[NSTAGE]), accum = g_smem_u32(&bars[2 * NSTAGE]);

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < NSTAGE; ++s) {
            g_mbar_init(full0 + 8 * s, 1);
            g_mbar_init(empty0 + 8 * s, 1);
        }
        g_mbar_init(accum, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {  // one warp allocates the CTA's TMEM columns (Eucl: 256, two CTAs share the SM's 512; SC: 512)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(g_smem_u32(&s_tmem)), "r"((unsigned)Cfg::TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const unsigned tmem = s_tmem;

    const int nkb = p.nkb;
    const int nks = (nkb * GK + KS - 1) / KS;  // K stages of the tile
    // operand (grp, stage kq, hi/lo): the KS-wide slice of the 64-wide block, chunk-major inside the block
    auto g_operand = [&](int64_t grp, int kq, int hl) -> const unsigned char* {
        const int kb = (kq * KS) / GK;
        const int chunk0 = ((kq * KS) % GK) / 8;
        return p.P + (((size_t)grp * nkb + kb) * 2 + hl) * GBLOCK_BYTES + (size_t)chunk0 * 2048;
    };
    const int64_t grp_a = row_base / GT, grp_b0 = col_base / GT;

    if (warp == 0 && lane == 0) {
        // ===== producer: two bulk copies for the rows and two per active column group =====
        unsigned stage_bytes = 2 * SUB_BYTES;
#pragma unroll
        for (int g = 0; g < NB; ++g) stage_bytes += act[g] ? 2 * SUB_BYTES : 0;
        for (int kq = 0; kq < nks; ++kq) {
            const int s = kq % NSTAGE;
            g_mbar_wait(empty0 + 8 * s, (unsigned)(((kq / NSTAGE) & 1) ^ 1));
            const unsigned dst = smem0 + s * STAGE_BYTES;
            if (MODE == GM_SC8) {
                // a 128-dimension stage = two 64-dimension blocks [h int8 8 KB | l int8 8 KB]; per operand the two
                // h planes go next to each other (8 chunks of 16 dimensions, 2 KB apart), then the two l planes
                const int nblk = min(2, nkb - 2 * kq);
                g_mbar_expect_tx(full0 + 8 * s, (unsigned)(nblk * 2 * GBLOCK_BYTES));
                for (int o = 0; o < 2; ++o) {
                    const unsigned d0 = dst + o * 2 * SUB_BYTES;
                    for (int b = 0; b < nblk; ++b) {
                        const unsigned char* blk = p.P + ((size_t)(o ? grp_b0 : grp_a) * nkb + 2 * kq + b) * GBLOCK_BYTES;
                        g_bulk_g2s(d0 + b * (GBLOCK_BYTES / 2), blk, GBLOCK_BYTES / 2, full0 + 8 * s);
                        g_bulk_g2s(d0 + SUB_BYTES + b * (GBLOCK_BYTES / 2), blk + GBLOCK_BYTES / 2, GBLOCK_BYTES / 2, full0 + 8 * s);
                    }
                }
                continue;
            }
            g_mbar_expect_tx(full0 + 8 * s, stage_bytes);
            if (MODE == GM_EUCL8) {
                // per operand: the float16 hi plane of the stage (8 KB), then hi and lo as e4m3 (4 KB each);
                // in memory a 64-dimension block is [hi f16 16 KB | hi e4m3 8 KB | lo e4m3 8 KB]
                const int kb = (kq * KS) / GK, half = ((kq * KS) % GK) / KS;  // KS = 32: two stages per block
                for (int o = 0; o < 2; ++o) {
                    const unsigned char* blk = p.P + ((size_t)(o ? grp_b0 : grp_a) * nkb + kb) * 2 * GBLOCK_BYTES;
                    const unsigned d0 = dst + o * 2 * SUB_BYTES;
                    g_bulk_g2s(d0, blk + (size_t)half * SUB_BYTES, SUB_BYTES, full0 + 8 * s);
                    g_bulk_g2s(d0 + SUB_BYTES, blk + GBLOCK_BYTES + (size_t)half * (SUB_BYTES / 2), SUB_BYTES / 2, full0 + 8 * s);
                    g_bulk_g2s(d0 + SUB_BYTES + SUB_BYTES / 2, blk + GBLOCK_BYTES + GBLOCK_BYTES / 2 + (size_t)half * (SUB_BYTES / 2),
                               SUB_BYTES / 2, full0 + 8 * s);
                }
                continue;
            }
            g_bulk_g2s(dst, g_operand(grp_a, kq, 0), SUB_BYTES, full0 + 8 * s);
            g_bulk_g2s(dst + SUB_BYTES, g_operand(grp_a, kq, 1), SUB_BYTES, full0 + 8 * s);
#pragma unroll
            for (int g = 0; g < NB; ++g) {
                if (!act[g]) continue;
                g_bulk_g2s(dst + (2 + 2 * g) * SUB_BYTES, g_operand(grp_b0 + g, kq, 0), SUB_BYTES, full0 + 8 * s);
                g_bulk_g2s(dst + (3 + 2 * g) * SUB_BYTES, g_operand(grp_b0 + g, kq, 1), SUB_BYTES, full0 + 8 * s);
            }
        }
    } else if (warp == 1 && lane == 0) {
        // ===== MMA issuer =====
        // instruction descriptor: D float32, A/B float16 K-major, N = 128, M = 128
        const unsigned idesc = (1u << 4) | ((unsigned)(GT >> 3) << 17) | ((unsigned)(GT >> 4) << 24);
        for (int kq = 0; kq < nks; ++kq) {
            const int s = kq % NSTAGE;
            g_mbar_wait(full0 + 8 * s, (unsigned)((kq / NSTAGE) & 1));
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const unsigned a_hi = smem0 + s * STAGE_BYTES, a_lo = a_hi + SUB_BYTES;
            if (MODE == GM_SC8) {
                // int8 digits, int32 accumulators: hh, hl + lh (one accumulator: integer sums do not care about
                // the order) and ll; issue order hh, hl, ll, lh keeps the two cross MMAs apart
                const unsigned idesc8 = (2u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(GT >> 3) << 17) | ((unsigned)(GT >> 4) << 24);
                const unsigned b_hi = a_hi + 2 * SUB_BYTES, b_lo = b_hi + SUB_BYTES;
                const int steps = 2 * min(2, nkb - 2 * kq);  // K = 32 per MMA, 64 dimensions per block
                for (int ks = 0; ks < steps; ++ks) {
                    const unsigned koff = ks * 2 * 2048;  // two 16-element chunks per MMA
                    const unsigned acc = (kq > 0 || ks > 0) ? 1u : 0u;
                    const uint64_t dah = g_smem_desc(a_hi + koff), dal = g_smem_desc(a_lo + koff);
                    const uint64_t dbh = g_smem_desc(b_hi + koff), dbl = g_smem_desc(b_lo + koff);
                    g_mma_i8(tmem, dah, dbh, idesc8, acc);
                    g_mma_i8(tmem + GT, dah, dbl, idesc8, acc);
                    g_mma_i8(tmem + 2 * GT, dal, dbl, idesc8, acc);
                    g_mma_i8(tmem + GT, dal, dbh, idesc8, 1u);
                }
                g_mma_commit(empty0 + 8 * s);
                continue;
            }
            if (MODE == GM_EUCL8) {
                // stage: A [hi f16 8 KB | hi e4m3 4 KB | lo e4m3 4 KB], then B the same.  Two float16 MMAs (K = 16
                // each) for hi.hi and two e4m3 MMAs (K = 32 each) for the cross terms, interleaved so that no
                // accumulator receives two MMAs back to back; a tile below the diagonal issues the cross terms
                // in the order its mirror image does (bitwise symmetry).
                const unsigned b_hi = a_hi + 2 * SUB_BYTES;
                const unsigned a_h8 = a_hi + SUB_BYTES, a_l8 = a_h8 + SUB_BYTES / 2;
                const unsigned b_h8 = b_hi + SUB_BYTES, b_l8 = b_h8 + SUB_BYTES / 2;
                const bool upper = col_base >= row_base;
                const unsigned acc = kq > 0 ? 1u : 0u;
                g_mma_f8(tmem + GT, g_smem_desc(upper ? a_h8 : a_l8), g_smem_desc(upper ? b_l8 : b_h8), idesc, acc);
                g_mma_f16(tmem, g_smem_desc(a_hi), g_smem_desc(b_hi), idesc, acc);
                g_mma_f8(tmem + GT, g_smem_desc(upper ? a_l8 : a_h8), g_smem_desc(upper ? b_h8 : b_l8), idesc, 1u);
                g_mma_f16(tmem, g_smem_desc(a_hi + 2 * 2048), g_smem_desc(b_hi + 2 * 2048), idesc, 1u);
                g_mma_commit(empty0 + 8 * s);
                continue;
            }
#pragma unroll
            for (int ks = 0; ks < KS / 16; ++ks) {
                const unsigned koff = ks * 2 * 2048;  // two 8-element chunks per MMA
                const uint64_t dah = g_smem_desc(a_hi + koff), dal = g_smem_desc(a_lo + koff);
                const unsigned acc = (kq > 0 || ks > 0) ? 1u : 0u;
                // Two MMAs into the same accumulator back to back serialise in the tensor pipe, so the
                // issue order keeps them apart: SC has four accumulators (hh, hl, lh, ll: distance 4);
                // Eucl issues cross(a) of both groups, hh of group 0, cross(b) of both groups, hh of
                // group 1 (distance 3 for the cross accumulators, 6 for hh).
                if (MODE == GM_SC) {
                    const unsigned b_hi = a_hi + 2 * SUB_BYTES, b_lo = b_hi + SUB_BYTES;
                    const uint64_t dbh = g_smem_desc(b_hi + koff), dbl = g_smem_desc(b_lo + koff);
                    g_mma_f16(tmem, dah, dbh, idesc, acc);
                    g_mma_f16(tmem + GT, dah, dbl, idesc, acc);
                    g_mma_f16(tmem + 2 * GT, dal, dbh, idesc, acc);
                    g_mma_f16(tmem + 3 * GT, dal, dbl, idesc, acc);
                } else {
                    uint64_t dbh[NB], dbl[NB];
                    bool upper[NB];
#pragma unroll
                    for (int g = 0; g < NB; ++g) {
                        const unsigned b_hi = a_hi + (2 + 2 * g) * SUB_BYTES;
                        dbh[g] = g_smem_desc(b_hi + koff);
                        dbl[g] = g_smem_desc(b_hi + SUB_BYTES + koff);
                        // hi.lo + lo.hi share an accumulator.  A group below the diagonal issues them in the
                        // order its mirror image above the diagonal does, so that (r, c) and (c, r) are the
                        // same float32 sum whichever group computes them.
                        upper[g] = col_base + (int64_t)g * GT >= row_base;
                    }
#pragma unroll
                    for (int g = 0; g < NB; ++g)
                        if (act[g]) g_mma_f16(tmem + g * Cfg::GROUP_COLS + GT, upper[g] ? dah : dal, upper[g] ? dbl[g] : dbh[g], idesc, acc);
                    if (act[0]) g_mma_f16(tmem, dah, dbh[0], idesc, acc);
#pragma unroll
                    for (int g = 0; g < NB; ++g)
                        if (act[g]) g_mma_f16(tmem + g * Cfg::GROUP_COLS + GT, upper[g] ? dal : dah, upper[g] ? dbh[g] : dbl[g], idesc, 1u);
                    if (NB > 1 && act[NB - 1]) g_mma_f16(tmem + (NB - 1) * Cfg::GROUP_COLS, dah, dbh[NB - 1], idesc, acc);
                }
            }
            g_mma_commit(empty0 + 8 * s);  // the stage is free once these MMAs have read it
        }
        g_mma_commit(accum);  // accumulators complete
    }
    __syncwarp();

    // ===== epilogue (gram_epilogue): all 16 warps, one 128-column group after the other =====
    if (tid < TILE_N) {
        const int64_t gc = col_base + tid;
        s_nb[tid] = (gc < p.n) ? p.aux[gc] : 0.0;
    }
    // the warps that do not drive the pipeline sleep on the accumulators' mbarrier (not on a CTA barrier)
    g_mbar_wait(accum, 0u);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    __syncthreads();  // s_nb is visible
#pragma unroll
    for (int g = 0; g < NB; ++g) {
        if (!act[g]) continue;
        const int64_t cb = col_base + (int64_t)g * GT;
        const unsigned tg = tmem + (unsigned)(g * Cfg::GROUP_COLS);
        // groups wholly inside the requested block (all but the ragged edges) skip the per-entry bounds tests
        const bool interior = row_base >= p.row0 && row_base + GT <= p.row1 && cb >= p.col0 && cb + GT <= p.col1;
        if (!gm_is_sc(MODE) && cb == row_base) {
            if (!MO) gram_epilogue<OUT_T, MODE, false, true, false>(p, tg, row_base, cb, s_nb + g * GT, gsmem);
        } else if (interior) {
            gram_epilogue<OUT_T, MODE, true, false, MO>(p, tg, row_base, cb, s_nb + g * GT, gsmem);
        } else {
            gram_epilogue<OUT_T, MODE, false, false, MO>(p, tg, row_base, cb, s_nb + g * GT, gsmem);
        }
        if (NB > 1) __syncthreads();  // the staging buffers are reused by the next group
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((unsigned)Cfg::TMEM_COLS));
}

template <typename OUT_T, int MODE, bool MO>
static int launch_gram_mo(GramParams p, int64_t row1, int64_t col1, cudaStream_t stream) {
    using Cfg = GramCfg<MODE>;
    const int64_t tile_n = (int64_t)Cfg::NB * GT;
    p.tile_col0 = p.col0 / tile_n * tile_n;
    const int64_t tr = (row1 - p.tile_row0 + GT - 1) / GT, tc = (col1 - p.tile_col0 + tile_n - 1) / tile_n;
    if (tr * tc > 0x7FFFFFFFll) {
        set_error("block too large: %lld x %lld tiles", (long long)tr, (long long)tc);
        return PO_ERR_UNSUPPORTED;
    }
    p.tiles_r = tr;
    p.tiles_c = tc;
    const size_t smem = (size_t)Cfg::STAGES * (1 + Cfg::NB) * 2 * GT * Cfg::KS * Cfg::ELEM_BYTES + 1024;
    PO_CUDA_CHECK(cudaFuncSetAttribute(gram_tile_kernel<OUT_T, MODE, MO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    gram_tile_kernel<OUT_T, MODE, MO><<<dim3((unsigned)(tr * tc), 1, 1), Cfg::THREADS, smem, stream>>>(p);
    return PO_OK;
}

template <typename OUT_T, int MODE>
static int launch_gram_t(GramParams p, int64_t row1, int64_t col1, cudaStream_t stream) {
    return (p.flags & PO_FLAG_MIRROR_ONLY) ? launch_gram_mo<OUT_T, MODE, true>(p, row1, col1, stream)
                                           : launch_gram_mo<OUT_T, MODE, false>(p, row1, col1, stream);
}

int launch_gram(int metric, const void* d_P, const double* d_aux, int64_t n, int64_t dim, int64_t row0, int64_t row1,
                int64_t col0, int64_t col1, void* d_out, int64_t ld_out, int64_t out_row0, int64_t out_col0, void* d_mir,
                int64_t ld_mir, int64_t mir_row0, int64_t mir_col0, int out_dtype, unsigned flags, cudaStream_t stream) {
    if (!d_aux) {
        set_error("the tensor-core path needs d_aux from po_prepare_profiles");
        return PO_ERR_ARG;
    }
    GramParams p;
    p.P = reinterpret_cast<const unsigned char*>(d_P);
    p.aux = d_aux;
    p.nkb = (int)(gram_ldk(dim) / GK);
    {
        const int64_t ldk = gram_ldk(dim), npad = (n + GT - 1) / GT * GT;
        p.X32 = reinterpret_cast<const float*>(p.P + npad * ldk * 4 + ldk * 8);
        p.scales = reinterpret_cast<const float*>(p.P + npad * ldk * 4 + ldk * 8 + n * ldk * 4 + (int64_t)GSUM_SLICES * ldk * 8);
    }
    p.n = n;
    p.row0 = row0; p.row1 = row1; p.col0 = col0; p.col1 = col1;
    p.tile_row0 = row0 / GT * GT;
    p.out = d_out; p.ld_out = ld_out; p.out_row0 = out_row0; p.out_col0 = out_col0;
    p.mir = d_mir; p.ld_mir = ld_mir; p.mir_row0 = mir_row0; p.mir_col0 = mir_col0;
    p.flags = flags;
    LaunchTimer tm(1, stream);
    int rc;
    if (metric == PO_SC && sc_digits8())
        rc = out_dtype == PO_F32 ? launch_gram_t<float, GM_SC8>(p, row1, col1, stream)
                                 : launch_gram_t<double, GM_SC8>(p, row1, col1, stream);
    else if (metric == PO_SC)
        rc = out_dtype == PO_F32 ? launch_gram_t<float, GM_SC>(p, row1, col1, stream)
                                 : launch_gram_t<double, GM_SC>(p, row1, col1, stream);
    else if (eucl_cross8(dim))
        rc = out_dtype == PO_F32 ? launch_gram_t<float, GM_EUCL8>(p, row1, col1, stream)
                                 : launch_gram_t<double, GM_EUCL8>(p, row1, col1, stream);
    else
        rc = out_dtype == PO_F32 ? launch_gram_t<float, GM_EUCL>(p, row1, col1, stream)
                                 : launch_gram_t<double, GM_EUCL>(p, row1, col1, stream);
    if (rc != PO_OK) return rc;
    count_launch(1);
    PO_LAUNCH_CHECK("gram_tile_kernel");
    return PO_OK;
}

}  // namespace po
