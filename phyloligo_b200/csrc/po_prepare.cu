// Per-row operand preparation for the distance tiles (sm_100a).
//
//   Eucl       : float32 copy of the profile, zero padded to a multiple of 4.
//   JSD        : float32 copy plus 1e-30: exact zeros (and the padding) become 1e-30
//                while every representable frequency (>= 1e-22) is unchanged, so the
//                tile kernel's a+b is never 0 and needs no clamp; the 1e-30 entries
//                change a term by < 1e-27 relative.  Stored "blocked" for the bulk
//                copies of po_jsd.cu: [n/64][dim/32] blocks of [32 dims][64 profiles]
//                (column operand) followed by [n/32][dim/32] blocks of
//                [32 dims][32 profiles] (row operand).
//   BC         : the same copy; aux = sum of the row (the sum|a+b| denominator of
//                scipy's braycurtis splits into row sums for non-negative profiles;
//                a negative entry poisons aux with NaN so the result is loudly NaN).
//   SC         : rank transform with average ranks for ties -- the
//                scipy.stats.spearmanr step of phylodist.SC (core/phylodist.py:82-85).
//                Stored as the integer 2*rank - (dim+1) = 2*less + equal - dim, which
//                is exact, already centred (ranks always average (dim+1)/2) and makes
//                the pairwise dot product an exact integer.  aux = sum of squares.
//   KT         : the per-row half of Bio.Cluster's kendall() loop
//                (core/phylodist.py:71-74).  Element pairs are enumerated as
//                (i, (i+d) mod dim), d = 1 .. dim/2, bit e = (d-1)*dim + i; one mask
//                holds "value_i > value_j", one "value_i < value_j".  Words are
//                interleaved in groups of 4 up-words then 4 down-words so the tile
//                kernel reads them with 128-bit loads.  aux = number of untied pairs.
#include "po_common.cuh"
#include "po_rank.cuh"

namespace po {

constexpr int JSD_MINMAX_SLICES = 64;  // row slices of the two-stage column min / max (fixed order: reproducible)

int64_t prepared_row_elems(int metric, int64_t dim) {
    if (metric == PO_KT) {
        const int64_t nbits = dim * (dim - 1) / 2;
        const int64_t groups = (nbits + 127) / 128;  // 4 words of 32 bits per group
        return (groups > 0 ? groups : 1) * 8;
    }
    // JSD rows are padded (with the 1e-30 bias) to a whole 32-element pipeline chunk so
    // the tile kernel never meets a zero-filled (a = b = 0) lane
    if (metric == PO_JSD) return (dim + 31) / 32 * 32;
    return (dim + 3) / 4 * 4;
}

// total bytes of the prepared operand buffer of n rows
int64_t prepared_bytes(int metric, int64_t n, int64_t dim) {
    const int64_t ldp = prepared_row_elems(metric, dim);
    if (metric == PO_JSD) {
        // blocked B + blocked A (rows padded to 64), the per-group value ranges, the dimension permutation
        // and the scratch of its computation (per-slice column minima / maxima, spreads)
        const int64_t npad = (n + 63) / 64 * 64;
        return 2 * npad * ldp * 4 + 2 * (npad / 64) * ldp * 4 + ldp * 4 + (2 * JSD_MINMAX_SLICES + 1) * ldp * 4;
    }
    if (eucl_use_gram(metric, dim)) return gram_prepared_bytes(n, dim);
    if (sc_use_gram(metric, dim)) return sc_gram_prepared_bytes(n, dim);
    return n * ldp * 4;
}

template <typename T>
__device__ __forceinline__ double load_as_double(const void* X, int64_t idx) {
    return (double)reinterpret_cast<const T*>(X)[idx];
}

template <typename T>
__global__ void __launch_bounds__(256) prepare_copy_kernel(const void* __restrict__ X, int64_t n, int64_t dim,
                                                           int64_t ldx, float* __restrict__ P, int64_t ldp,
                                                           double* __restrict__ aux, int want_sum, float bias) {
    const int64_t row = blockIdx.x;
    double s = 0.0;
    bool neg = false;
    for (int64_t e = threadIdx.x; e < ldp; e += blockDim.x) {
        float v = 0.f;
        if (e < dim) {
            const double x = load_as_double<T>(X, row * ldx + e);
            v = (float)x;
            s += (double)v;
            neg |= (v < 0.f);
        }
        P[row * ldp + e] = v + bias;
    }
    if (want_sum) {
        __shared__ double red[8];
        __shared__ int sneg;
        if (threadIdx.x == 0) sneg = 0;
        __syncthreads();
        if (neg) atomicOr(&sneg, 1);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
            aux[row] = sneg ? __longlong_as_double(0x7FF8000000000000ll) : t;
        }
    }
}


// JSD, step 1: smallest and largest (biased float32) value of every dimension over all profiles, in two
// stages with a fixed order; step 2: spread = max / min per dimension; step 3: the permutation that
// sorts the dimensions by ascending spread (ties by index; padding dimensions last).  po_jsd.cu runs a
// cheaper loop on chunks of dimensions whose values are provably close together, and narrow dimensions
// only share chunks when they are sorted; a sum over dimensions does not care about their order.
template <typename T>
__global__ void __launch_bounds__(256) jsd_colminmax_kernel(const void* __restrict__ X, int64_t n, int64_t dim, int64_t ldx,
                                                            float* __restrict__ pmin, float* __restrict__ pmax, int64_t ldp) {
    const int64_t col = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (col >= dim) return;
    const int64_t rows_per = (n + JSD_MINMAX_SLICES - 1) / JSD_MINMAX_SLICES;
    const int64_t r0 = (int64_t)blockIdx.y * rows_per, r1 = min(n, r0 + rows_per);
    float lo = __int_as_float(0x7F800000), hi = 0.f;
    for (int64_t r = r0; r < r1; ++r) {
        const float v = (float)load_as_double<T>(X, r * ldx + col) + 1e-30f;
        lo = fminf(lo, v);
        hi = fmaxf(hi, v);
    }
    pmin[(int64_t)blockIdx.y * ldp + col] = lo;
    pmax[(int64_t)blockIdx.y * ldp + col] = hi;
}

__global__ void __launch_bounds__(256) jsd_spread_kernel(const float* __restrict__ pmin, const float* __restrict__ pmax,
                                                         int64_t dim, int64_t ldp, float* __restrict__ spread) {
    const int64_t col = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (col >= ldp) return;
    float sp = __int_as_float(0x7F800000);  // padding dimensions sort last
    if (col < dim) {
        float lo = __int_as_float(0x7F800000), hi = 0.f;
        for (int y = 0; y < JSD_MINMAX_SLICES; ++y) {
            lo = fminf(lo, pmin[(int64_t)y * ldp + col]);
            hi = fmaxf(hi, pmax[(int64_t)y * ldp + col]);
        }
        sp = hi / lo;
        if (!(sp == sp)) sp = __int_as_float(0x7F800000);  // NaN profiles: keep the order total
    }
    spread[col] = sp;
}

__global__ void __launch_bounds__(256) jsd_rank_kernel(const float* __restrict__ spread, int64_t ldp, int* __restrict__ perm) {
    const int64_t d = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (d >= ldp) return;
    const float mine = spread[d];
    int64_t before = 0;
    for (int64_t e = 0; e < ldp; ++e) {
        const float v = spread[e];
        before += (v < mine) || (v == mine && e < d);
    }
    perm[before] = (int)d;
}

// JSD: biased float32 profiles in the blocked layout of po_jsd.cu, dimensions permuted.  One CTA per
// (group of 64 profiles, chunk of 32 dimensions); the transpose goes through shared memory.  Also the
// smallest and largest value of the group per dimension (profiles beyond n do not count: their tiles'
// results are never stored).
template <typename T>
__global__ void __launch_bounds__(256) prepare_jsd_kernel(const void* __restrict__ X, int64_t n, int64_t dim,
                                                          int64_t ldx, float* __restrict__ PB, float* __restrict__ PA,
                                                          int nchunks, const int* __restrict__ perm,
                                                          float* __restrict__ gmin, float* __restrict__ gmax) {
    __shared__ float tile[64][33];
    const int64_t grp = blockIdx.x;
    const int kc = blockIdx.y;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t e = perm[(int64_t)kc * 32 + lane];  // source dimension of this lane's column
    for (int r = w; r < 64; r += 8) {
        const int64_t row = grp * 64 + r;
        float v = 0.f;
        if (row < n && e < dim) v = (float)load_as_double<T>(X, row * ldx + e);
        tile[r][lane] = v + 1e-30f;
    }
    __syncthreads();
    float* blkB = PB + ((size_t)grp * nchunks + kc) * 2048;
    for (int q = threadIdx.x; q < 2048; q += 256) blkB[q] = tile[q & 63][q >> 6];  // [d][c]
    // two row-operand blocks (profiles 0..31 and 32..63 of the group): [d][r]
    for (int h = 0; h < 2; ++h) {
        float* blkA = PA + ((size_t)(grp * 2 + h) * nchunks + kc) * 1024;
        for (int q = threadIdx.x; q < 1024; q += 256) blkA[q] = tile[h * 32 + (q & 31)][q >> 5];
    }
    if (w == 0) {
        float lo = __int_as_float(0x7F800000), hi = 0.f;
        const int64_t rows = min((int64_t)64, n - grp * 64);
        for (int r = 0; r < rows; ++r) {
            lo = fminf(lo, tile[r][lane]);
            hi = fmaxf(hi, tile[r][lane]);
        }
        gmin[((size_t)grp * nchunks + kc) * 32 + lane] = lo;
        gmax[((size_t)grp * nchunks + kc) * 32 + lane] = hi;
    }
}

// SC: centred doubled average ranks (po_rank.cuh: shared-memory sort + tie groups).
template <typename T>
__global__ void __launch_bounds__(256) prepare_rank_kernel(const void* __restrict__ X, int64_t n, int64_t dim,
                                                           int64_t ldx, int* __restrict__ P, int64_t ldp, int dpad,
                                                           double* __restrict__ aux) {
    extern __shared__ __align__(8) unsigned char rank_smem[];
    __shared__ unsigned long long s_ss;
    const int64_t row = blockIdx.x;
    if (threadIdx.x == 0) s_ss = 0ull;
    for (int64_t e = dim + threadIdx.x; e < ldp; e += blockDim.x) P[row * ldp + e] = 0;  // padding
    unsigned long long ss = rank_transform_row<T>(reinterpret_cast<const T*>(X) + row * ldx, (int)dim, dpad, rank_smem,
                                                  [&](int e, int val) { P[row * ldp + e] = val; });
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xFFFFFFFFu, ss, o);
    if ((threadIdx.x & 31) == 0 && ss) atomicAdd(&s_ss, ss);
    __syncthreads();
    if (threadIdx.x == 0) aux[row] = (double)s_ss;
}

// Average ranks 1..dim as float64 (scipy.stats.rankdata(method="average")): the stand-alone form of
// the SC prologue, po_rank_transform.
template <typename T>
__global__ void __launch_bounds__(256) rank_average_kernel(const void* __restrict__ X, int64_t dim, int64_t ldx,
                                                           double* __restrict__ R, int64_t ldr, int dpad) {
    extern __shared__ __align__(8) unsigned char rank_smem[];
    const int64_t row = blockIdx.x;
    rank_transform_row<T>(reinterpret_cast<const T*>(X) + row * ldx, (int)dim, dpad, rank_smem,
                          [&](int e, int val) { R[row * ldr + e] = 0.5 * (double)(val + (int)dim + 1); });
}

int launch_rank_transform(const void* d_X, int dtype, int64_t n, int64_t dim, int64_t ldx, double* d_R, int64_t ldr,
                          cudaStream_t stream) {
    if (n == 0) return PO_OK;
    const size_t sm = rank_smem_bytes(dim);
    if (sm > 200 * 1024 || n > 0x7FFFFFFFll) {
        set_error("po_rank_transform: %lld rows of dimension %lld are outside the supported envelope", (long long)n,
                  (long long)dim);
        return PO_ERR_UNSUPPORTED;
    }
    const int dpad = (int)rank_pad(dim);
    if (dtype == PO_F32) {
        PO_CUDA_CHECK(cudaFuncSetAttribute(rank_average_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        rank_average_kernel<float><<<(unsigned)n, 256, sm, stream>>>(d_X, dim, ldx, d_R, ldr, dpad);
    } else {
        PO_CUDA_CHECK(cudaFuncSetAttribute(rank_average_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        rank_average_kernel<double><<<(unsigned)n, 256, sm, stream>>>(d_X, dim, ldx, d_R, ldr, dpad);
    }
    count_launch(2);
    PO_LAUNCH_CHECK("rank_average_kernel");
    return PO_OK;
}

// KT: packed order-relation masks.
template <typename T>
__global__ void __launch_bounds__(256) prepare_kendall_kernel(const void* __restrict__ X, int64_t n, int64_t dim,
                                                              int64_t ldx, uint32_t* __restrict__ P, int64_t ldp,
                                                              double* __restrict__ aux) {
    extern __shared__ double srow[];
    __shared__ unsigned long long s_untied;
    const int64_t row = blockIdx.x;
    for (int64_t e = threadIdx.x; e < dim; e += blockDim.x) srow[e] = load_as_double<T>(X, row * ldx + e);
    if (threadIdx.x == 0) s_untied = 0ull;
    __syncthreads();
    const int64_t nbits = dim * (dim - 1) / 2;
    const int64_t nwords = ldp / 2;  // up-words (the same number of down-words)
    unsigned long long untied = 0ull;
    for (int64_t w = threadIdx.x; w < nwords; w += blockDim.x) {
        uint32_t up = 0u, dn = 0u;
        const int64_t e0 = w * 32;
        if (e0 < nbits) {
            int64_t d = e0 / dim + 1;
            int64_t i = e0 % dim;
#pragma unroll 4
            for (int b = 0; b < 32; ++b) {
                if (e0 + b < nbits) {
                    int64_t j = i + d;
                    if (j >= dim) j -= dim;
                    const double vi = srow[i], vj = srow[j];
                    up |= (uint32_t)(vi > vj) << b;
                    dn |= (uint32_t)(vi < vj) << b;
                }
                if (++i == dim) { i = 0; ++d; }
            }
        }
        untied += (unsigned)(__popc(up) + __popc(dn));
        const int64_t g = w >> 2, q = w & 3;
        P[row * ldp + g * 8 + q] = up;
        P[row * ldp + g * 8 + 4 + q] = dn;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) untied += __shfl_xor_sync(0xFFFFFFFFu, untied, o);
    if ((threadIdx.x & 31) == 0 && untied) atomicAdd(&s_untied, untied);
    __syncthreads();
    if (threadIdx.x == 0) aux[row] = (double)s_untied;
}

template <typename T>
static int launch_prepare_t(int metric, const void* d_X, int64_t n, int64_t dim, int64_t ldx, void* d_P,
                            double* d_aux, cudaStream_t stream) {
    const int64_t ldp = prepared_row_elems(metric, dim);
    const unsigned grid = (unsigned)n;
    switch (metric) {
        case PO_JSD: {
            const int nchunks = (int)(ldp / 32);
            const int64_t npad = (n + 63) / 64 * 64;
            float* PB = (float*)d_P;
            float* PA = PB + npad * ldp;
            float* gmin = PA + npad * ldp;
            float* gmax = gmin + (npad / 64) * ldp;
            int* perm = reinterpret_cast<int*>(gmax + (npad / 64) * ldp);
            float* pmin = reinterpret_cast<float*>(perm + ldp);
            float* pmax = pmin + (int64_t)JSD_MINMAX_SLICES * ldp;
            float* spread = pmax + (int64_t)JSD_MINMAX_SLICES * ldp;
            dim3 g1((unsigned)((dim + 255) / 256), JSD_MINMAX_SLICES, 1);
            jsd_colminmax_kernel<T><<<g1, 256, 0, stream>>>(d_X, n, dim, ldx, pmin, pmax, ldp);
            count_launch(2);
            PO_LAUNCH_CHECK("jsd_colminmax_kernel");
            jsd_spread_kernel<<<(unsigned)((ldp + 255) / 256), 256, 0, stream>>>(pmin, pmax, dim, ldp, spread);
            count_launch(2);
            PO_LAUNCH_CHECK("jsd_spread_kernel");
            jsd_rank_kernel<<<(unsigned)((ldp + 255) / 256), 256, 0, stream>>>(spread, ldp, perm);
            count_launch(2);
            PO_LAUNCH_CHECK("jsd_rank_kernel");
            dim3 g((unsigned)(npad / 64), (unsigned)nchunks, 1);
            prepare_jsd_kernel<T><<<g, 256, 0, stream>>>(d_X, n, dim, ldx, PB, PA, nchunks, perm, gmin, gmax);
            count_launch(2);
            PO_LAUNCH_CHECK("prepare_jsd_kernel");
            return PO_OK;
        }
        case PO_EUCL:
        case PO_EUCL_GRAM:
        case PO_BC: {
            const int want_sum = (metric == PO_BC);
            if (want_sum && !d_aux) {
                set_error("BC needs d_aux");
                return PO_ERR_ARG;
            }
            prepare_copy_kernel<T><<<grid, 256, 0, stream>>>(d_X, n, dim, ldx, (float*)d_P, ldp, d_aux, want_sum, 0.0f);
            count_launch(2);
            PO_LAUNCH_CHECK("prepare_copy_kernel");
            return PO_OK;
        }
        case PO_SC: {
            if (!d_aux) {
                set_error("SC needs d_aux");
                return PO_ERR_ARG;
            }
            const size_t sm = rank_smem_bytes(dim);
            auto kern = prepare_rank_kernel<T>;
            if (sm > 200 * 1024) {
                set_error("SC: profile dimension %lld too large for the rank kernel", (long long)dim);
                return PO_ERR_UNSUPPORTED;
            }
            if (sm > 32 * 1024)  // static + dynamic shared memory beyond the 48 KB default needs the opt-in
                PO_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
            kern<<<grid, 256, sm, stream>>>(d_X, n, dim, ldx, (int*)d_P, ldp, (int)rank_pad(dim), d_aux);
            count_launch(2);
            PO_LAUNCH_CHECK("prepare_rank_kernel");
            return PO_OK;
        }
        case PO_KT: {
            if (!d_aux) {
                set_error("KT needs d_aux");
                return PO_ERR_ARG;
            }
            const size_t sm = (size_t)dim * sizeof(double);
            auto kern = prepare_kendall_kernel<T>;
            if (sm > 200 * 1024) {
                set_error("KT: profile dimension %lld too large for the mask kernel", (long long)dim);
                return PO_ERR_UNSUPPORTED;
            }
            if (sm > 48 * 1024)
                PO_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
            kern<<<grid, 256, sm, stream>>>(d_X, n, dim, ldx, (uint32_t*)d_P, ldp, d_aux);
            count_launch(2);
            PO_LAUNCH_CHECK("prepare_kendall_kernel");
            return PO_OK;
        }
    }
    set_error("unknown metric %d", metric);
    return PO_ERR_ARG;
}

int launch_prepare(int metric, const void* d_X, int dtype, int64_t n, int64_t dim, int64_t ldx,
                   void* d_P, double* d_aux, cudaStream_t stream) {
    if (n == 0) return PO_OK;
    if (eucl_use_gram(metric, dim) && (dtype == PO_F32 || dtype == PO_F64))
        return launch_gram_prepare(d_X, dtype, n, dim, ldx, d_P, d_aux, stream);
    if (sc_use_gram(metric, dim) && (dtype == PO_F32 || dtype == PO_F64)) {
        if (n > 0x7FFFFFFFll) {
            set_error("too many rows (%lld)", (long long)n);
            return PO_ERR_UNSUPPORTED;
        }
        return launch_sc_gram_prepare(d_X, dtype, n, dim, ldx, d_P, d_aux, stream);
    }
    if (n > 0x7FFFFFFFll) {
        set_error("too many rows (%lld)", (long long)n);
        return PO_ERR_UNSUPPORTED;
    }
    if (dtype == PO_F32) return launch_prepare_t<float>(metric, d_X, n, dim, ldx, d_P, d_aux, stream);
    if (dtype == PO_F64) return launch_prepare_t<double>(metric, d_X, n, dim, ldx, d_P, d_aux, stream);
    set_error("unknown dtype %d", dtype);
    return PO_ERR_ARG;
}

}  // namespace po
