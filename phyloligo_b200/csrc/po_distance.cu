// All-by-all distance tiles on sm_100a CUDA cores: Eucl, BC, SC, KT (JSD lives in po_jsd.cu).
//
// Replaces phylodist.Eucl/KT/BC/SC (reference core/phylodist.py:36-41, 71-85) and the
// block-row slice workers *_loc / *_h5py (bin/phyloligo.py:195-301).
//
// One CTA (256 threads) computes a 64 x 64 tile of the matrix.  Thread (ty, tx) owns the
// 4 x 4 pairs (rows ty + 16 i, cols tx + 16 j).  Operand rows are "prepared rows" of 32-bit
// elements (po_prepare_profiles): float32 profiles (Eucl, BC), int32 centred doubled ranks
// (SC) or packed order-relation bit masks (KT).  The K dimension is streamed in chunks of 32
// elements through a double-buffered cp.async pipeline into shared memory with a row pitch
// of 36 words, which makes the strided 128-bit operand reads bank-conflict free.  Partial
// sums are kept in float32 for one chunk (32 non-negative terms) and folded into float64
// (or int64) accumulators per chunk, so the result carries no long-sum rounding.
#include <stdlib.h>
#include "po_common.cuh"

namespace po {

constexpr int TILE = PO_TILE;   // 64
constexpr int DK = 32;          // K elements per pipeline stage
constexpr int PITCH = DK + 4;   // smem row pitch in words

enum Kind { K_EUCL = 0, K_KT = 2, K_BC = 3, K_SC = 4 };

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, bool valid) {
    unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    int sz = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(sa), "l"(gsrc), "r"(sz));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

template <int KIND>
struct Accum {};

template <>
struct Accum<K_EUCL> {
    float c[4][4];
    double t[4][4];
    __device__ __forceinline__ void init() {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) { c[i][j] = 0.f; t[i][j] = 0.0; }
    }
    __device__ __forceinline__ void term(int i, int j, float a, float b) {
        const float d = a - b;
        c[i][j] = fmaf(d, d, c[i][j]);
    }
    __device__ __forceinline__ void fold() {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) { t[i][j] += (double)c[i][j]; c[i][j] = 0.f; }
    }
    __device__ __forceinline__ double result(int i, int j, double, double) const { return sqrt(t[i][j]); }
};

template <>
struct Accum<K_BC> {  // sum|a-b|; the denominator sum|a+b| = sum a + sum b for non-negative profiles (aux)
    float c[4][4];
    double t[4][4];
    __device__ __forceinline__ void init() {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) { c[i][j] = 0.f; t[i][j] = 0.0; }
    }
    __device__ __forceinline__ void term(int i, int j, float a, float b) { c[i][j] += fabsf(a - b); }
    __device__ __forceinline__ void fold() {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) { t[i][j] += (double)c[i][j]; c[i][j] = 0.f; }
    }
    __device__ __forceinline__ double result(int i, int j, double sa, double sb) const {
        return t[i][j] / (sa + sb);  // 0/0 -> NaN, as scipy's braycurtis
    }
};

template <>
struct Accum<K_SC> {  // exact integer dot product of centred doubled ranks
    // The products go straight into 64-bit accumulators (one IMAD.WIDE per term): a centred doubled
    // rank reaches dim - 1, so at dim = 16384 (k = 7) 32 products of correlated rows already exceed
    // 2^31, and above dim = 46341 a single product does.  (64 <= dim <= 4096 runs on the tensor cores.)
    long long t[4][4];
    __device__ __forceinline__ void init() {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) t[i][j] = 0;
    }
    __device__ __forceinline__ void term(int i, int j, float a, float b) {
        t[i][j] += (long long)__float_as_int(a) * (long long)__float_as_int(b);
    }
    __device__ __forceinline__ void fold() {}
    __device__ __forceinline__ double result(int i, int j, double ssa, double ssb) const {
        const double den = sqrt(ssa * ssb);
        if (den == 0.0) return __longlong_as_double(0x7FF8000000000000ll);  // scipy: NaN for a constant row
        return 1.0 - (double)t[i][j] / den;
    }
};

template <>
struct Accum<K_KT> {  // concordant - discordant element pairs from packed order masks
    int c[4][4];
    __device__ __forceinline__ void init() {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) c[i][j] = 0;
    }
    __device__ __forceinline__ void fold() {}
    __device__ __forceinline__ double result(int i, int j, double ua, double ub) const {
        // Bio.Cluster kendall(): distance 1 when a row is constant -> KT = 0;
        // otherwise KT = 1 - (1 - tau), evaluated in that order for bit parity.
        if (ua == 0.0 || ub == 0.0) return 0.0;
        const double tau = (double)c[i][j] / sqrt(ua * ub);
        return 1.0 - (1.0 - tau);
    }
};

struct TileParams {
    const uint32_t* P;    // prepared rows
    const double* aux;    // per-row constants (SC, KT) or null
    int64_t ldp;          // elements per prepared row (multiple of 4)
    int64_t n;
    int64_t row0, row1, col0, col1;
    void* out;
    int64_t ld_out, out_row0, out_col0;
    void* mir;            // where mirrored tiles go (== out unless the caller gave a separate buffer)
    int64_t ld_mir, mir_row0, mir_col0;
    unsigned flags;
    int kdim;             // number of elements to stream (== ldp)
};

// TM = tile rows; tile columns are always 64; threads = 4 * TM.  MO (PO_FLAG_MIRROR_ONLY): the tile goes to the
// mirror buffer only; the instantiations of the other flags do not contain the branch.
template <int KIND, typename OUT_T, int TM, bool MO>
__global__ void __launch_bounds__(4 * TM, 2) distance_tile_kernel(const TileParams p) {
    constexpr int NT = 4 * TM;          // threads
    constexpr int RS = TM / 4;          // row stride between the 4 rows a thread owns
    constexpr int TN = TILE;            // 64 columns
    constexpr int SP = PITCH;
    constexpr int STAGE_WORDS = (TM + TN) * PITCH;
    constexpr int TP = TN + 1;          // pitch of the output staging tile
    constexpr int SMEM_WORDS = (2 * STAGE_WORDS * 4 > (int)sizeof(OUT_T) * TM * TP)
                                   ? 2 * STAGE_WORDS : ((int)sizeof(OUT_T) * TM * TP + 3) / 4;
    __shared__ __align__(16) uint32_t smem[SMEM_WORDS];  // [stage][A rows | B rows][SP]
    const int64_t row_base = p.row0 + (int64_t)blockIdx.y * TM;
    const int64_t col_base = p.col0 + (int64_t)blockIdx.x * TN;
    if ((p.flags & PO_FLAG_SKIP_LOWER) && col_base + TN <= row_base) return;

    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;  // ty in [0, RS)

    const int64_t nlast = p.n - 1;
    const int nchunks = (p.kdim + DK - 1) / DK;
    const int lrow = tid >> 3, lc4 = tid & 7;    // 128-bit loader: 8 float4 per row
    constexpr int LROWS = NT / 8;

    auto issue = [&](int chunk, int stage) {
        uint32_t* sA = smem + stage * STAGE_WORDS;
        uint32_t* sB = sA + TM * PITCH;
        const int k0 = chunk * DK;
        {
            const bool ok = (k0 + lc4 * 4) < p.kdim;
#pragma unroll
            for (int r = lrow; r < TM; r += LROWS)
                cp_async16(sA + r * SP + lc4 * 4, p.P + min(row_base + r, nlast) * p.ldp + k0 + lc4 * 4, ok);
#pragma unroll
            for (int r = lrow; r < TN; r += LROWS)
                cp_async16(sB + r * SP + lc4 * 4, p.P + min(col_base + r, nlast) * p.ldp + k0 + lc4 * 4, ok);
        }
        cp_async_commit();
    };

    Accum<KIND> acc;
    acc.init();

    issue(0, 0);
    for (int ch = 0; ch < nchunks; ++ch) {
        const int stage = ch & 1;
        if (ch + 1 < nchunks) {
            issue(ch + 1, stage ^ 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        const uint32_t* sA = smem + stage * STAGE_WORDS;
        const uint32_t* sB = sA + TM * PITCH;
        if constexpr (KIND == K_KT) {
            // elements come in groups of 8 words: 4 "up" masks then 4 "down" masks
#pragma unroll
            for (int g8 = 0; g8 < DK / 8; ++g8) {
                uint4 ua[4], da[4], ub[4], db[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    ua[i] = *reinterpret_cast<const uint4*>(sA + (ty + RS * i) * SP + g8 * 8);
                    da[i] = *reinterpret_cast<const uint4*>(sA + (ty + RS * i) * SP + g8 * 8 + 4);
                    ub[i] = *reinterpret_cast<const uint4*>(sB + (tx + 16 * i) * SP + g8 * 8);
                    db[i] = *reinterpret_cast<const uint4*>(sB + (tx + 16 * i) * SP + g8 * 8 + 4);
                }
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const uint32_t au[4] = {ua[i].x, ua[i].y, ua[i].z, ua[i].w};
                        const uint32_t ad[4] = {da[i].x, da[i].y, da[i].z, da[i].w};
                        const uint32_t bu[4] = {ub[j].x, ub[j].y, ub[j].z, ub[j].w};
                        const uint32_t bd[4] = {db[j].x, db[j].y, db[j].z, db[j].w};
#pragma unroll
                        for (int w = 0; w < 4; ++w) {
                            const uint32_t con = (au[w] & bu[w]) | (ad[w] & bd[w]);
                            const uint32_t dis = (au[w] & bd[w]) | (ad[w] & bu[w]);
                            acc.c[i][j] += __popc(con) - __popc(dis);
                        }
                    }
            }
        } else {
#pragma unroll
            for (int d4 = 0; d4 < DK / 4; ++d4) {
                float4 a4[4], b4[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    a4[i] = *reinterpret_cast<const float4*>(sA + (ty + RS * i) * SP + d4 * 4);
                    b4[i] = *reinterpret_cast<const float4*>(sB + (tx + 16 * i) * SP + d4 * 4);
                }
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        acc.term(i, j, a4[i].x, b4[j].x);
                        acc.term(i, j, a4[i].y, b4[j].y);
                        acc.term(i, j, a4[i].z, b4[j].z);
                        acc.term(i, j, a4[i].w, b4[j].w);
                    }
            }
            acc.fold();
        }
        __syncthreads();
    }

    // ---- epilogue: stage the tile in shared memory, then coalesced stores (and the mirror) ----
    OUT_T* tile = reinterpret_cast<OUT_T*>(smem);  // [TM][TP]
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int64_t r = row_base + ty + RS * i;
        const double auxr = (p.aux && r < p.n) ? p.aux[r] : 0.0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int64_t c = col_base + tx + 16 * j;
            const double auxc = (p.aux && c < p.n) ? p.aux[c] : 0.0;
            tile[(ty + RS * i) * TP + tx + 16 * j] = (OUT_T)acc.result(i, j, auxr, auxc);
        }
    }
    __syncthreads();
    OUT_T* out = reinterpret_cast<OUT_T*>(p.out);
    const int64_t rmax = min((int64_t)TM, p.row1 - row_base);
    const int64_t cmax = min((int64_t)TN, p.col1 - col_base);
    if (!MO) {
        for (int e = tid; e < TM * TN; e += NT) {
            const int r = e >> 6, c = e & 63;
            if (r < rmax && c < cmax)
                out[(row_base + r - p.out_row0) * p.ld_out + (col_base + c - p.out_col0)] = tile[r * TP + c];
        }
    }
    if ((p.flags & PO_FLAG_MIRROR) && row_base + TM <= col_base) {
        OUT_T* mir = reinterpret_cast<OUT_T*>(p.mir);
        for (int e = tid; e < TM * TN; e += NT) {
            const int c = e / TM, r = e % TM;  // consecutive threads walk r: contiguous in the mirrored row
            if (r < rmax && c < cmax)
                mir[(col_base + c - p.mir_row0) * p.ld_mir + (row_base + r - p.mir_col0)] = tile[r * TP + c];
        }
    }
}

template <int KIND, int TM>
static int launch_kind(const TileParams& p, int out_dtype, cudaStream_t stream) {
    const int64_t tr = (p.row1 - p.row0 + TM - 1) / TM, tc = (p.col1 - p.col0 + TILE - 1) / TILE;
    if (tr > 65535) {
        set_error("row block too tall: %lld rows (max %d per call)", (long long)(p.row1 - p.row0), 65535 * TM);
        return PO_ERR_UNSUPPORTED;
    }
    dim3 grid((unsigned)tc, (unsigned)tr, 1);
    LaunchTimer t(1, stream);
    const bool mo = (p.flags & PO_FLAG_MIRROR_ONLY) != 0;
    if (out_dtype == PO_F32 && !mo)
        distance_tile_kernel<KIND, float, TM, false><<<grid, 4 * TM, 0, stream>>>(p);
    else if (out_dtype == PO_F32)
        distance_tile_kernel<KIND, float, TM, true><<<grid, 4 * TM, 0, stream>>>(p);
    else if (!mo)
        distance_tile_kernel<KIND, double, TM, false><<<grid, 4 * TM, 0, stream>>>(p);
    else
        distance_tile_kernel<KIND, double, TM, true><<<grid, 4 * TM, 0, stream>>>(p);
    count_launch(1);
    PO_LAUNCH_CHECK("distance_tile_kernel");
    return PO_OK;
}

int launch_distance(int metric, const void* d_P, const double* d_aux, int64_t n, int64_t dim,
                    int64_t row0, int64_t row1, int64_t col0, int64_t col1,
                    void* d_out, int64_t ld_out, int64_t out_row0, int64_t out_col0,
                    void* d_mir, int64_t ld_mir, int64_t mir_row0, int64_t mir_col0,
                    int out_dtype, unsigned flags, cudaStream_t stream) {
    if (row1 <= row0 || col1 <= col0) return PO_OK;
    if (eucl_use_gram(metric, dim) || sc_use_gram(metric, dim))
        return launch_gram(metric, d_P, d_aux, n, dim, row0, row1, col0, col1, d_out, ld_out, out_row0, out_col0, d_mir, ld_mir,
                           mir_row0, mir_col0, out_dtype, flags, stream);
    TileParams p;
    p.P = reinterpret_cast<const uint32_t*>(d_P);
    p.aux = d_aux;
    p.ldp = prepared_row_elems(metric, dim);
    p.kdim = (int)p.ldp;
    p.n = n;
    p.row0 = row0; p.row1 = row1; p.col0 = col0; p.col1 = col1;
    p.out = d_out; p.ld_out = ld_out; p.out_row0 = out_row0; p.out_col0 = out_col0;
    p.mir = d_mir; p.ld_mir = ld_mir; p.mir_row0 = mir_row0; p.mir_col0 = mir_col0;
    p.flags = flags;
    switch (metric) {
        case PO_EUCL_GRAM:
        case PO_EUCL: return launch_kind<K_EUCL, 64>(p, out_dtype, stream);
        case PO_JSD:
            return launch_jsd(d_P, n, dim, row0, row1, col0, col1, d_out, ld_out, out_row0, out_col0, d_mir, ld_mir,
                              mir_row0, mir_col0, out_dtype, flags, stream);
        case PO_BC: return launch_kind<K_BC, 64>(p, out_dtype, stream);
        case PO_SC: return launch_kind<K_SC, 64>(p, out_dtype, stream);
        case PO_KT: return launch_kind<K_KT, 64>(p, out_dtype, stream);
    }
    set_error("unknown metric %d", metric);
    return PO_ERR_ARG;
}

}  // namespace po
