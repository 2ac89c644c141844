// Jensen-Shannon divergence tiles on sm_100a: packed FP32x2 (FFMA2) math on operand
// blocks staged by bulk asynchronous copies (cp.async.bulk + mbarrier).
//
// Replaces phylodist.JSD / KL (reference core/phylodist.py:18-34, 43-68) and the JSD
// slice workers JSD_loc / JSD_h5py (bin/phyloligo.py:204-207, 248-257).
//
// Math.  The reference computes 0.5*sum(a ln(a/h) + b ln(b/h)), h = (a+b)/2, in nats
// with 0*ln0 := 0.  Per dimension this kernel evaluates the identical quantity in a
// cancellation-free form.  With s = a+b, d = a-b, x = d/s, u = x^2:
//     a ln(a/h) + b ln(b/h) = (s/2) * f(x),   f(x) = (1+x)ln(1+x) + (1-x)ln(1-x) >= 0
//     f(x) = u * G(u),  G(u) = sum_{n>=1} u^(n-1) / (n(2n-1))        (u <= 1/2)
//     f(x) = E(w) + w ln w,  w = 1-|x| = 2 min(a,b)/s, E(w)=(2-w)ln(2-w)  (u > 1/2)
// Every term is >= 0, so the sum has no cancellation; G and E are polynomial fits at
// float32 rounding level (tools/jsd_poly_fit.py) and the only transcendental is one
// MUFU.LG2 whose argument is < 0.15, where its error is relative.  No fast-math flags;
// a = b gives exactly 0; an all-zero row against a profile gives ln(2)/2.
//
// Layout.  po_prepare_profiles(JSD) writes the operands "blocked": for every group of
// 64 profiles and every chunk of 32 dimensions one 8 KB block [32 dims][64 profiles]
// (the column operand, B), and for every group of 32 profiles one 4 KB block
// [32 dims][32 profiles] (the row operand, A).  A CTA computes a 32 x 64 tile; per chunk
// it needs exactly one A block and one B block, each a single contiguous cp.async.bulk
// into a 3-stage shared-memory ring.  Thread (ty, tx) owns rows 4ty..4ty+3 and columns
// 4tx..4tx+3: per dimension it reads its four row values and its {b_j, b_j+1} pairs with
// two 128-bit shared loads and evaluates 16 terms as 8 packed f32x2 operations per step
// of the recipe (add, sub, mul, mul, Horner FMAs, mul, FMA).  The row value enters the
// add and the subtract as pk2(a, a) of one register, which ptxas emits as the scalar
// broadcast operand (R.F32) of FADD2: three 32-bit register reads instead of four.  The
// FP32 pipe of this loop is fed by register-file reads (DESIGN.md section 4.3), so the
// operand that is the same in both halves is stored and read once.
//
// Two-phase evaluation.  Phase 1 adds the series value q*G(u) for every term and tracks
// the largest u it met.  If some lane of the warp met u > 1/2 in this dimension, phase 2
// walks the 8 packed term pairs and, for those in which some lane has u > 1/2 (a
// warp-uniform test: typically the pairs of one outlier profile of the tile), forms the
// log-based value and adds the difference to the series value for exactly the terms with
// u > 1/2 (G's polynomial is finite on [0, 1], so the provisional value is harmless).
// Dense profiles (4^k bins well covered) need phase 2 in a few percent of the (warp,
// dimension) steps; sparse ones (5 kb contigs at k = 5) need it almost always and run
// about 1.6x slower per term.
//
// Chunk variants.  Whether a chunk of 32 dimensions of a tile can meet u > 1/2 at all is known
// before its loop starts: po_prepare_profiles stores, per group of 64 profiles and dimension, the
// smallest and largest value of the group, and a pair (a, b) with max/min <= r has
// u <= ((r-1)/(r+1))^2.  Per (tile, chunk) the warp evaluates the bound from the two groups' ranges
// (one dimension per lane, loaded a chunk ahead) and runs one of three loops:
//   V0  ratio <= 3   (u <= 1/4): degree-4 fit of G, no tracking of u, no phase 2   (10 FP32-pipe ops per term)
//   V1  ratio <= 5.8 (u < 1/2): the degree-6 fit, no tracking, no phase 2          (12 ops)
//   V2  anything else: the two-phase loop above.
// The dimensions are permuted (the same permutation for every profile: a sum does not care) in
// ascending order of their spread max/min over all profiles, so that the narrow dimensions share
// chunks: at C2, 55 % of the (tile, chunk) pairs run V0 and 11 % V1, against 0 % and 18 % in the natural
// order.  Both groups are the 64-aligned groups of the global profile index, for rows and columns
// alike, so the variant of an entry (r, c) is that of (c, r) and does not depend on which call or tile
// computes it: matrices stay bitwise symmetric and block rows equal the symmetric run bit for bit.
#include "po_common.cuh"

namespace po {

typedef unsigned long long u64;

constexpr int JT_M = 32;           // tile rows
constexpr int JT_N = 64;           // tile columns
constexpr int JDK = 32;            // dimensions per chunk
#ifndef JSD_STAGES
#define JSD_STAGES 3
#endif
#ifndef JSD_UNROLL
#define JSD_UNROLL 2
#endif
#ifndef JSD_CTAS
#define JSD_CTAS 4
#endif
#ifndef JSD_P2_BITS
#define JSD_P2_BITS 0x3F000000u  // 0.5f: a warp that met a larger u in a dimension runs phase 2 for it
#endif
#ifndef JSD_BLOCK_P2
#define JSD_BLOCK_P2 1  // phase 2 only for the term pairs that need it
#endif
constexpr int JSTAGES = JSD_STAGES;
constexpr int JUNROLL = JSD_UNROLL;
constexpr int JA_FLOATS = JDK * JT_M;  // one row-operand block: 4 KB
constexpr int JB_FLOATS = JDK * JT_N;  // one column-operand block: 8 KB
constexpr int JSTAGE_BYTES = (JA_FLOATS + JB_FLOATS) * 4;
constexpr int JTHREADS = 128;
constexpr int JT_TOTALS_BYTES = 16 * JTHREADS * 8;  // every thread's 16 float64 totals
constexpr int JRASTER = 128;        // tile columns per rasterisation chunk

// ---- packed f32x2 helpers (sm_100 FADD2 / FMUL2 / FFMA2) ----
__device__ __forceinline__ u64 pk2(float lo, float hi) {
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk2(u64 v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ u64 add2(u64 a, u64 b) {
    u64 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ u64 sub2(u64 a, u64 b) {
    u64 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ u64 mul2(u64 a, u64 b) {
    u64 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) {
    u64 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
// .ftz forms: a single MUFU each.  Arguments are never denormal (operand bias 1e-30).
__device__ __forceinline__ float lg2_approx(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// regime A factor G(u), u in [0, 1/2]: degree-6 minimax fit (tools/jsd_poly_fit.py),
// relative error 5.4e-8 in exact arithmetic, 1.7e-7 in float32 Horner arithmetic
#define JG6 5.813299561e-02f
#define JG5 -2.857199317e-02f
#define JG4 3.964714137e-02f
#define JG3 3.233825144e-02f
#define JG2 6.697004847e-02f
#define JG1 1.666565838e-01f
#define JG0 1.000000054e+00f

// u in [0, 0.26]: degree-4 fit, relative error 7.0e-8 in exact arithmetic, 1.9e-7 in float32 Horner arithmetic
#define JH4 3.614963273e-02f
#define JH3 3.220779540e-02f
#define JH2 6.700734910e-02f
#define JH1 1.666553656e-01f
#define JH0 1.000000059e+00f
#define JSD_RATIO_V0 3.0f   // max/min <= 3   -> u <= 0.25
#define JSD_RATIO_V1 5.8f   // max/min <= 5.8 -> u <= 0.4983 (the two-phase threshold is 1/2)

__device__ __forceinline__ float jsd_G(float u) {
    float G = JG6;
    G = fmaf(G, u, JG5);
    G = fmaf(G, u, JG4);
    G = fmaf(G, u, JG3);
    G = fmaf(G, u, JG2);
    G = fmaf(G, u, JG1);
    G = fmaf(G, u, JG0);
    return G;
}
// regime B value f = E(w) + w ln w with v = w/2 = min(a,b)/s in [0, 0.1465]
__device__ __forceinline__ float jsd_fB(float v) {
    float E = 2.100300184e-01f;
    E = fmaf(E, v, 3.274813073e-01f);
    E = fmaf(E, v, 1.000313256e+00f);
    E = fmaf(E, v, -2.000005795e+00f);
    E = fmaf(E, v, 1.386294378e+00f);
    const float vl = v * 1.386294361f;  // 2 ln2 * v
    return fmaf(vl, lg2_approx(v), E);
}

// ---- mbarrier / bulk copy ----
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}

struct JsdParams {
    const float* B;   // column-operand blocks  [n/64 groups][nchunks][32][64]
    const float* A;   // row-operand blocks     [n/32 groups][nchunks][32][32]
    const float* gmin;  // [n/64 groups][nchunks * 32] smallest / largest value of the group per (permuted) dimension
    const float* gmax;
    int nchunks;
    int64_t n;
    int64_t row0, row1, col0, col1;
    int64_t tile_row0, tile_col0;  // first tile origin (multiples of 32 / 64)
    int64_t tiles_r, tiles_c;      // tile grid, walked in chunks of JRASTER tile columns (L2 reuse)
    void* out;
    int64_t ld_out, out_row0, out_col0;
    void* mir;  // where mirrored tiles go (== out unless the caller gave a separate buffer)
    int64_t ld_mir, mir_row0, mir_col0;
    unsigned flags;
};

// One chunk (32 dimensions) of a thread's 4 x 4 pairs, as 8 packed term pairs per dimension.
// V = 0: degree-4 fit, u <= 1/4 guaranteed; V = 1: degree-6 fit, u < 1/2 guaranteed; V = 2: two phases.
// V = 2 tracks u only in the dimensions whose bit is set in p2dims: in the others the value ranges of the
// warp's rows and of the column group bound u below 1/2, so phase 2 cannot run there and the loop computes
// exactly what V = 1 computes.
template <int V>
__device__ __forceinline__ void jsd_chunk(const float4* __restrict__ sA, const ulonglong2* __restrict__ sB, u64 (&c2)[4][2],
                                          unsigned p2dims) {
    const u64 g6 = pk2(JG6, JG6), g5 = pk2(JG5, JG5), g4 = pk2(JG4, JG4);
    const u64 g3 = pk2(JG3, JG3), g2 = pk2(JG2, JG2), g1 = pk2(JG1, JG1), g0 = pk2(JG0, JG0);
    const u64 h4 = pk2(JH4, JH4), h3 = pk2(JH3, JH3), h2 = pk2(JH2, JH2), h1 = pk2(JH1, JH1), h0 = pk2(JH0, JH0);
#pragma unroll JUNROLL
    for (int d = 0; d < JDK; ++d) {
        const float4 Av = sA[d * (JT_M / 4)];
        const ulonglong2 Bv = sB[d * (JT_N / 4)];
        const float a[4] = {Av.x, Av.y, Av.z, Av.w};
        const u64 a2[4] = {pk2(a[0], a[0]), pk2(a[1], a[1]), pk2(a[2], a[2]), pk2(a[3], a[3])};
        const u64 b2[2] = {Bv.x, Bv.y};
        u64 dd[4][2], xx[4][2], uu[4][2];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const u64 sm = add2(a2[i], b2[j]);
                dd[i][j] = sub2(a2[i], b2[j]);
                float s0, s1;
                upk2(sm, s0, s1);
                xx[i][j] = mul2(dd[i][j], pk2(rcp_approx(s0), rcp_approx(s1)));
                uu[i][j] = mul2(xx[i][j], xx[i][j]);
            }
        u64 G[4][2];
#define JSD_HORNER_FIRST(ga, gb)                  \
    _Pragma("unroll") for (int i = 0; i < 4; ++i) \
        _Pragma("unroll") for (int j = 0; j < 2; ++j) G[i][j] = fma2(ga, uu[i][j], gb);
#define JSD_HORNER(gk)                            \
    _Pragma("unroll") for (int i = 0; i < 4; ++i) \
        _Pragma("unroll") for (int j = 0; j < 2; ++j) G[i][j] = fma2(G[i][j], uu[i][j], gk);
        if (V == 0) {
            JSD_HORNER_FIRST(h4, h3)
            JSD_HORNER(h2)
            JSD_HORNER(h1)
            JSD_HORNER(h0)
        } else {
            JSD_HORNER_FIRST(g6, g5)
            JSD_HORNER(g4)
            JSD_HORNER(g3)
            JSD_HORNER(g2)
            JSD_HORNER(g1)
            JSD_HORNER(g0)
        }
#undef JSD_HORNER
#undef JSD_HORNER_FIRST
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j) c2[i][j] = fma2(mul2(dd[i][j], xx[i][j]), G[i][j], c2[i][j]);

        if (V == 2 && ((p2dims >> d) & 1u)) {
            float umax = 0.f;
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    float u0, u1;
                    upk2(uu[i][j], u0, u1);
                    umax = fmaxf(umax, fmaxf(u0, u1));
                }
            // largest u of the warp's 512 terms in this dimension (u >= 0: bit order = value order)
            const unsigned umax_w = __reduce_max_sync(0xFFFFFFFFu, __float_as_uint(umax));
            if (umax_w > JSD_P2_BITS) {
                // phase 2, packed: for the term pairs in which some lane met u > 1/2, form the log-based
                // value s * fB(min(a,b)/s) and add (that - series value) where u > 1/2, 0 elsewhere.
                // Typically a few of the 8 pairs are concerned (one outlier profile of the tile); sparse
                // profiles flag all of them.
                float b[4];
                upk2(b2[0], b[0], b[1]);
                upk2(b2[1], b[2], b[3]);
                const u64 e4 = pk2(2.100300184e-01f, 2.100300184e-01f), e3 = pk2(3.274813073e-01f, 3.274813073e-01f);
                const u64 e2 = pk2(1.000313256e+00f, 1.000313256e+00f), e1 = pk2(-2.000005795e+00f, -2.000005795e+00f);
                const u64 e0 = pk2(1.386294378e+00f, 1.386294378e+00f), ln4 = pk2(1.386294361f, 1.386294361f);
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        float u0, u1;
                        upk2(uu[i][j], u0, u1);
#if JSD_BLOCK_P2
                        if (!__any_sync(0xFFFFFFFFu, (u0 > 0.5f) | (u1 > 0.5f))) continue;
#endif
                        const u64 sm = add2(a2[i], b2[j]);
                        float s0, s1;
                        upk2(sm, s0, s1);  // 1/s again (same MUFU result as in phase 1) rather than 16 live registers
                        const u64 v = mul2(pk2(fminf(a[i], b[2 * j]), fminf(a[i], b[2 * j + 1])),
                                           pk2(rcp_approx(s0), rcp_approx(s1)));
                        u64 E = fma2(e4, v, e3);
                        E = fma2(E, v, e2);
                        E = fma2(E, v, e1);
                        E = fma2(E, v, e0);
                        float v0, v1;
                        upk2(v, v0, v1);
                        const u64 fB = fma2(mul2(v, ln4), pk2(lg2_approx(v0), lg2_approx(v1)), E);
                        const u64 series = mul2(mul2(dd[i][j], xx[i][j]), G[i][j]);
                        const u64 delta = sub2(mul2(sm, fB), series);
                        float d0, d1;
                        upk2(delta, d0, d1);
                        c2[i][j] = add2(c2[i][j], pk2(u0 > 0.5f ? d0 : 0.f, u1 > 0.5f ? d1 : 0.f));
                    }
            }
        }
    }
}

template <typename OUT_T>
__global__ void __launch_bounds__(JTHREADS, JSD_CTAS) jsd_tile_kernel(const JsdParams p) {
    extern __shared__ __align__(128) unsigned char jsmem[];
    __shared__ __align__(8) unsigned long long bars[JSTAGES];
    __shared__ unsigned done_warps[JSTAGES];  // warps that have finished reading a stage
    // rasterisation: chunks of JRASTER tile columns, all tile rows inside a chunk, so that the
    // chunk's column operands (JRASTER x 64 KB at 256 dimensions) stay in L2 while the rows stream
    const int64_t per_chunk = p.tiles_r * JRASTER;
    const int64_t chunk = (int64_t)blockIdx.x / per_chunk;
    const int64_t rem = (int64_t)blockIdx.x - chunk * per_chunk;
    const int64_t gw = min((int64_t)JRASTER, p.tiles_c - chunk * JRASTER);
    const int64_t row_base = p.tile_row0 + (rem / gw) * JT_M;
    const int64_t col_base = p.tile_col0 + (chunk * JRASTER + rem % gw) * JT_N;
    if ((p.flags & PO_FLAG_SKIP_LOWER) && col_base + JT_N <= row_base) return;

    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int nchunks = p.nchunks;
    const float* gA = p.A + (size_t)(row_base / JT_M) * nchunks * JA_FLOATS;
    const float* gB = p.B + (size_t)(col_base / JT_N) * nchunks * JB_FLOATS;
    const unsigned smem0 = smem_u32(jsmem);
    const unsigned bar0 = smem_u32(bars);

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < JSTAGES; ++s) {
            mbar_init(bar0 + 8 * s, 1);
            done_warps[s] = 0;
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    auto issue = [&](int chunk) {
        const int s = chunk % JSTAGES;
        const unsigned bar = bar0 + 8 * s;
        const unsigned dst = smem0 + s * JSTAGE_BYTES;
        mbar_expect_tx(bar, JSTAGE_BYTES);
        bulk_g2s(dst, gA + (size_t)chunk * JA_FLOATS, JA_FLOATS * 4, bar);
        bulk_g2s(dst + JA_FLOATS * 4, gB + (size_t)chunk * JB_FLOATS, JB_FLOATS * 4, bar);
    };
    if (tid == 0) {
        for (int c = 0; c < JSTAGES && c < nchunks; ++c) issue(c);
    }

    // variant of a chunk from the value ranges of the two 64-profile groups: one dimension per lane.
    // Bit 2 of a lane's code flags the dimensions in which this warp may meet u > 1/2: the range of the
    // warp's own 8 rows (read from the A block in global memory) against the column group's range.  Where
    // it is clear, phase 2 cannot run, so V2 skips tracking u there; the results do not change.
    const float* rW = gA + (tid & 31) * JT_M + 8 * (tid >> 5);
    const float* rI_min = p.gmin + (size_t)(row_base / 64) * nchunks * JDK + (tid & 31);
    const float* rI_max = p.gmax + (size_t)(row_base / 64) * nchunks * JDK + (tid & 31);
    const float* rJ_min = p.gmin + (size_t)(col_base / 64) * nchunks * JDK + (tid & 31);
    const float* rJ_max = p.gmax + (size_t)(col_base / 64) * nchunks * JDK + (tid & 31);
    auto lane_code = [&](int ch) -> unsigned {
#ifdef JSD_FORCE_VARIANT
        return JSD_FORCE_VARIANT | 4u;  // every dimension flagged
#else
        const float ilo = rI_min[ch * JDK], ihi = rI_max[ch * JDK], jlo = rJ_min[ch * JDK], jhi = rJ_max[ch * JDK];
        const float4 w0 = *reinterpret_cast<const float4*>(rW + (size_t)ch * JA_FLOATS);
        const float4 w1 = *reinterpret_cast<const float4*>(rW + (size_t)ch * JA_FLOATS + 4);
        const float wlo = fminf(fminf(fminf(w0.x, w0.y), fminf(w0.z, w0.w)), fminf(fminf(w1.x, w1.y), fminf(w1.z, w1.w)));
        const float whi = fmaxf(fmaxf(fmaxf(w0.x, w0.y), fmaxf(w0.z, w0.w)), fmaxf(fmaxf(w1.x, w1.y), fmaxf(w1.z, w1.w)));
        const unsigned flag = (whi <= JSD_RATIO_V1 * jlo && jhi <= JSD_RATIO_V1 * wlo) ? 0u : 4u;
        // a in [ilo, ihi], b in [jlo, jhi]: max(a/b, b/a) <= max(ihi/jlo, jhi/ilo)
        if (ihi <= JSD_RATIO_V0 * jlo && jhi <= JSD_RATIO_V0 * ilo) return flag;
        if (ihi <= JSD_RATIO_V1 * jlo && jhi <= JSD_RATIO_V1 * ilo) return flag | 1u;
        return flag | 2u;
#endif
    };
    unsigned code_next = lane_code(0);

    // The float64 totals are touched once per chunk: they live in shared memory behind the ring
    // ([16][JTHREADS], conflict-free), which leaves the registers to the chunk loops and keeps them
    // free of spills at JSD_CTAS CTAs per SM.
    double* t = reinterpret_cast<double*>(jsmem + JSTAGES * JSTAGE_BYTES) + tid;
    u64 c2[4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        c2[i][0] = 0ull;
        c2[i][1] = 0ull;
#pragma unroll
        for (int j = 0; j < 4; ++j) t[(4 * i + j) * JTHREADS] = 0.0;
    }

    for (int ch = 0; ch < nchunks; ++ch) {
        const int s = ch % JSTAGES;
        const unsigned variant = __reduce_max_sync(0xFFFFFFFFu, code_next & 3u);
        const unsigned p2dims = __ballot_sync(0xFFFFFFFFu, (code_next & 4u) != 0u);  // lane = dimension of the chunk
        if (ch + 1 < nchunks) code_next = lane_code(ch + 1);  // in flight during this chunk's loop
        mbar_wait(bar0 + 8 * s, (unsigned)((ch / JSTAGES) & 1));
        const float4* sA = reinterpret_cast<const float4*>(jsmem + s * JSTAGE_BYTES) + ty;
        const ulonglong2* sB = reinterpret_cast<const ulonglong2*>(jsmem + s * JSTAGE_BYTES + JA_FLOATS * 4) + tx;
        if (variant == 0u) jsd_chunk<0>(sA, sB, c2, 0u);
        else if (variant == 1u) jsd_chunk<1>(sA, sB, c2, 0u);
        else jsd_chunk<2>(sA, sB, c2, p2dims);
        // fold the chunk's float32 partial sums (32 non-negative terms each) into float64
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                float c0, c1;
                upk2(c2[i][j], c0, c1);
                t[(4 * i + 2 * j) * JTHREADS] += (double)c0;
                t[(4 * i + 2 * j + 1) * JTHREADS] += (double)c1;
                c2[i][j] = 0ull;
            }
        // Stage s is refilled by whichever warp finishes reading it last: no block-wide barrier in the
        // chunk loop, the warps drift by up to JSTAGES - 1 chunks.
        __syncwarp();
        if ((tid & 31) == 0 && ch + JSTAGES < nchunks) {
            __threadfence_block();
            // the counter only grows: every JTHREADS / 32-th arrival is the last warp of a round
            if (atomicAdd(&done_warps[s], 1u) % (JTHREADS / 32) == JTHREADS / 32 - 1) issue(ch + JSTAGES);
        }
    }
    __syncthreads();  // the epilogue reuses the ring as the tile buffer (the totals lie behind it)

    // ---- epilogue: stage the tile in shared memory, then coalesced stores (and the mirror) ----
    constexpr int TP = JT_N + 1;
    OUT_T* tile = reinterpret_cast<OUT_T*>(jsmem);  // [32][65]
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) tile[(4 * ty + i) * TP + 4 * tx + j] = (OUT_T)(0.25 * t[(4 * i + j) * JTHREADS]);
    __syncthreads();
    OUT_T* out = reinterpret_cast<OUT_T*>(p.out);
    const int r_lo = (int)max((int64_t)0, p.row0 - row_base), r_hi = (int)min((int64_t)JT_M, p.row1 - row_base);
    const int c_lo = (int)max((int64_t)0, p.col0 - col_base), c_hi = (int)min((int64_t)JT_N, p.col1 - col_base);
    for (int e = tid; e < JT_M * JT_N; e += JTHREADS) {
        const int r = e >> 6, c = e & 63;
        if (r >= r_lo && r < r_hi && c >= c_lo && c < c_hi)
            out[(row_base + r - p.out_row0) * p.ld_out + (col_base + c - p.out_col0)] = tile[r * TP + c];
    }
    if ((p.flags & PO_FLAG_MIRROR) && row_base + JT_M <= col_base) {
        OUT_T* mir = reinterpret_cast<OUT_T*>(p.mir);
        for (int e = tid; e < JT_M * JT_N; e += JTHREADS) {
            const int c = e >> 5, r = e & 31;  // consecutive threads walk r: contiguous in the mirrored row
            if (r >= r_lo && r < r_hi && c >= c_lo && c < c_hi)
                mir[(col_base + c - p.mir_row0) * p.ld_mir + (row_base + r - p.mir_col0)] = tile[r * TP + c];
        }
    }
}

int launch_jsd(const void* d_P, int64_t n, int64_t dim, int64_t row0, int64_t row1, int64_t col0, int64_t col1,
               void* d_out, int64_t ld_out, int64_t out_row0, int64_t out_col0, void* d_mir, int64_t ld_mir,
               int64_t mir_row0, int64_t mir_col0, int out_dtype, unsigned flags, cudaStream_t stream) {
    const int64_t ldp = prepared_row_elems(PO_JSD, dim);
    const int64_t npad = (n + 63) / 64 * 64;
    JsdParams p;
    p.B = reinterpret_cast<const float*>(d_P);
    p.A = p.B + npad * ldp;
    p.gmin = p.A + npad * ldp;
    p.gmax = p.gmin + (npad / 64) * ldp;
    p.nchunks = (int)(ldp / JDK);
    p.n = n;
    p.row0 = row0; p.row1 = row1; p.col0 = col0; p.col1 = col1;
    p.tile_row0 = row0 / JT_M * JT_M;
    p.tile_col0 = col0 / JT_N * JT_N;
    p.out = d_out; p.ld_out = ld_out; p.out_row0 = out_row0; p.out_col0 = out_col0;
    p.mir = d_mir; p.ld_mir = ld_mir; p.mir_row0 = mir_row0; p.mir_col0 = mir_col0;
    p.flags = flags;
    const int64_t tr = (row1 - p.tile_row0 + JT_M - 1) / JT_M, tc = (col1 - p.tile_col0 + JT_N - 1) / JT_N;
    if (tr * tc > 0x7FFFFFFFll) {
        set_error("block too large: %lld x %lld tiles", (long long)tr, (long long)tc);
        return PO_ERR_UNSUPPORTED;
    }
    p.tiles_r = tr;
    p.tiles_c = tc;
    const size_t smem = (size_t)JSTAGES * JSTAGE_BYTES + JT_TOTALS_BYTES;
    dim3 grid((unsigned)(tr * tc), 1, 1);
    LaunchTimer tm(1, stream);
    // the opt-in is per device: set it on every launch (a process may drive several GPUs)
    if (out_dtype == PO_F32) {
        PO_CUDA_CHECK(cudaFuncSetAttribute(jsd_tile_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        jsd_tile_kernel<float><<<grid, JTHREADS, smem, stream>>>(p);
    } else {
        PO_CUDA_CHECK(cudaFuncSetAttribute(jsd_tile_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        jsd_tile_kernel<double><<<grid, JTHREADS, smem, stream>>>(p);
    }
    count_launch(1);
    PO_LAUNCH_CHECK("jsd_tile_kernel");
    return PO_OK;
}

}  // namespace po
