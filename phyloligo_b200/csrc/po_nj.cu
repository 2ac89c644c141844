// phyloselect.R's neighbour-joining trees (reference bin/phyloselect.R:22-35, ape's nj / bionj) on the resident
// N x N matrix, bit for bit in the order of float64 operations DESIGN.md section 4.11 fixes.
//
// State.  A float64 working copy W with C = round_up(n + NJ_HEADROOM, 32) slots per side (row stride C).  Slot
// order is list order: the live members occupy slots in [f, C) in the order of the active list, with dead slots
// ("holes") between them.  A join's new node goes first in the list, so it takes the free slot f - 1 in front.
// When the front is used up, or holes make up an eighth of the span, a compaction packs the live members into
// [C - m, C) in the same order (po_nj_run's host loop knows f and m: both follow from the join count).
//   - Only the upper triangle W[r][c], r < c, holds D.  BIONJ keeps its variance V in the lower triangle
//     (Gascuel's packed layout), so both methods need one C x C array.
//   - Every upper entry in a dead slot's row or column is +0.0.  Sums start at +0.0 and can never become -0.0, so
//     adding such a zero leaves a sum bitwise unchanged: the row sums skip holes without a branch.
//   - S of a dead slot is NaN, so its pairs never enter the strict-< Q scan.
//   - Because slot order is list order, the Q tie key (list positions, lexicographic) is the slot pair.
//
// A join is four launches on the stream, with no host synchronisation:
//   nj_rowsum_kernel  S_s for every slot, one lane per slot.  The sum runs sequentially in the fixed order: first
//                     row s right of the diagonal (the members after s), then column s from f down to s (the members
//                     before s), both in ascending slot order.  A CTA owns 32 slots and streams 64-entry tiles of its
//                     32 rows, then of its 32 columns, through shared memory so that every global load is coalesced;
//                     warp 0 adds while the CTA loads the next tile.  8 m^2 bytes.
//   nj_qscan_kernel   Q over the upper triangle, one warp per row; per-CTA (Q, key) minimum.  4 m^2 bytes.
//   nj_finish_kernel  one CTA: the global minimum, the branch lengths, the two edges, BIONJ's lambda (its sequential
//                     sum over the list is one thread's chain of adds, fed through shared memory), the join record.
//   nj_update_kernel  row u (and, for BIONJ, V in column u); zeroes the upper entries of a and b.  O(m).
// All float64 arithmetic whose order is fixed is written with __dadd_rn / __dsub_rn / __dmul_rn / __ddiv_rn, so
// no FMA contraction changes a bit.  There is no floating-point atomic.  A join that finds no pair with Q below
// ape's bound 1e50 sets the status, and every later kernel returns at once.
#include <algorithm>
#include <climits>
#include <cmath>
#include "po_common.cuh"

namespace po {

namespace {

constexpr int NJ_HEADROOM = 256;  // front slots for new nodes before the first compaction
constexpr int RS_THREADS = 256;
constexpr int RS_SLOTS = 32;  // slots of one row-sum CTA (one lane each)
constexpr int RS_DEPTH = 64;  // entries of one tile per slot
constexpr int RS_PAD = RS_DEPTH + 1;
constexpr int QS_THREADS = 512;
constexpr int QS_MAX_CTAS = 1024;
constexpr int FIN_THREADS = 512;
constexpr int LAM_CHUNK = 2048;
constexpr long long NO_KEY = LLONG_MAX;
constexpr double Q_BOUND = 1e50;

enum { NJ_NJ = 0, NJ_BIONJ = 1 };
enum { ST_OK = 0, ST_NO_PAIR = 1 };

struct Rec {  // the join just decided
    int a, b, u, pad;
    double A, la, lb, lam, vab;
};

// workspace: S double[C], partial q double[QS_MAX_CTAS], partial key int64[QS_MAX_CTAS], record, alive int32[C],
// node int32[C], live int32[C], status int32[2]
struct Work {
    double* S;
    double* pq;
    long long* pk;
    Rec* rec;
    int *alive, *node, *live, *status;
};
int64_t capacity(int64_t n) { return (n + NJ_HEADROOM + 31) / 32 * 32; }
Work carve(void* d_work, int64_t C) {
    Work w;
    char* p = reinterpret_cast<char*>(d_work);
    w.S = reinterpret_cast<double*>(p);
    w.pq = w.S + C;
    w.pk = reinterpret_cast<long long*>(w.pq + QS_MAX_CTAS);
    w.rec = reinterpret_cast<Rec*>(w.pk + QS_MAX_CTAS);
    w.alive = reinterpret_cast<int*>(w.rec + 1);
    w.node = w.alive + C;
    w.live = w.node + C;
    w.status = w.live + C;
    return w;
}
int64_t workspace_bytes(int64_t n) {
    const int64_t C = capacity(n);
    return C * 8 + QS_MAX_CTAS * 16 + (int64_t)sizeof(Rec) + 3 * C * 4 + 2 * 4;
}
// rows of the compaction's staging buffer: at most 256 MB, at least one row
int64_t stage_rows(int64_t n) { return std::max<int64_t>(1, std::min<int64_t>(n, (int64_t(1) << 25) / std::max<int64_t>(n, 1))); }

__device__ __forceinline__ double up(const double* W, int64_t C, int r, int c) {  // D(r, c), r != c
    return r < c ? __ldcg(W + (int64_t)r * C + c) : __ldcg(W + (int64_t)c * C + r);
}
__device__ __forceinline__ double lo(const double* W, int64_t C, int r, int c) {  // V(r, c), r != c
    return r > c ? __ldcg(W + (int64_t)r * C + c) : __ldcg(W + (int64_t)c * C + r);
}
__device__ __forceinline__ double half(double x) { return __ddiv_rn(x, 2.0); }

template <typename T>
__global__ void nj_copy_kernel(const T* __restrict__ D, int64_t ld, int n, double* __restrict__ W, int64_t C, int f) {
    for (int r = blockIdx.x; r < n; r += gridDim.x) {
        const T* src = D + (int64_t)r * ld;
        double* dst = W + (int64_t)(f + r) * C + f;
        for (int c = threadIdx.x; c < n; c += blockDim.x) dst[c] = (double)src[c];
    }
}

__global__ void nj_init_kernel(int n, int64_t C, int f, Work w) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < C) {
        const bool leaf = i >= f && i < f + n;
        w.alive[i] = leaf ? 1 : 0;
        w.node[i] = leaf ? i - f : -1;
    }
    if (i == 0) w.status[0] = w.status[1] = ST_OK;
}

// one tile: phase 1 (k < t1) rows s0 .. s0+31, columns c0 .. c0+63 -> sm[i * RS_PAD + j];
// phase 2 rows r0 .. r0+63 (r < rend), columns s0 .. s0+31 -> sm[j * 32 + i]
struct Tile {
    double v[RS_DEPTH * RS_SLOTS / RS_THREADS];
};
__device__ __forceinline__ void rs_load(Tile& t, const double* W, int64_t C, int s0, int f, int t1, int rend, int k) {
#pragma unroll
    for (int e = 0; e < RS_DEPTH * RS_SLOTS / RS_THREADS; ++e) {
        const int idx = e * RS_THREADS + threadIdx.x;
        double v = 0.0;
        if (k < t1) {
            const int i = idx / RS_DEPTH, j = idx % RS_DEPTH, c = s0 + k * RS_DEPTH + j;
            if (s0 + i < C && c < C) v = __ldcg(W + (int64_t)(s0 + i) * C + c);
        } else {
            const int j = idx / RS_SLOTS, i = idx % RS_SLOTS, r = f + (k - t1) * RS_DEPTH + j;
            if (r < rend && s0 + i < C) v = __ldcg(W + (int64_t)r * C + s0 + i);
        }
        t.v[e] = v;
    }
}
__device__ __forceinline__ void rs_store(const Tile& t, double* sm, int t1, int k) {
#pragma unroll
    for (int e = 0; e < RS_DEPTH * RS_SLOTS / RS_THREADS; ++e) {
        const int idx = e * RS_THREADS + threadIdx.x;
        if (k < t1)
            sm[(idx / RS_DEPTH) * RS_PAD + idx % RS_DEPTH] = t.v[e];
        else
            sm[idx] = t.v[e];
    }
}

__global__ void __launch_bounds__(RS_THREADS) nj_rowsum_kernel(const double* __restrict__ W, int64_t C, int f, Work w) {
    if (__ldcg(w.status)) return;
    __shared__ double sm[2][RS_SLOTS * RS_PAD];
    const int s0 = (f / RS_SLOTS + blockIdx.x) * RS_SLOTS;  // aligned block of 32 slots meeting [f, C)
    const int lane = threadIdx.x;                           // warp 0: lane i sums slot s0 + i
    const int s = s0 + (lane & 31);
    const int t1 = (int)((C - s0 + RS_DEPTH - 1) / RS_DEPTH);  // row tiles: columns s0 .. C
    const int rend = (int)(s0 + RS_SLOTS < C ? s0 + RS_SLOTS : C);  // column tiles: rows f .. s0 + 31
    const int t2 = (rend - f + RS_DEPTH - 1) / RS_DEPTH;
    double acc = 0.0;
    Tile t;
    rs_load(t, W, C, s0, f, t1, rend, 0);
    for (int k = 0; k < t1 + t2; ++k) {
        double* b = sm[k & 1];
        rs_store(t, b, t1, k);
        __syncthreads();
        if (k + 1 < t1 + t2) rs_load(t, W, C, s0, f, t1, rend, k + 1);
        if (threadIdx.x < 32) {
            if (k < t1) {  // the members after s: W[s][c], c > s
                const int c0 = s0 + k * RS_DEPTH;
                const double* row = b + lane * RS_PAD;
#pragma unroll 16
                for (int j = 0; j < RS_DEPTH; ++j)
                    if (c0 + j > s) acc = __dadd_rn(acc, row[j]);
            } else {  // the members before s: W[r][s], f <= r < s
                const int r0 = f + (k - t1) * RS_DEPTH;
#pragma unroll 16
                for (int j = 0; j < RS_DEPTH; ++j)
                    if (r0 + j < s) acc = __dadd_rn(acc, b[j * RS_SLOTS + lane]);
            }
        }
        // the next iteration stores into the other buffer, which warp 0 finished before this __syncthreads
    }
    if (threadIdx.x < 32 && s >= f && s < C) w.S[s] = __ldcg(w.alive + s) ? acc : __longlong_as_double(0x7ff8000000000000ll);
}

__device__ __forceinline__ void take_min(double& v, long long& k, double v2, long long k2) {
    if (v2 < v || (v2 == v && k2 < k)) {
        v = v2;
        k = k2;
    }
}
__device__ __forceinline__ void warp_min(double& v, long long& k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double v2 = __shfl_xor_sync(0xFFFFFFFFu, v, o);
        const long long k2 = __shfl_xor_sync(0xFFFFFFFFu, k, o);
        take_min(v, k, v2, k2);
    }
}

// Q(r, c) = ((m - 2) W[r][c] - S_r) - S_c over r < c, taken only below 1e50 (NaN never is)
__global__ void __launch_bounds__(QS_THREADS) nj_qscan_kernel(const double* __restrict__ W, int64_t C, int f, int m, Work w) {
    if (__ldcg(w.status)) return;
    __shared__ double sv[QS_THREADS / 32];
    __shared__ long long sk[QS_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nw = gridDim.x * (QS_THREADS / 32);
    const double mm2 = (double)(m - 2);
    double bv = INFINITY;
    long long bk = NO_KEY;
    for (int r = f + blockIdx.x * (QS_THREADS / 32) + warp; r < C - 1; r += nw) {
        const double sr = __ldcg(w.S + r);
        if (isnan(sr)) continue;  // dead row
        const double* row = W + (int64_t)r * C;
        for (int c = r + 1 + lane; c < C; c += 32) {
            const double q = __dsub_rn(__dsub_rn(__dmul_rn(mm2, __ldcg(row + c)), sr), __ldcg(w.S + c));
            if (q < Q_BOUND) take_min(bv, bk, q, ((long long)r << 32) | c);
        }
    }
    warp_min(bv, bk);
    if (lane == 0) {
        sv[warp] = bv;
        sk[warp] = bk;
    }
    __syncthreads();
    if (warp == 0) {
        bv = lane < QS_THREADS / 32 ? sv[lane] : INFINITY;
        bk = lane < QS_THREADS / 32 ? sk[lane] : NO_KEY;
        warp_min(bv, bk);
        if (lane == 0) {
            w.pq[blockIdx.x] = bv;
            w.pk[blockIdx.x] = bk;
        }
    }
}

// the join's decision: pair, branch lengths, edges, BIONJ's lambda, the record; marks a and b dead and u live
__global__ void __launch_bounds__(FIN_THREADS) nj_finish_kernel(const double* __restrict__ W, int64_t C, int f, int m, int t,
                                                                 int n, int method, int nq, Work w, int64_t* edge, double* length) {
    if (__ldcg(w.status)) return;
    __shared__ double sv[32];
    __shared__ long long sk[32];
    __shared__ double chunk[2][LAM_CHUNK];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double bv = INFINITY;
    long long bk = NO_KEY;
    for (int g = threadIdx.x; g < nq; g += FIN_THREADS) take_min(bv, bk, __ldcg(w.pq + g), __ldcg(w.pk + g));
    warp_min(bv, bk);
    if (lane == 0) {
        sv[warp] = bv;
        sk[warp] = bk;
    }
    __syncthreads();
    bv = lane < FIN_THREADS / 32 ? sv[lane] : INFINITY;
    bk = lane < FIN_THREADS / 32 ? sk[lane] : NO_KEY;
    warp_min(bv, bk);  // every warp reduces the warp minima
    if (bk == NO_KEY) {
        if (threadIdx.x == 0) {
            w.status[0] = ST_NO_PAIR;
            w.status[1] = t;
        }
        return;
    }
    const int a = (int)(bk >> 32), b = (int)(bk & 0xFFFFFFFFll);
    const double A = __ldcg(W + (int64_t)a * C + b);
    const double Sa = __ldcg(w.S + a), Sb = __ldcg(w.S + b);
    const double B = __ddiv_rn(__dsub_rn(Sa, Sb), (double)(m - 2));
    const double la = half(__dadd_rn(A, B)), lb = half(__dsub_rn(A, B));
    double lam = 0.5, vab = 0.0;
    if (method == NJ_BIONJ) {
        vab = __ldcg(W + (int64_t)b * C + a);
        if (vab != 0.0) {
            // sum over the other members in list order of V_bk - V_ak: the differences are staged in shared
            // memory, thread 0 adds them in order (dead slots and a, b stage +0.0)
            double sum = 0.0;
            const int span = (int)(C - f);
            const int chunks = (span + LAM_CHUNK - 1) / LAM_CHUNK;
            for (int ch = 0; ch < chunks; ++ch) {
                double* buf = chunk[ch & 1];
                for (int j = threadIdx.x; j < LAM_CHUNK; j += FIN_THREADS) {
                    const int k = f + ch * LAM_CHUNK + j;
                    double d = 0.0;
                    if (k < C && k != a && k != b && __ldcg(w.alive + k)) d = __dsub_rn(lo(W, C, b, k), lo(W, C, a, k));
                    buf[j] = d;
                }
                __syncthreads();
                if (threadIdx.x == 0) {
                    const int len = min(LAM_CHUNK, span - ch * LAM_CHUNK);
#pragma unroll 8
                    for (int j = 0; j < len; ++j) sum = __dadd_rn(sum, buf[j]);
                }
            }
            lam = __dadd_rn(0.5, __ddiv_rn(sum, __dmul_rn((double)(2 * (m - 2)), vab)));
            if (lam < 0.0) lam = 0.0;
            if (lam > 1.0) lam = 1.0;
        }
    }
    if (threadIdx.x == 0) {
        const int u = f - 1, id = 2 * n - 3 - t;
        edge[4 * t + 0] = id;
        edge[4 * t + 1] = __ldcg(w.node + a);
        edge[4 * t + 2] = id;
        edge[4 * t + 3] = __ldcg(w.node + b);
        length[2 * t] = la;
        length[2 * t + 1] = lb;
        Rec* r = w.rec;
        r->a = a;
        r->b = b;
        r->u = u;
        r->A = A;
        r->la = la;
        r->lb = lb;
        r->lam = lam;
        r->vab = vab;
        w.alive[a] = w.alive[b] = 0;
        w.alive[u] = 1;
        w.node[u] = id;
    }
}

// row u over the old span [f, C): d(u, k) for live k, 0 elsewhere; BIONJ: V(u, k) into column u; the upper entries
// of a and b become 0
__global__ void nj_update_kernel(double* __restrict__ W, int64_t C, int f, int method, Work w) {
    if (__ldcg(w.status)) return;
    const Rec r = *w.rec;
    for (int k = f + blockIdx.x * blockDim.x + threadIdx.x; k < C; k += gridDim.x * blockDim.x) {
        double du = 0.0;
        const bool live = __ldcg(w.alive + k);  // a and b are already dead
        if (live) {
            const double dak = up(W, C, r.a, k), dbk = up(W, C, r.b, k);
            if (method == NJ_NJ) {
                du = half(__dsub_rn(__dadd_rn(dak, dbk), r.A));
            } else {
                const double oml = __dsub_rn(1.0, r.lam);
                du = __dadd_rn(__dmul_rn(r.lam, __dsub_rn(dak, r.la)), __dmul_rn(oml, __dsub_rn(dbk, r.lb)));
                const double vak = lo(W, C, r.a, k), vbk = lo(W, C, r.b, k);
                const double vu = __dsub_rn(__dadd_rn(__dmul_rn(r.lam, vak), __dmul_rn(oml, vbk)), __dmul_rn(__dmul_rn(r.lam, oml), r.vab));
                W[(int64_t)k * C + r.u] = vu;
            }
        }
        W[(int64_t)r.u * C + k] = du;
        if (k != r.a) W[(int64_t)min(r.a, k) * C + max(r.a, k)] = 0.0;
        if (k != r.b) W[(int64_t)min(r.b, k) * C + max(r.b, k)] = 0.0;
    }
}

// the three root edges from the members x < y < z left in [f, C)
__global__ void nj_root_kernel(const double* __restrict__ W, int64_t C, int f, int n, int t, Work w, int64_t* edge, double* length) {
    if (threadIdx.x != 0 || __ldcg(w.status)) return;
    int s[3], j = 0;
    for (int k = f; k < C && j < 3; ++k)
        if (__ldcg(w.alive + k)) s[j++] = k;
    if (j < 3) {
        w.status[0] = ST_NO_PAIR;
        w.status[1] = t;
        return;
    }
    const double dxy = __ldcg(W + (int64_t)s[0] * C + s[1]), dxz = __ldcg(W + (int64_t)s[0] * C + s[2]),
                 dyz = __ldcg(W + (int64_t)s[1] * C + s[2]);
    const double l[3] = {half(__dsub_rn(__dadd_rn(dxy, dxz), dyz)), half(__dsub_rn(__dadd_rn(dxy, dyz), dxz)),
                         half(__dsub_rn(__dadd_rn(dyz, dxz), dxy))};
    for (int i = 0; i < 3; ++i) {
        edge[4 * t + 2 * i] = n;
        edge[4 * t + 2 * i + 1] = __ldcg(w.node + s[i]);
        length[2 * t + i] = l[i];
    }
}

// compaction, step 1 (one CTA): live[] = the live slots of [f, C) in order; node[] and alive[] move to [C - m, C).
// node[] of the new slots is staged in `stage` (at least m ints) first, since old and new ranges overlap.
__global__ void nj_live_kernel(int64_t C, int f, int m, Work w, int* stage) {
    if (__ldcg(w.status)) return;
    __shared__ int wsum[32];
    __shared__ int base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    for (int k0 = f; k0 < C; k0 += blockDim.x) {
        const int k = k0 + threadIdx.x;
        const bool on = k < C && w.alive[k];
        const unsigned bal = __ballot_sync(0xFFFFFFFFu, on);
        if (lane == 0) wsum[warp] = __popc(bal);
        __syncthreads();
        int before = base;
        for (int i = 0; i < warp; ++i) before += wsum[i];
        before += __popc(bal & ((1u << lane) - 1u));
        if (on) {
            w.live[before] = k;
            stage[before] = w.node[k];
        }
        __syncthreads();
        if (threadIdx.x == 0)
            for (int i = 0; i < (int)(blockDim.x >> 5); ++i) base += wsum[i];
        __syncthreads();
    }
    for (int k = f + threadIdx.x; k < C; k += blockDim.x) {
        const int i = k - (int)(C - m);
        w.alive[k] = i >= 0 ? 1 : 0;
        w.node[k] = i >= 0 ? stage[i] : -1;
    }
}

// compaction, step 2: new rows x0 .. x0 + rows - 1 (counted from C - m) gathered from their old slots into the stage
__global__ void nj_gather_kernel(const double* __restrict__ W, int64_t C, int m, int x0, int rows, const int* live, double* stage) {
    for (int j = blockIdx.x; j < rows; j += gridDim.x) {
        const double* src = W + (int64_t)live[x0 + j] * C;
        double* dst = stage + (int64_t)j * m;
        for (int y = threadIdx.x; y < m; y += blockDim.x) dst[y] = __ldcg(src + live[y]);
    }
}
// compaction, step 3: the stage into the new rows
__global__ void nj_scatter_kernel(double* __restrict__ W, int64_t C, int m, int x0, int rows, const double* stage) {
    for (int j = blockIdx.x; j < rows; j += gridDim.x) {
        double* dst = W + (int64_t)(C - m + x0 + j) * C + (C - m);
        const double* src = stage + (int64_t)j * m;
        for (int y = threadIdx.x; y < m; y += blockDim.x) dst[y] = src[y];
    }
}

int sm_count() {
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
        return 148;
    return sms;
}

}  // namespace

}  // namespace po

using namespace po;

extern "C" {

int64_t po_nj_workspace(int64_t n) { return n < 3 ? -1 : workspace_bytes(n); }
int64_t po_nj_capacity(int64_t n) { return n < 3 ? -1 : capacity(n); }
int64_t po_nj_stage_bytes(int64_t n) { return n < 3 ? -1 : stage_rows(n) * n * 8; }

int po_nj_run(const void* d_D, int64_t ld, int dtype, int64_t n, int method, double* d_W, void* d_stage, void* d_work,
              int64_t* d_edge, double* d_length, int64_t* h_compactions, po_stream_t stream) {
    if (!d_D || !d_W || !d_stage || !d_work || !d_edge || !d_length || n < 3 || capacity(n) > INT_MAX / 2 || ld < n ||
        (dtype != PO_F32 && dtype != PO_F64) || (method != NJ_NJ && method != NJ_BIONJ)) {
        set_error("po_nj_run: bad arguments (n = %lld, method = %d)", (long long)n, method);
        return PO_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t C = capacity(n);
    Work w = carve(d_work, C);
    int f = (int)(C - n);
    const int sms = sm_count();
    const int nq = std::min(QS_MAX_CTAS, 4 * sms);
    const int64_t srows = stage_rows(n);
    long long compactions = 0;
    {
        LaunchTimer tm(3, st);  // po_timing_read(3): the copy, every join and the root edges
        const unsigned cb = (unsigned)std::min<int64_t>(n, 65535);
        if (dtype == PO_F32)
            nj_copy_kernel<float><<<cb, 256, 0, st>>>((const float*)d_D, ld, (int)n, d_W, C, f);
        else
            nj_copy_kernel<double><<<cb, 256, 0, st>>>((const double*)d_D, ld, (int)n, d_W, C, f);
        count_launch(3);
        nj_init_kernel<<<(unsigned)((C + 255) / 256), 256, 0, st>>>((int)n, C, f, w);
        count_launch(3);
        PO_LAUNCH_CHECK("nj_copy_kernel / nj_init_kernel");
        int t = 0;
        for (int m = (int)n; m > 3; --m, ++t) {  // n - 3 joins
            const int holes = (int)(C - f) - m;
            if (f == 0 || holes >= std::max(64, m / 8)) {
                nj_live_kernel<<<1, 1024, 0, st>>>(C, f, m, w, (int*)d_stage);
                count_launch(3);
                // descending: new row C - m + x is old row live[x'] only for x' >= x, so a batch overwrites rows
                // that this batch or an earlier one has already gathered
                for (int x1 = m; x1 > 0; x1 -= (int)srows) {
                    const int x0 = (int)std::max<int64_t>(0, x1 - srows), rows = x1 - x0;
                    const unsigned g = (unsigned)std::min(rows, 8 * sms);
                    nj_gather_kernel<<<g, 256, 0, st>>>(d_W, C, m, x0, rows, w.live, (double*)d_stage);
                    nj_scatter_kernel<<<g, 256, 0, st>>>(d_W, C, m, x0, rows, (const double*)d_stage);
                    count_launch(3);
                    count_launch(3);
                }
                f = (int)(C - m);
                ++compactions;
            }
            const unsigned rb = (unsigned)((C - f / RS_SLOTS * RS_SLOTS + RS_SLOTS - 1) / RS_SLOTS);
            nj_rowsum_kernel<<<rb, RS_THREADS, 0, st>>>(d_W, C, f, w);
            nj_qscan_kernel<<<nq, QS_THREADS, 0, st>>>(d_W, C, f, m, w);
            nj_finish_kernel<<<1, FIN_THREADS, 0, st>>>(d_W, C, f, m, t, (int)n, method, nq, w, d_edge, d_length);
            const unsigned ub = (unsigned)std::min<int64_t>((C - f + 255) / 256, 4 * sms);
            nj_update_kernel<<<ub, 256, 0, st>>>(d_W, C, f, method, w);
            for (int i = 0; i < 4; ++i) count_launch(3);
            PO_LAUNCH_CHECK("nj join kernels");
            --f;
        }
        nj_root_kernel<<<1, 32, 0, st>>>(d_W, C, f, (int)n, t, w, d_edge, d_length);
        count_launch(3);
        PO_LAUNCH_CHECK("nj_root_kernel");
    }
    int status[2];
    PO_CUDA_CHECK(cudaMemcpyAsync(status, w.status, sizeof(status), cudaMemcpyDeviceToHost, st));
    PO_CUDA_CHECK(cudaStreamSynchronize(st));
    if (h_compactions) *h_compactions = compactions;
    if (status[0] == ST_NO_PAIR) {
        set_error("po_nj_run: no pair has Q below 1e50 at join %d", status[1]);
        return PO_ERR_ARG;
    }
    return PO_OK;
}

}  // extern "C"
