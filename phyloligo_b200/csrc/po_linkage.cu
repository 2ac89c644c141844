// phyloselect.R's hierarchical tree of the contigs (reference bin/phyloselect.R:22-35, hclust) on the resident
// N x N matrix: what scipy.cluster.hierarchy.linkage(squareform(D), method) returns, bit for bit.
//   complete / average / weighted / ward   scipy's nn_chain: a nearest-neighbour chain over a float64 working
//                                          copy of D, Lance-Williams updates of row y and column y per merge
//   single                                 scipy's mst_single_linkage: Prim from vertex 0, reading D in place
//   the stable sort by height and label    -> po_linkage_tree (host)
//
// The loop runs in one persistent cooperative launch.  Every CTA owns a contiguous slice of the columns; a scan
// takes the minimum of its slice of row x (smallest index on ties) into a per-CTA partial, and after one
// grid.sync() every CTA reduces all partials itself, so every CTA holds the same chain state and takes the same
// decision without a second barrier.  A merge rewrites row y and column y, so the matrix stays symmetric and
// every scan reads one contiguous row; the next scan reads what other CTAs wrote, so a merge ends with a barrier.
// Cluster sizes and Prim's best[] / merged[] of a column are written only by the CTA that owns the column.
#include <cooperative_groups.h>
#include <algorithm>
#include <climits>
#include <cmath>
#include <numeric>
#include <vector>
#include "po_common.cuh"

namespace cg = cooperative_groups;

namespace po {

namespace {

constexpr int LK_THREADS = 512;
constexpr int LK_MAX_CTAS = 1024;
constexpr int NONE = INT_MAX;

enum { LK_SINGLE = 0, LK_COMPLETE = 1, LK_AVERAGE = 2, LK_WEIGHTED = 3, LK_WARD = 4 };
enum { ST_OK = 0, ST_BOUND = 1, ST_NO_CANDIDATE = 2 };

// workspace: best double[n], chain int32[n], size int32[n] (Prim: merged flags), partials (double, int32) x 2
// buffers x LK_MAX_CTAS, status int32[2] (code, step), phase count int64
struct Work {
    double* best;
    int *chain, *size;
    double* pv;
    int* pi;
    int* status;
    long long* phases;
};
Work carve(void* d_work, int64_t n) {
    Work w;
    char* p = reinterpret_cast<char*>(d_work);
    w.best = reinterpret_cast<double*>(p);
    w.pv = w.best + n;
    w.phases = reinterpret_cast<long long*>(w.pv + 2 * LK_MAX_CTAS);
    w.chain = reinterpret_cast<int*>(w.phases + 1);
    w.size = w.chain + n;
    w.pi = w.size + n;
    w.status = w.pi + 2 * LK_MAX_CTAS;
    return w;
}
int64_t workspace_bytes(int64_t n) { return n * 8 + 2 * LK_MAX_CTAS * 8 + 8 + 2 * n * 4 + 2 * LK_MAX_CTAS * 4 + 2 * 4; }

// (v, i) lexicographic minimum: the smallest value by IEEE <, the smallest index among equal values.  Values
// that a strict-< scan never takes (NaN, a +inf that nothing beats) never enter a partial.
__device__ __forceinline__ void take_min(double& v, int& i, double v2, int i2) {
    if (v2 < v || (v2 == v && i2 < i)) {
        v = v2;
        i = i2;
    }
}
__device__ __forceinline__ void warp_min(double& v, int& i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double v2 = __shfl_xor_sync(0xFFFFFFFFu, v, o);
        const int i2 = __shfl_xor_sync(0xFFFFFFFFu, i, o);
        take_min(v, i, v2, i2);
    }
}

struct Shared {
    double wv[LK_THREADS / 32];
    int wi[LK_THREADS / 32];
    double v;
    int i;
};

// the CTA's minimum into partial slot `slot`
__device__ void block_partial(double v, int i, Shared& s, double* pv, int* pi, int slot) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    warp_min(v, i);
    if (lane == 0) {
        s.wv[warp] = v;
        s.wi[warp] = i;
    }
    __syncthreads();
    if (warp == 0) {
        v = lane < LK_THREADS / 32 ? s.wv[lane] : INFINITY;
        i = lane < LK_THREADS / 32 ? s.wi[lane] : NONE;
        warp_min(v, i);
        if (lane == 0) {
            pv[slot] = v;
            pi[slot] = i;
        }
    }
}

// every CTA reduces the G partials of one buffer; the minimum is unique, so the order does not matter
__device__ void grid_min(const double* pv, const int* pi, int G, Shared& s, double& v, int& i) {
    if (threadIdx.x < 32) {
        double a = INFINITY;
        int b = NONE;
        for (int g = threadIdx.x; g < G; g += 32) take_min(a, b, __ldcg(pv + g), __ldcg(pi + g));
        warp_min(a, b);
        if (threadIdx.x == 0) {
            s.v = a;
            s.i = b;
        }
    }
    __syncthreads();
    v = s.v;
    i = s.i;
}

// scipy's _hierarchy_distance_update.pxi, each operation rounded on its own (no FMA contraction)
__device__ __forceinline__ double lance_williams(int method, double dxi, double dyi, double dxy, int nx, int ny, int ni) {
    switch (method) {
        case LK_COMPLETE:
            return dyi > dxi ? dyi : dxi;
        case LK_AVERAGE:
            return __ddiv_rn(__dadd_rn(__dmul_rn((double)nx, dxi), __dmul_rn((double)ny, dyi)), (double)(nx + ny));
        case LK_WEIGHTED:
            return __dmul_rn(0.5, __dadd_rn(dxi, dyi));
        default: {  // ward
            const double t = __ddiv_rn(1.0, (double)(nx + ny + ni));
            const double a = __dmul_rn(__dmul_rn(__dmul_rn((double)(ni + nx), t), dxi), dxi);
            const double b = __dmul_rn(__dmul_rn(__dmul_rn((double)(ni + ny), t), dyi), dyi);
            const double c = __dmul_rn(__dmul_rn(__dmul_rn((double)ni, t), dxy), dxy);
            return __dsqrt_rn(__dsub_rn(__dadd_rn(a, b), c));
        }
    }
}

template <typename T>
__global__ void copy_kernel(const T* __restrict__ D, int64_t ld, int n, double* __restrict__ W) {
    for (int r = blockIdx.x; r < n; r += gridDim.x) {
        const T* src = D + (int64_t)r * ld;
        double* dst = W + (int64_t)r * n;
        for (int c = threadIdx.x; c < n; c += blockDim.x) dst[c] = (double)src[c];
    }
}

__global__ void init_kernel(int n, Work w, int size0) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        w.best[i] = INFINITY;
        w.size[i] = size0;
    }
    if (i == 0) {
        w.status[0] = ST_OK;
        w.status[1] = 0;
        *w.phases = 0;
    }
}

struct Args {
    const void* D;  // Prim: the input; NN-chain: the float64 working copy (row stride n)
    int64_t ld;
    int n, method;
    Work w;
    int64_t *zx, *zy;
    double* zh;
};

// scipy's nn_chain.  Each loop turn: [owners apply the previous merge's size changes] scan row x -> partial,
// grid.sync, reduce, then either push y (no barrier: nothing was written that the next scan reads) or merge
// and grid.sync.
__global__ void __launch_bounds__(LK_THREADS, 1) nn_chain_kernel(Args a) {
    cg::grid_group grid = cg::this_grid();
    __shared__ Shared s;
    const int G = gridDim.x, n = a.n;
    const int c0 = (int)((int64_t)n * blockIdx.x / G), c1 = (int)((int64_t)n * (blockIdx.x + 1) / G);
    double* W = const_cast<double*>(reinterpret_cast<const double*>(a.D));
    const int64_t ld = a.ld;
    int* chain = a.w.chain;
    int* size = a.w.size;
    const bool lead = blockIdx.x == 0 && threadIdx.x == 0;
    const long long max_scans = 3ll * (n - 1);
    long long scans = 0, phases = 0;
    int len = 1, x = 0, y = 0, lo = 0, merges = 0, parity = 0;
    int dead = -1, grown = -1, grown_size = 0;  // the last merge, applied by the owners at the next loop turn
    int status = ST_OK;
    // chain[] holds the entries below the tip; the tip x lives in registers.  A slot is written only by a push
    // (the tip's slot and the new one) and read as prev (two below the new tip) or as the tip after a merge:
    // never a slot another CTA may still read in the same phase.
    while (true) {
        if (threadIdx.x == 0) {
            if (dead >= c0 && dead < c1) size[dead] = 0;
            if (grown >= c0 && grown < c1) size[grown] = grown_size;
        }
        dead = grown = -1;
        __syncthreads();
        double bv = INFINITY;
        int bi = NONE;
        const double* row = W + (int64_t)x * ld;
        for (int i = c0 + threadIdx.x; i < c1; i += LK_THREADS) {
            if (i == x || size[i] == 0) continue;
            const double v = __ldcg(row + i);
            if (v < bv) {
                bv = v;
                bi = i;
            }
        }
        block_partial(bv, bi, s, a.w.pv, a.w.pi, parity * LK_MAX_CTAS + blockIdx.x);
        ++scans;
        ++phases;
        grid.sync();
        double m;
        int j;
        grid_min(a.w.pv + parity * LK_MAX_CTAS, a.w.pi + parity * LK_MAX_CTAS, G, s, m, j);
        parity ^= 1;
        bool merge = false;
        double cur = m;
        if (len >= 2) {
            const int prev = __ldcg(chain + len - 2);
            const double dp = __ldcg(W + (int64_t)x * ld + prev);
            if (j != NONE && m < dp) {
                y = j;
            } else {  // d(x, prev) holds the minimum (or is NaN, which nothing beats): keep prev
                y = prev;
                cur = dp;
                merge = true;
            }
        } else if (j != NONE) {
            y = j;
        } else if (y == x || __ldcg(size + y) == 0) {
            // every candidate is NaN and scipy's stale y is unusable
            status = ST_NO_CANDIDATE;
            break;
        }  // else scipy pushes the y of the previous scan
        if (!merge) {
            if (len >= n || scans >= max_scans) {
                status = ST_BOUND;
                break;
            }
            if (lead) {
                chain[len - 1] = x;
                chain[len] = y;
            }
            ++len;
            x = y;
            continue;
        }
        len -= 2;
        const int p = min(x, y), q = max(x, y);
        y = q;  // scipy swaps x and y so that x < y; a later all-NaN scan pushes this stale y
        const int np_ = __ldcg(size + p), nq = __ldcg(size + q);
        if (lead) {
            a.zx[merges] = p;
            a.zy[merges] = q;
            a.zh[merges] = cur;
        }
        const double* rp = W + (int64_t)p * ld;
        double* rq = W + (int64_t)q * ld;
        for (int i = c0 + threadIdx.x; i < c1; i += LK_THREADS) {
            if (i == p || i == q) continue;
            const int ni = size[i];
            if (ni == 0) continue;
            const double v = lance_williams(a.method, __ldcg(rp + i), __ldcg(rq + i), cur, np_, nq, ni);
            rq[i] = v;
            W[(int64_t)i * ld + q] = v;
        }
        dead = p;
        grown = q;
        grown_size = np_ + nq;
        if (++merges == n - 1) break;
        if (len == 0) {  // the lowest-index active cluster; sizes of other slices are settled except p's
            while (lo == p || (lo != q && __ldcg(size + lo) == 0)) ++lo;
            x = lo;
            len = 1;
        } else {
            x = __ldcg(chain + len - 1);
        }
        ++phases;
        grid.sync();
    }
    if (lead) {
        a.w.status[0] = status;
        a.w.status[1] = merges;
        *a.w.phases = phases;
    }
}

// scipy's mst_single_linkage (Prim from vertex 0) on D in place: one scan and one barrier per step
template <typename T>
__global__ void __launch_bounds__(LK_THREADS, 1) prim_kernel(Args a) {
    cg::grid_group grid = cg::this_grid();
    __shared__ Shared s;
    const int G = gridDim.x, n = a.n;
    const int c0 = (int)((int64_t)n * blockIdx.x / G), c1 = (int)((int64_t)n * (blockIdx.x + 1) / G);
    const T* D = reinterpret_cast<const T*>(a.D);
    double* best = a.w.best;
    int* merged = a.w.size;
    const bool lead = blockIdx.x == 0 && threadIdx.x == 0;
    int x = 0, parity = 0, status = ST_OK, k = 0;
    for (; k < n - 1; ++k) {
        double bv = INFINITY;
        int bi = NONE;
        const T* row = D + (int64_t)x * a.ld;
        for (int i = c0 + threadIdx.x; i < c1; i += LK_THREADS) {  // column i is always this thread's
            if (merged[i]) continue;
            if (i == x) {
                merged[i] = 1;
                continue;
            }
            const double d = (double)__ldg(row + i);
            double b = best[i];
            if (b > d) {
                b = d;
                best[i] = b;
            }
            if (b < bv) {
                bv = b;
                bi = i;
            }
        }
        block_partial(bv, bi, s, a.w.pv, a.w.pi, parity * LK_MAX_CTAS + blockIdx.x);
        grid.sync();
        double cur;
        int y;
        grid_min(a.w.pv + parity * LK_MAX_CTAS, a.w.pi + parity * LK_MAX_CTAS, G, s, cur, y);
        parity ^= 1;
        if (y == NONE) {
            status = ST_NO_CANDIDATE;
            break;
        }
        if (lead) {
            a.zx[k] = x;
            a.zy[k] = y;
            a.zh[k] = cur;
        }
        x = y;
    }
    if (lead) {
        a.w.status[0] = status;
        a.w.status[1] = k;
        *a.w.phases = k;
    }
}

__global__ void __launch_bounds__(LK_THREADS, 1) barrier_kernel(int iters) {
    cg::grid_group grid = cg::this_grid();
    for (int k = 0; k < iters; ++k) grid.sync();
}

}  // namespace

// CTAs of the linkage launch: one per SM at most (the barrier's cost grows with the CTA count, and a slice of a
// 100 000-row matrix is already about one load per thread), fewer for small n; the occupancy API confirms that
// the kernel fits once per SM, which the cooperative launch needs for co-residency
int linkage_grid(const void* kernel, int64_t n, int* ctas) {
    int dev = 0, sms = 0, occ = 0, coop = 0;
    PO_CUDA_CHECK(cudaGetDevice(&dev));
    PO_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    PO_CUDA_CHECK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
    PO_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, LK_THREADS, 0));
    if (!coop || occ < 1) {
        set_error("linkage: the device cannot run a cooperative launch of %d threads per CTA", LK_THREADS);
        return PO_ERR_UNSUPPORTED;
    }
    const int64_t want = (n + LK_THREADS - 1) / LK_THREADS;
    *ctas = (int)std::max<int64_t>(1, std::min<int64_t>(std::min(sms, LK_MAX_CTAS), want));
    return PO_OK;
}

// microbench kind 4: microseconds per grid.sync() of the linkage kernels' largest grid (one CTA per SM)
int barrier_latency_us(double* result) {
    int G = 0;
    const int rc = linkage_grid((const void*)barrier_kernel, (int64_t)LK_THREADS * LK_MAX_CTAS, &G);
    if (rc != PO_OK) return rc;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    int iters = 20000;
    void* args[] = {&iters};
    double best = 1e30;
    cudaError_t e = cudaEventCreate(&e0);
    if (e == cudaSuccess) e = cudaEventCreate(&e1);
    for (int rep = 0; rep < 5 && e == cudaSuccess; ++rep) {
        float ms = 0.f;
        e = cudaEventRecord(e0, 0);
        if (e == cudaSuccess) e = cudaLaunchCooperativeKernel((const void*)barrier_kernel, dim3(G), dim3(LK_THREADS), args, 0, 0);
        if (e == cudaSuccess) e = cudaEventRecord(e1, 0);
        if (e == cudaSuccess) e = cudaEventSynchronize(e1);
        if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
        if (e == cudaSuccess && rep > 0) best = std::min(best, (double)ms * 1e3 / iters);
    }
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
    if (e != cudaSuccess) {
        set_error("po_microbench kind 4: %s", cudaGetErrorString(e));
        (void)cudaGetLastError();
        return PO_ERR_CUDA;
    }
    *result = best;
    return PO_OK;
}

}  // namespace po

using namespace po;

extern "C" {

int64_t po_linkage_workspace(int64_t n) { return n < 0 ? -1 : workspace_bytes(n); }

int po_linkage_run(const void* d_D, int64_t ld, int dtype, int64_t n, int method, double* d_W, void* d_work, int64_t* d_zx,
                   int64_t* d_zy, double* d_zh, int64_t* h_phases, po_stream_t stream) {
    if (!d_D || !d_work || !d_zx || !d_zy || !d_zh || n < 2 || n > INT_MAX || ld < n || (dtype != PO_F32 && dtype != PO_F64) ||
        method < LK_SINGLE || method > LK_WARD || (method != LK_SINGLE && !d_W)) {
        set_error("po_linkage_run: bad arguments (n = %lld, method = %d)", (long long)n, method);
        return PO_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    Work w = carve(d_work, n);
    Args a;
    a.ld = ld;
    a.n = (int)n;
    a.method = method;
    a.w = w;
    a.zx = d_zx;
    a.zy = d_zy;
    a.zh = d_zh;
    const void* kernel;
    if (method == LK_SINGLE) {
        a.D = d_D;
        kernel = dtype == PO_F32 ? (const void*)prim_kernel<float> : (const void*)prim_kernel<double>;
    } else {
        const unsigned blocks = (unsigned)std::min<int64_t>(n, 65535);
        if (dtype == PO_F32)
            copy_kernel<float><<<blocks, 256, 0, st>>>((const float*)d_D, ld, (int)n, d_W);
        else
            copy_kernel<double><<<blocks, 256, 0, st>>>((const double*)d_D, ld, (int)n, d_W);
        count_launch(2);
        PO_LAUNCH_CHECK("linkage copy_kernel");
        a.D = d_W;
        a.ld = n;
        kernel = (const void*)nn_chain_kernel;
    }
    init_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((int)n, w, method == LK_SINGLE ? 0 : 1);
    count_launch(2);
    PO_LAUNCH_CHECK("linkage init_kernel");
    int G = 0;
    const int rc = linkage_grid(kernel, n, &G);
    if (rc != PO_OK) return rc;
    void* args[] = {&a};
    {
        LaunchTimer tm(2, st);  // po_timing_read(2): the cooperative launch alone
        PO_CUDA_CHECK(cudaLaunchCooperativeKernel(kernel, dim3(G), dim3(LK_THREADS), args, 0, st));
    }
    count_launch(2);
    int status[2];
    long long phases = 0;
    PO_CUDA_CHECK(cudaMemcpyAsync(status, w.status, sizeof(status), cudaMemcpyDeviceToHost, st));
    PO_CUDA_CHECK(cudaMemcpyAsync(&phases, w.phases, sizeof(phases), cudaMemcpyDeviceToHost, st));
    PO_CUDA_CHECK(cudaStreamSynchronize(st));
    if (h_phases) *h_phases = phases;
    if (status[0] == ST_BOUND) {
        set_error("po_linkage_run: the nearest-neighbour chain passed its bound of 3 (n - 1) scans after %d merges", status[1]);
        return PO_ERR_CUDA;
    }
    if (status[0] == ST_NO_CANDIDATE) {
        set_error("po_linkage_run: every distance from the chain's tip is NaN after %d merges", status[1]);
        return PO_ERR_ARG;
    }
    if (status[1] != n - 1) {
        set_error("po_linkage_run: %d merges for %lld points", status[1], (long long)n);
        return PO_ERR_CUDA;
    }
    return PO_OK;
}

int po_linkage_tree(int64_t n, const int64_t* zx, const int64_t* zy, const double* zh, double* Z) {
    if (n < 2 || !zx || !zy || !zh || !Z) {
        set_error("po_linkage_tree: bad arguments (n = %lld)", (long long)n);
        return PO_ERR_ARG;
    }
    const int64_t m = n - 1;
    for (int64_t k = 0; k < m; ++k) {
        if (zx[k] < 0 || zx[k] >= n || zy[k] < 0 || zy[k] >= n || zx[k] == zy[k]) {
            set_error("po_linkage_tree: merge %lld = (%lld, %lld) is not a pair of %lld points", (long long)k, (long long)zx[k],
                      (long long)zy[k], (long long)n);
            return PO_ERR_ARG;
        }
    }
    // np.argsort(Z[:, 2], kind="mergesort"): stable, NaN last
    std::vector<int64_t> order(m);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int64_t a, int64_t b) {
        const double x = zh[a], y = zh[b];
        return !std::isnan(x) && (std::isnan(y) || x < y);
    });
    // scipy's label: union-find over the sorted rows, new clusters n, n + 1, ...
    std::vector<int64_t> parent(2 * n - 1), size(2 * n - 1, 1);
    std::iota(parent.begin(), parent.end(), 0);
    auto find = [&](int64_t x) {
        int64_t r = x;
        while (parent[r] != r) r = parent[r];
        while (parent[x] != r) {
            const int64_t nx = parent[x];
            parent[x] = r;
            x = nx;
        }
        return r;
    };
    for (int64_t k = 0; k < m; ++k) {
        const int64_t r = order[k];
        int64_t a = find(zx[r]), b = find(zy[r]);
        if (a == b) {
            set_error("po_linkage_tree: merge %lld joins a cluster with itself", (long long)r);
            return PO_ERR_ARG;
        }
        if (a > b) std::swap(a, b);
        parent[a] = parent[b] = n + k;
        size[n + k] = size[a] + size[b];
        Z[4 * k + 0] = (double)a;
        Z[4 * k + 1] = (double)b;
        Z[4 * k + 2] = zh[r];
        Z[4 * k + 3] = (double)size[n + k];
    }
    return PO_OK;
}

}  // extern "C"
