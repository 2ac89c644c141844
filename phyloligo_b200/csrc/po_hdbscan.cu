// phyloselect's HDBSCAN on the resident N x N matrix (reference bin/phyloselect.py:403-428, which calls
// hdbscan.HDBSCAN(min_cluster_size, min_samples, metric="precomputed") with every other argument at its
// default).  Replaces, in scikit-learn-contrib/hdbscan:
//   mutual_reachability + mst_linkage_core   the float64 N x N copy and the O(N^2) Prim loop on one core
//                                            -> po_hdbscan_check, po_matrix_kth (po_select.cu: core
//                                               distances), po_hdbscan_mst_init / po_hdbscan_mst_scan /
//                                               po_hdbscan_mst_merge (Boruvka; mutual reachability computed
//                                               on the fly, the matrix read whole or in row panels)
//   label, condense_tree, compute_stability,
//   get_clusters, get_probabilities          -> po_hdbscan_tree (host, O(N log N))
//
// Tie rule: edges compare by (mr, min(i, j), max(i, j)).  It is a strict total order on the edges, so the
// MST is unique and Boruvka's per-component lightest edges never close a cycle.
#include <algorithm>
#include <cmath>
#include <limits>
#include <numeric>
#include <vector>
#include "po_common.cuh"

namespace po {

namespace {

// ---------------------------------------------------------------------------------------------------
// input check: square (the caller), finite and bitwise symmetric; the smallest row-major index
// min(i, j) * n + max(i, j) of an offending pair, or i * n + j of a non-finite entry, goes to *first_bad
// ---------------------------------------------------------------------------------------------------
template <typename T> struct Bits;
template <> struct Bits<float> { using type = unsigned; };
template <> struct Bits<double> { using type = unsigned long long; };

constexpr int CHK = 32;

template <typename T>
__global__ void __launch_bounds__(256) check_kernel(const void* __restrict__ D, int64_t ld, int64_t n,
                                                    unsigned long long* __restrict__ first_bad) {
    using B = typename Bits<T>::type;
    const int64_t bi = blockIdx.y, bj = blockIdx.x;
    if (bi > bj) return;  // every pair of tiles once: (bi, bj) with its mirror (bj, bi)
    __shared__ B a[CHK][CHK + 1], b[CHK][CHK + 1];
    const B* M = reinterpret_cast<const B*>(D);
    const int c = threadIdx.x & 31;
    unsigned long long bad = ~0ull;
    for (int r = threadIdx.x >> 5; r < CHK; r += 8) {
        const int64_t i = bi * CHK + r, j = bj * CHK + c;  // tile (bi, bj)
        const int64_t i2 = bj * CHK + r, j2 = bi * CHK + c;  // tile (bj, bi)
        a[r][c] = (i < n && j < n) ? M[i * ld + j] : (B)0;
        b[r][c] = (i2 < n && j2 < n) ? M[i2 * ld + j2] : (B)0;
    }
    __syncthreads();
    for (int r = threadIdx.x >> 5; r < CHK; r += 8) {
        const int64_t i = bi * CHK + r, j = bj * CHK + c;
        if (i < n && j < n) {
            const T x = reinterpret_cast<const T&>(a[r][c]);
            if (!isfinite(x)) bad = min(bad, (unsigned long long)(i * n + j));
            if (a[r][c] != b[c][r]) bad = min(bad, (unsigned long long)(min(i, j) * n + max(i, j)));
        }
        const int64_t i2 = bj * CHK + r, j2 = bi * CHK + c;
        if (bi != bj && i2 < n && j2 < n && !isfinite(reinterpret_cast<const T&>(b[r][c])))
            bad = min(bad, (unsigned long long)(i2 * n + j2));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) bad = min(bad, __shfl_xor_sync(0xFFFFFFFFu, bad, o));
    if ((threadIdx.x & 31) == 0 && bad != ~0ull) atomicMin(first_bad, bad);
}

// The same test on the row panel [row0, row0 + rows) x [0, n): entry (i, j) against (j, i), read from the column
// strip S ([0, n) x [row0, row0 + rows), pitch lds) or, without a strip, from the panel itself when j lies in the
// panel's rows (a source symmetric by construction is tested on its diagonal square only).  Keys are absolute.
template <typename T>
__global__ void __launch_bounds__(256) panel_check_kernel(const void* __restrict__ D, int64_t ld, int64_t rows, int64_t n,
                                                          int64_t row0, const void* __restrict__ S, int64_t lds,
                                                          unsigned long long* __restrict__ first_bad) {
    using B = typename Bits<T>::type;
    const int64_t bi = blockIdx.y, bj = blockIdx.x;
    __shared__ B a[CHK][CHK + 1], b[CHK][CHK + 1];
    __shared__ bool has[CHK][CHK + 1];
    const B* M = reinterpret_cast<const B*>(D);
    const B* ST = reinterpret_cast<const B*>(S);
    const int c = threadIdx.x & 31;
    unsigned long long bad = ~0ull;
    for (int r = threadIdx.x >> 5; r < CHK; r += 8) {
        const int64_t li = bi * CHK + r, j = bj * CHK + c;     // entry (row0 + li, j)
        const int64_t tj = bj * CHK + r, tli = bi * CHK + c;   // entry (tj, row0 + tli)
        a[r][c] = (li < rows && j < n) ? M[li * ld + j] : (B)0;
        bool h = tj < n && tli < rows;
        B v = (B)0;
        if (h && S) v = ST[tj * lds + tli];
        else if (h && tj >= row0 && tj < row0 + rows) v = M[(tj - row0) * ld + row0 + tli];
        else h = false;
        b[r][c] = v;
        has[r][c] = h;
    }
    __syncthreads();
    for (int r = threadIdx.x >> 5; r < CHK; r += 8) {
        const int64_t li = bi * CHK + r, j = bj * CHK + c, i = row0 + li;
        if (li < rows && j < n) {
            if (!isfinite(reinterpret_cast<const T&>(a[r][c]))) bad = min(bad, (unsigned long long)(i * n + j));
            if (has[c][r] && a[r][c] != b[c][r]) bad = min(bad, (unsigned long long)(min(i, j) * n + max(i, j)));
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) bad = min(bad, __shfl_xor_sync(0xFFFFFFFFu, bad, o));
    if ((threadIdx.x & 31) == 0 && bad != ~0ull) atomicMin(first_bad, bad);
}

// ---------------------------------------------------------------------------------------------------
// Boruvka over the mutual-reachability graph
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long wkey(double v) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(v + 0.0);  // -0 and +0 compare equal
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
template <typename T>
__device__ __forceinline__ T mr(T core_i, T core_j, T d) {
    const T c = core_i > core_j ? core_i : core_j;
    return c > d ? c : d;
}

// workspace (all n entries): row_key, comp_key, comp_edge uint64; row_d float64 (D[i, row_j[i]], so that the
// merge needs no access to the matrix); comp, P, P2, row_j int32; then two int32 counters (edges found so far,
// components)
struct Work {
    int *comp, *P, *P2, *row_j;
    unsigned long long *row_key, *comp_key, *comp_edge;
    double* row_d;
    int* counters;
};
Work carve(void* d_work, int64_t n) {
    Work w;
    char* p = reinterpret_cast<char*>(d_work);
    w.row_key = reinterpret_cast<unsigned long long*>(p);
    w.comp_key = w.row_key + n;
    w.comp_edge = w.comp_key + n;
    w.row_d = reinterpret_cast<double*>(w.comp_edge + n);
    int* q = reinterpret_cast<int*>(w.row_d + n);
    w.comp = q;
    w.P = q + n;
    w.P2 = q + 2 * n;
    w.row_j = q + 3 * n;
    w.counters = q + 4 * n;
    return w;
}

constexpr int RM_THREADS = 256;
constexpr int RM_ROWS = 8;    // rows per CTA: the column's core distance and component are loaded once for all of them
constexpr int RM_UNROLL = 4;  // columns per thread per step: RM_ROWS x RM_UNROLL loads in flight

// For every row i of the panel [row0, row0 + n_rows) (D points at its first row), its lightest edge (mr(i, j), j)
// to a column of another component.  For a fixed row the tie rule's (min(i, j), max(i, j)) orders the columns as
// j does, so the per-row minimum is taken over (mr, j).
template <typename T>
__global__ void __launch_bounds__(RM_THREADS) rowmin_kernel(const void* __restrict__ D, int64_t ld, int row0, int n_rows, int n,
                                                            const T* __restrict__ core, const int* __restrict__ comp,
                                                            unsigned long long* __restrict__ row_key, int* __restrict__ row_j,
                                                            double* __restrict__ row_d) {
    const int l0 = blockIdx.x * RM_ROWS;  // first panel row of this CTA
    const int r0 = row0 + l0;             // its matrix row
    const T* base = reinterpret_cast<const T*>(D) + (int64_t)l0 * ld;
    T ci[RM_ROWS], bw[RM_ROWS], bd[RM_ROWS];
    int cc[RM_ROWS], bj[RM_ROWS];
#pragma unroll
    for (int r = 0; r < RM_ROWS; ++r) {
        const bool ok = l0 + r < n_rows;
        ci[r] = ok ? core[r0 + r] : (T)0;
        cc[r] = ok ? comp[r0 + r] : -1;
        bw[r] = (T)__longlong_as_double(0x7FF0000000000000ll);  // +inf
        bd[r] = (T)0;
        bj[r] = -1;
    }
    const int rows = min(RM_ROWS, n_rows - l0);
    // rows past the end re-read the last row (never written back): no branch between the loads, so all
    // RM_ROWS x RM_UNROLL of them are in flight together
    int64_t roff[RM_ROWS];
#pragma unroll
    for (int r = 0; r < RM_ROWS; ++r) roff[r] = (int64_t)min(r, rows - 1) * ld;
    for (int j0 = threadIdx.x; j0 < n; j0 += RM_THREADS * RM_UNROLL) {
        T cj[RM_UNROLL], d[RM_ROWS][RM_UNROLL];
        int gj[RM_UNROLL];
#pragma unroll
        for (int u = 0; u < RM_UNROLL; ++u) {
            const int j = min(j0 + u * RM_THREADS, n - 1);
#pragma unroll
            for (int r = 0; r < RM_ROWS; ++r) d[r][u] = __ldcs(base + roff[r] + j);
            cj[u] = __ldg(core + j);
            gj[u] = j0 + u * RM_THREADS < n ? __ldg(comp + j) : -2;
        }
#pragma unroll
        for (int r = 0; r < RM_ROWS; ++r) {
#pragma unroll
            for (int u = 0; u < RM_UNROLL; ++u) {
                const T w = mr(ci[r], cj[u], d[r][u]);
                // columns are visited in increasing order by each thread: strict < keeps the first on ties
                if (gj[u] >= 0 && gj[u] != cc[r] && w < bw[r]) {
                    bw[r] = w;
                    bd[r] = d[r][u];
                    bj[r] = j0 + u * RM_THREADS;
                }
            }
        }
    }
    __shared__ unsigned long long s_key[RM_THREADS / 32][RM_ROWS];
    __shared__ int s_j[RM_THREADS / 32][RM_ROWS];
    __shared__ double s_d[RM_THREADS / 32][RM_ROWS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int r = 0; r < RM_ROWS; ++r) {
        unsigned long long k = bj[r] >= 0 ? wkey((double)bw[r]) : ~0ull;
        int j = bj[r] >= 0 ? bj[r] : 0x7FFFFFFF;
        double dv = (double)bd[r];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long k2 = __shfl_xor_sync(0xFFFFFFFFu, k, o);
            const int j2 = __shfl_xor_sync(0xFFFFFFFFu, j, o);
            const double d2 = __shfl_xor_sync(0xFFFFFFFFu, dv, o);
            if (k2 < k || (k2 == k && j2 < j)) {
                k = k2;
                j = j2;
                dv = d2;
            }
        }
        if (lane == 0) {
            s_key[warp][r] = k;
            s_j[warp][r] = j;
            s_d[warp][r] = dv;
        }
    }
    __syncthreads();
    if (threadIdx.x < rows) {
        const int r = threadIdx.x;
        unsigned long long k = s_key[0][r];
        int j = s_j[0][r];
        double dv = s_d[0][r];
        for (int w = 1; w < RM_THREADS / 32; ++w) {
            if (s_key[w][r] < k || (s_key[w][r] == k && s_j[w][r] < j)) {
                k = s_key[w][r];
                j = s_j[w][r];
                dv = s_d[w][r];
            }
        }
        row_key[r0 + r] = k;
        row_j[r0 + r] = (k == ~0ull) ? -1 : j;
        row_d[r0 + r] = dv;
    }
}

// per component: the smallest weight key among its rows' edges, then the smallest (min, max) among the edges
// that have it
__global__ void comp_key_kernel(int n, const int* __restrict__ comp, const unsigned long long* __restrict__ row_key,
                                unsigned long long* __restrict__ comp_key) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && row_key[i] != ~0ull) atomicMin(&comp_key[comp[i]], row_key[i]);
}
__global__ void comp_edge_kernel(int n, const int* __restrict__ comp, const unsigned long long* __restrict__ row_key,
                                 const int* __restrict__ row_j, const unsigned long long* __restrict__ comp_key,
                                 unsigned long long* __restrict__ comp_edge) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || row_key[i] == ~0ull || row_key[i] != comp_key[comp[i]]) return;
    const int j = row_j[i];
    atomicMin(&comp_edge[comp[i]], ((unsigned long long)(unsigned)min(i, j) << 32) | (unsigned)max(i, j));
}

// hooking: every component (root c, comp[c] == c) points at the component across its lightest edge.  Two
// components that chose the same edge point at each other; the smaller id stays a root and the edge is
// emitted once, by the other.  Non-roots keep pointing at their root.  The edge (u, v) came from row u or row v,
// whose scan kept D[u, v] or D[v, u]: the same bits, the matrix having passed the symmetry check.
template <typename T>
__global__ void hook_kernel(int n, const T* __restrict__ core, const int* __restrict__ comp, const int* __restrict__ row_j,
                            const double* __restrict__ row_d, const unsigned long long* __restrict__ comp_edge, int* __restrict__ P,
                            int* __restrict__ counters, int64_t* __restrict__ out_u, int64_t* __restrict__ out_v,
                            T* __restrict__ out_w) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    if (comp[c] != c || comp_edge[c] == ~0ull) {
        P[c] = comp[c];
        return;
    }
    const unsigned long long e = comp_edge[c];
    const int u = (int)(e >> 32), v = (int)(e & 0xFFFFFFFFull);
    const int other = comp[u] == c ? comp[v] : comp[u];
    if (comp_edge[other] == e && c < other) {
        P[c] = c;
        return;
    }
    P[c] = other;
    const int pos = atomicAdd(&counters[0], 1);
    if (pos < n - 1) {
        out_u[pos] = u;
        out_v[pos] = v;
        out_w[pos] = mr(core[u], core[v], (T)(row_j[u] == v ? row_d[u] : row_d[v]));
    }
}

__global__ void jump_kernel(int n, const int* __restrict__ P, int* __restrict__ P2) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) P2[i] = P[P[i]];
}

__global__ void relabel_kernel(int n, const int* __restrict__ P, int* __restrict__ comp, int* __restrict__ counters) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    comp[i] = P[i];
    if (P[i] == i) atomicAdd(&counters[1], 1);
}

__global__ void init_kernel(int n, int* comp, int* counters) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) comp[i] = i;
    if (i == 0) {
        counters[0] = 0;
        counters[1] = n;
    }
}

// ---------------------------------------------------------------------------------------------------
// host stage
// ---------------------------------------------------------------------------------------------------
struct Edge {
    int64_t a, b;
    double w;
};

// breadth-first order of the single-linkage subtree under `root` (contrib's bfs_from_hierarchy)
void bfs(const std::vector<int64_t>& left, const std::vector<int64_t>& right, int64_t n, int64_t root, std::vector<int64_t>& out) {
    out.clear();
    out.push_back(root);
    for (size_t head = 0; head < out.size(); ++head) {
        const int64_t x = out[head];
        if (x >= n) {
            out.push_back(left[x - n]);
            out.push_back(right[x - n]);
        }
    }
    // contrib visits level by level; a FIFO over the nodes gives the same order
}

}  // namespace

}  // namespace po

using namespace po;

extern "C" {

int po_hdbscan_check(const void* d_D, int64_t ld, int dtype, int64_t n_rows, int64_t n_cols, int64_t row0, const void* d_cols,
                     int64_t ld_cols, void* d_work, po_stream_t stream) {
    if (!d_D || !d_work || n_rows < 0 || n_cols < 0 || ld < n_cols || (dtype != PO_F32 && dtype != PO_F64) || row0 < 0 ||
        ld_cols < 0 || (d_cols && ld_cols < n_rows) || (ld_cols == 0 && (d_cols || row0 != 0))) {
        set_error("po_hdbscan_check: bad arguments");
        return PO_ERR_ARG;
    }
    const bool whole = ld_cols == 0;
    if (whole ? n_rows != n_cols : row0 + n_rows > n_cols) {
        set_error("po_hdbscan_check: the matrix is not square (%lld x %lld)", (long long)(row0 + n_rows), (long long)n_cols);
        return PO_ERR_ARG;
    }
    const int64_t n = n_cols;
    if (n_rows == 0) return PO_OK;
    const int64_t nb = (n + CHK - 1) / CHK, rb = (n_rows + CHK - 1) / CHK;
    if (rb > 65535 || (whole && nb > 65535)) {
        set_error("po_hdbscan_check: %lld rows is more than this check supports", (long long)n_rows);
        return PO_ERR_UNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long* first = reinterpret_cast<unsigned long long*>(d_work);
    PO_CUDA_CHECK(cudaMemsetAsync(first, 0xFF, sizeof(unsigned long long), st));
    if (whole) {
        const dim3 grid((unsigned)nb, (unsigned)nb);
        if (dtype == PO_F32)
            check_kernel<float><<<grid, 256, 0, st>>>(d_D, ld, n, first);
        else
            check_kernel<double><<<grid, 256, 0, st>>>(d_D, ld, n, first);
    } else {
        const dim3 grid((unsigned)nb, (unsigned)rb);
        if (dtype == PO_F32)
            panel_check_kernel<float><<<grid, 256, 0, st>>>(d_D, ld, n_rows, n, row0, d_cols, ld_cols, first);
        else
            panel_check_kernel<double><<<grid, 256, 0, st>>>(d_D, ld, n_rows, n, row0, d_cols, ld_cols, first);
    }
    count_launch(2);
    PO_LAUNCH_CHECK("check_kernel");
    unsigned long long bad = 0;
    PO_CUDA_CHECK(cudaMemcpyAsync(&bad, first, sizeof(bad), cudaMemcpyDeviceToHost, st));
    PO_CUDA_CHECK(cudaStreamSynchronize(st));
    if (bad == ~0ull) return PO_OK;
    const int64_t i = (int64_t)(bad / (unsigned long long)n), j = (int64_t)(bad % (unsigned long long)n);
    const size_t es = dtype == PO_F32 ? 4 : 8;
    double x[2];
    for (int q = 0; q < 2; ++q) {
        const int64_t r = q ? j : i, c = q ? i : j;
        // entry (r, c): in the panel when r is one of its rows, else in the column strip.  Without a strip the source
        // is symmetric and a pair outside the diagonal square can only be named for a non-finite (i, j)
        if (q && !whole && !d_cols && !(r >= row0 && r < row0 + n_rows)) {
            x[1] = x[0];
            continue;
        }
        const char* src = (r >= row0 && r < row0 + n_rows)
                              ? reinterpret_cast<const char*>(d_D) + ((r - row0) * ld + c) * (int64_t)es
                              : reinterpret_cast<const char*>(d_cols) + (r * ld_cols + (c - row0)) * (int64_t)es;
        unsigned char raw[8];
        PO_CUDA_CHECK(cudaMemcpy(raw, src, es, cudaMemcpyDeviceToHost));
        if (dtype == PO_F32) {
            float f;
            memcpy(&f, raw, 4);
            x[q] = f;
        } else {
            memcpy(&x[q], raw, 8);
        }
    }
    if (std::isnan(x[0]))
        set_error("po_hdbscan_check: entry (%lld, %lld) is NaN", (long long)i, (long long)j);
    else if (std::isinf(x[0]))
        set_error("po_hdbscan_check: entry (%lld, %lld) is infinite (%g)", (long long)i, (long long)j, x[0]);
    else
        set_error("po_hdbscan_check: the matrix is not symmetric: entry (%lld, %lld) = %.17g, entry (%lld, %lld) = %.17g",
                  (long long)i, (long long)j, x[0], (long long)j, (long long)i, x[1]);
    return PO_ERR_ARG;
}

int64_t po_hdbscan_mst_workspace(int64_t n) { return n < 0 ? -1 : n * 4 * 8 + n * 4 * 4 + 2 * 4; }

int po_hdbscan_mst_init(int64_t n, void* d_work, po_stream_t stream) {
    if (!d_work || n < 1 || n > 0x7FFFFFFFll) {
        set_error("po_hdbscan_mst_init: bad arguments");
        return PO_ERR_ARG;
    }
    Work w = carve(d_work, n);
    init_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>((int)n, w.comp, w.counters);
    count_launch(2);
    PO_LAUNCH_CHECK("init_kernel");
    return PO_OK;
}

int po_hdbscan_mst_scan(const void* d_D, int64_t ld, int dtype, int64_t row0, int64_t n_rows, int64_t n, const void* d_core,
                        void* d_work, po_stream_t stream) {
    if (!d_D || !d_core || !d_work || n < 1 || n > 0x7FFFFFFFll || row0 < 0 || n_rows < 0 || row0 + n_rows > n || ld < n ||
        (dtype != PO_F32 && dtype != PO_F64)) {
        set_error("po_hdbscan_mst_scan: bad arguments");
        return PO_ERR_ARG;
    }
    if (n_rows == 0) return PO_OK;
    cudaStream_t st = (cudaStream_t)stream;
    Work w = carve(d_work, n);
    const unsigned grows = (unsigned)((n_rows + RM_ROWS - 1) / RM_ROWS);
    if (dtype == PO_F32)
        rowmin_kernel<float><<<grows, RM_THREADS, 0, st>>>(d_D, ld, (int)row0, (int)n_rows, (int)n, (const float*)d_core, w.comp,
                                                          w.row_key, w.row_j, w.row_d);
    else
        rowmin_kernel<double><<<grows, RM_THREADS, 0, st>>>(d_D, ld, (int)row0, (int)n_rows, (int)n, (const double*)d_core, w.comp,
                                                           w.row_key, w.row_j, w.row_d);
    count_launch(2);
    PO_LAUNCH_CHECK("rowmin_kernel");
    return PO_OK;
}

int po_hdbscan_mst_merge(int64_t n, int dtype, const void* d_core, void* d_work, int64_t* d_u, int64_t* d_v, void* d_w,
                         int64_t* h_components, po_stream_t stream) {
    if (!d_core || !d_work || !d_u || !d_v || !d_w || !h_components || n < 1 || n > 0x7FFFFFFFll ||
        (dtype != PO_F32 && dtype != PO_F64)) {
        set_error("po_hdbscan_mst_merge: bad arguments");
        return PO_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    Work w = carve(d_work, n);
    const int ni = (int)n;
    int counters[2];
    PO_CUDA_CHECK(cudaMemcpyAsync(counters, w.counters, sizeof(counters), cudaMemcpyDeviceToHost, st));
    PO_CUDA_CHECK(cudaStreamSynchronize(st));
    const int before = counters[1], edges_before = counters[0];
    if (before <= 1) {
        *h_components = before;
        return PO_OK;
    }
    const unsigned g = (unsigned)((n + 255) / 256);
    PO_CUDA_CHECK(cudaMemsetAsync(w.comp_key, 0xFF, 2 * n * sizeof(unsigned long long), st));
    comp_key_kernel<<<g, 256, 0, st>>>(ni, w.comp, w.row_key, w.comp_key);
    comp_edge_kernel<<<g, 256, 0, st>>>(ni, w.comp, w.row_key, w.row_j, w.comp_key, w.comp_edge);
    if (dtype == PO_F32)
        hook_kernel<float><<<g, 256, 0, st>>>(ni, (const float*)d_core, w.comp, w.row_j, w.row_d, w.comp_edge, w.P, w.counters, d_u,
                                              d_v, (float*)d_w);
    else
        hook_kernel<double><<<g, 256, 0, st>>>(ni, (const double*)d_core, w.comp, w.row_j, w.row_d, w.comp_edge, w.P, w.counters,
                                               d_u, d_v, (double*)d_w);
    // the hook forest is at most `before` deep: ceil(log2(before)) + 1 jumps reach every root
    int jumps = 1;
    while ((1 << (jumps - 1)) < before) ++jumps;
    int* src = w.P;
    int* dst = w.P2;
    for (int q = 0; q < jumps; ++q) {
        jump_kernel<<<g, 256, 0, st>>>(ni, src, dst);
        std::swap(src, dst);
    }
    PO_CUDA_CHECK(cudaMemsetAsync(w.counters + 1, 0, sizeof(int), st));
    relabel_kernel<<<g, 256, 0, st>>>(ni, src, w.comp, w.counters);
    for (int q = 0; q < 4 + jumps; ++q) count_launch(2);  // comp_key, comp_edge, hook, the jumps, relabel
    PO_LAUNCH_CHECK("Boruvka merge kernels");
    PO_CUDA_CHECK(cudaMemcpyAsync(counters, w.counters, sizeof(counters), cudaMemcpyDeviceToHost, st));
    PO_CUDA_CHECK(cudaStreamSynchronize(st));
    // a forest over n vertices: edges + components == n, and every component lost at least half
    if (counters[0] + counters[1] != ni || counters[1] > before / 2 || counters[0] <= edges_before) {
        set_error("po_hdbscan_mst_merge: inconsistent round (%d components before, %d after, %d edges); is the matrix "
                  "symmetric and free of NaN, and was every row scanned once since the last merge?", before, counters[1],
                  counters[0]);
        return PO_ERR_CUDA;
    }
    *h_components = counters[1];
    return PO_OK;
}

int po_hdbscan_tree(int64_t n, int64_t min_cluster_size, int64_t* u, int64_t* v, double* w, int64_t* sl_left, int64_t* sl_right,
                    double* sl_dist, int64_t* sl_size, int64_t* ct_parent, int64_t* ct_child, double* ct_lambda, int64_t* ct_size,
                    int64_t* ct_rows, int64_t* labels, double* probabilities) {
    if (n < 2 || min_cluster_size < 2 || !u || !v || !w || !sl_left || !sl_right || !sl_dist || !sl_size || !ct_parent ||
        !ct_child || !ct_lambda || !ct_size || !ct_rows || !labels || !probabilities) {
        set_error("po_hdbscan_tree: bad arguments (n = %lld, min_cluster_size = %lld)", (long long)n, (long long)min_cluster_size);
        return PO_ERR_ARG;
    }
    const int64_t m = n - 1;
    // 1. the edges in tie-rule order, oriented (min, max)
    std::vector<Edge> e(m);
    for (int64_t k = 0; k < m; ++k) {
        if (u[k] < 0 || u[k] >= n || v[k] < 0 || v[k] >= n || u[k] == v[k] || std::isnan(w[k])) {
            set_error("po_hdbscan_tree: edge %lld = (%lld, %lld) is not an edge between two of %lld points", (long long)k,
                      (long long)u[k], (long long)v[k], (long long)n);
            return PO_ERR_ARG;
        }
        e[k] = {std::min(u[k], v[k]), std::max(u[k], v[k]), w[k] + 0.0};
    }
    std::sort(e.begin(), e.end(), [](const Edge& x, const Edge& y) {
        if (x.w != y.w) return x.w < y.w;
        if (x.a != y.a) return x.a < y.a;
        return x.b < y.b;
    });
    for (int64_t k = 0; k < m; ++k) {
        u[k] = e[k].a;
        v[k] = e[k].b;
        w[k] = e[k].w;
    }
    // 2. single-linkage tree (contrib's label): union-find, node n + k is made by edge k
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
        const int64_t a = find(e[k].a), b = find(e[k].b);
        if (a == b) {
            set_error("po_hdbscan_tree: the edges are not a spanning tree (edge %lld closes a cycle)", (long long)k);
            return PO_ERR_ARG;
        }
        sl_left[k] = a;
        sl_right[k] = b;
        sl_dist[k] = e[k].w;
        sl_size[k] = size[a] + size[b];
        parent[a] = parent[b] = n + k;
        size[n + k] = sl_size[k];
    }
    // 3. condensed tree (contrib's condense_tree)
    std::vector<int64_t> left(sl_left, sl_left + m), right(sl_right, sl_right + m);
    const int64_t root = 2 * n - 2;
    std::vector<int64_t> relabel(root + 1, 0), order, sub;
    std::vector<char> ignore(root + 1, 0);
    relabel[root] = n;
    int64_t next_label = n + 1, rows = 0;
    auto emit = [&](int64_t p, int64_t c, double lam, int64_t sz) {
        ct_parent[rows] = p;
        ct_child[rows] = c;
        ct_lambda[rows] = lam;
        ct_size[rows] = sz;
        ++rows;
    };
    auto count = [&](int64_t x) { return x >= n ? sl_size[x - n] : (int64_t)1; };
    bfs(left, right, n, root, order);
    for (const int64_t node : order) {
        if (ignore[node] || node < n) continue;
        const int64_t l = left[node - n], r = right[node - n];
        const double d = sl_dist[node - n];
        const double lam = d > 0.0 ? 1.0 / d : std::numeric_limits<double>::infinity();
        const int64_t lc = count(l), rc = count(r);
        if (lc >= min_cluster_size && rc >= min_cluster_size) {
            relabel[l] = next_label++;
            emit(relabel[node], relabel[l], lam, lc);
            relabel[r] = next_label++;
            emit(relabel[node], relabel[r], lam, rc);
            continue;
        }
        int64_t drop[2];
        int nd = 0;
        if (lc < min_cluster_size && rc < min_cluster_size) {
            drop[nd++] = l;
            drop[nd++] = r;
        } else if (lc < min_cluster_size) {
            relabel[r] = relabel[node];
            drop[nd++] = l;
        } else {
            relabel[l] = relabel[node];
            drop[nd++] = r;
        }
        for (int q = 0; q < nd; ++q) {
            bfs(left, right, n, drop[q], sub);
            for (const int64_t s : sub) {
                if (s < n) emit(relabel[node], s, lam, 1);
                ignore[s] = 1;
            }
        }
    }
    *ct_rows = rows;
    // 4. stability (contrib's compute_stability), accumulated in condensed-tree order
    const int64_t first = n, last = next_label - 1;  // cluster ids: the root n, then n + 1 .. next_label - 1
    std::vector<double> births(next_label, std::numeric_limits<double>::quiet_NaN()), stability(next_label, 0.0);
    std::vector<double> deaths(next_label, 0.0);
    std::vector<char> seen(next_label, 0);
    std::vector<std::vector<int64_t>> children(next_label);
    for (int64_t k = 0; k < rows; ++k) {
        if (ct_child[k] >= n) {
            births[ct_child[k]] = ct_lambda[k];
            children[ct_parent[k]].push_back(ct_child[k]);
        }
    }
    births[first] = 0.0;
    for (int64_t k = 0; k < rows; ++k) {
        const int64_t p = ct_parent[k];
        stability[p] += (ct_lambda[k] - births[p]) * (double)ct_size[k];
        deaths[p] = seen[p] ? std::max(deaths[p], ct_lambda[k]) : ct_lambda[k];
        seen[p] = 1;
    }
    // 5. excess of mass over the clusters below the root, deepest id first (contrib's get_clusters, "eom").
    //    Whether a node keeps itself depends only on its children's (updated) stabilities; contrib then
    //    unmarks the whole subtree of every kept node.  Here one top-down pass does that: a cluster is selected
    //    when it keeps itself and no ancestor below the root does.  Cluster ids grow downwards, so ascending
    //    id order visits parents first.
    std::vector<char> keeps(next_label, 0), is_cluster(next_label, 0), covered(next_label, 0);
    std::vector<int64_t> cluster_parent(next_label, -1);
    for (int64_t k = 0; k < rows; ++k)
        if (ct_child[k] >= n) cluster_parent[ct_child[k]] = ct_parent[k];
    for (int64_t node = last; node > first; --node) {
        double subtree = 0.0;
        for (const int64_t c : children[node]) subtree += stability[c];
        if (subtree > stability[node])
            stability[node] = subtree;
        else
            keeps[node] = 1;
    }
    for (int64_t c = first + 1; c <= last; ++c) {
        const int64_t p = cluster_parent[c];
        covered[c] = p > first && (covered[p] || keeps[p]);
        is_cluster[c] = keeps[c] && !covered[c];
    }
    // 6. labels: a point's nearest selected ancestor, numbered in ascending cluster id; probabilities as
    //    contrib's get_probabilities
    std::vector<int64_t> label_of(next_label, -1), top(next_label, -1), cluster_of_label;
    for (int64_t c = first + 1; c <= last; ++c) {
        if (is_cluster[c]) {
            label_of[c] = (int64_t)cluster_of_label.size();
            cluster_of_label.push_back(c);
        }
    }
    for (int64_t k = 0; k < rows; ++k)  // parents precede their children in the condensed tree
        if (ct_child[k] >= n) top[ct_child[k]] = is_cluster[ct_child[k]] ? label_of[ct_child[k]] : top[ct_parent[k]];
    for (int64_t k = 0; k < rows; ++k) {
        const int64_t c = ct_child[k];
        if (c >= n) continue;
        const int64_t lab = top[ct_parent[k]];
        labels[c] = lab;
        probabilities[c] = 0.0;
        if (lab < 0) continue;
        const double ml = deaths[cluster_of_label[lab]], lam = ct_lambda[k];
        probabilities[c] = (ml == 0.0 || std::isinf(lam)) ? 1.0 : std::min(lam, ml) / ml;
    }
    return PO_OK;
}

}  // extern "C"
