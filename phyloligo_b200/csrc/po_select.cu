// The front half of phyloselect.py on the device: what its K-medoids (PAM) loop and its nearest-
// neighbour consumers (t-SNE / HDBSCAN on a precomputed matrix) read out of the N x N distance
// matrix, computed while the matrix (or a block row of it) is still resident in HBM instead of from
// a 40 GB file read back into host RAM (reference doc: 800 GB of RAM for phyloselect on large data).
//
// Replaces, in reference phylopackage/bin/phyloselect.py:
//   KMedoids._get_initial_medoid_indices  :291-309  np.argsort(np.sum(D, axis=1))[:k]      -> po_matrix_rowsums
//   KMedoids._get_cluster_ics             :187-195  np.argmin(D[medoid_ics, :], axis=0)     -> po_matrix_argmin_rows
//   KMedoids._update_medoid_ics_in_place  :197-240  per cluster: sum of D over its members for
//                                                   every member, argmin, compare with the
//                                                   current medoid's cost                    -> po_matrix_rowsums (masked)
//                                                                                              + po_cluster_argmin
//   TSNE(metric="precomputed") / HDBSCAN(metric="precomputed") :381-428: the k nearest
//   neighbours of every row (sklearn kneighbors_graph on a precomputed matrix)                -> po_matrix_knn
//   HDBSCAN's core distances (hdbscan's mutual_reachability: np.partition(D, min_samples,
//   axis=0)[min_samples], an exact entry of the matrix)                                       -> po_matrix_kth
//
// The first four are single passes over rows of the matrix: HBM bound, 4 bytes per entry read once.
#include <float.h>
#include "po_common.cuh"

namespace po {

template <typename T>
__device__ __forceinline__ double ld_entry(const void* D, int64_t idx) {
    return (double)reinterpret_cast<const T*>(D)[idx];
}

// out[i] = sum over columns j of D[row(i), j], restricted to labels[j] == row_label[i] when labels are
// given.  One CTA of 256 threads per row, float64 accumulation in a fixed order (reproducible).
template <typename T>
__global__ void __launch_bounds__(256) rowsums_kernel(const void* __restrict__ D, int64_t ld, const int64_t* __restrict__ rows,
                                                      int64_t ncols, const int* __restrict__ labels,
                                                      const int* __restrict__ row_labels, double* __restrict__ out) {
    const int64_t i = blockIdx.x;
    const int64_t r = rows ? rows[i] : i;
    const T* row = reinterpret_cast<const T*>(D) + r * ld;
    const int want = labels ? row_labels[i] : 0;
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    // four independent accumulators per thread: four loads in flight, summation order fixed by the indices
    int64_t j = threadIdx.x;
    for (; j + 3 * 256 < ncols; j += 4 * 256) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t c = j + u * 256;
            const double v = (double)row[c];
            if (!labels || labels[c] == want) acc[u] += v;
        }
    }
    for (; j < ncols; j += 256) {
        const double v = (double)row[j];
        if (!labels || labels[j] == want) acc[0] += v;
    }
    double s = (acc[0] + acc[1]) + (acc[2] + acc[3]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
    __shared__ double red[8];
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += red[w];
        out[i] = t;
    }
}

// out[j] = index c (0 .. k-1) of the smallest D[rows[c], j] as np.argmin picks it: the first NaN when there is
// one (whatever its sign), else the first of the smallest values (-0.0 == +0.0).
template <typename T>
__global__ void __launch_bounds__(256) argmin_rows_kernel(const void* __restrict__ D, int64_t ld, const int64_t* __restrict__ rows,
                                                          int k, int64_t ncols, int* __restrict__ out) {
    const int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (j >= ncols) return;
    double best = ld_entry<T>(D, rows[0] * ld + j);
    int arg = 0;
    for (int c = 1; c < k && best == best; ++c) {
        const double v = ld_entry<T>(D, rows[c] * ld + j);
        if (v < best || v != v) {
            best = v;
            arg = c;
        }
    }
    out[j] = arg;
}

// order-preserving map of a double onto an unsigned 64-bit key; -0.0 takes the key of +0.0 (they compare equal)
__device__ __forceinline__ unsigned long long dkey(double v) {
    unsigned long long b = (unsigned long long)__double_as_longlong(v);
    if (b == 0x8000000000000000ull) b = 0ull;
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
// np.argmin's order of the costs: a NaN of either sign comes first, then the values ascending
__device__ __forceinline__ unsigned long long argmin_key(double v) { return (v != v) ? 0ull : dkey(v); }

// per cluster: members, smallest cost among the members and the first member that has it (np.argmin: the first
// NaN cost when there is one)
__global__ void __launch_bounds__(256) cluster_min_kernel(const double* __restrict__ cost, const int* __restrict__ labels, int64_t n,
                                                          int k, unsigned long long* __restrict__ min_key,
                                                          long long* __restrict__ count) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const int c = labels[i];
    if (c < 0 || c >= k) return;
    atomicMin(&min_key[c], argmin_key(cost[i]));
    atomicAdd(reinterpret_cast<unsigned long long*>(&count[c]), 1ull);
}
__global__ void __launch_bounds__(256) cluster_argmin_kernel(const double* __restrict__ cost, const int* __restrict__ labels, int64_t n,
                                                             int k, const unsigned long long* __restrict__ min_key,
                                                             long long* __restrict__ arg) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const int c = labels[i];
    if (c < 0 || c >= k) return;
    if (argmin_key(cost[i]) == min_key[c]) atomicMin(&arg[c], (long long)i);
}
__global__ void cluster_init_kernel(unsigned long long* min_key, long long* arg, long long* count, int k) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < k) {
        min_key[c] = ~0ull;
        arg[c] = 0x7FFFFFFFFFFFFFFFll;
        count[c] = 0;
    }
}
__global__ void cluster_finish_kernel(const unsigned long long* min_key, const long long* arg, const double* cost, double* best_cost,
                                      long long* best_idx, int k) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < k) {
        const bool any = min_key[c] != ~0ull;
        best_idx[c] = any ? arg[c] : -1;
        best_cost[c] = any ? cost[arg[c]] : 0.0;
    }
}

// k nearest neighbours of every row, the row's own column excluded: ascending distance, ties by
// column index, -0.0 equal to +0.0, NaN (either sign) last.  One CTA per row.  Float32 rows:
// Fast path (one pass over the row, HBM bound): 8192 entries of the row -- 64 evenly spaced runs of 128
// consecutive columns, or the whole row when it is that short -- are loaded into shared memory and a radix
// select over them gives a threshold at about twice the sample rank that corresponds to k; one pass over
// the row then gathers every entry at or below the threshold (k of them are guaranteed to be the k
// smallest; about 2k + 200 are expected), which are sorted by (distance, column).  When fewer than k or
// more than 4096 entries pass (an unlucky sample, massive ties, NaN rows) the row falls back to the
// exact path.
// Exact path (five passes): a radix select over the order-preserving 32-bit keys of the row's
// entries (four 8-bit passes, each a shared-memory histogram of the still undecided prefix class) finds
// the key of the k-th smallest entry; everything strictly below it, then the first ties in column
// order, are gathered and sorted in shared memory (bitonic, keys = (distance key, column)).
// Float64 rows take the exact path only, over the entries' full-width 64-bit keys (eight histogram passes):
// float64 distances that round to one float32 are ordered by value, not as ties.  Such matrices come from
// text files and are small; the float32 path is what the resident matrix of the distance stage takes.
constexpr int KNN_THREADS = 256;
constexpr int KNN_MAX_K = 1024;
constexpr int KNN_CAP = 4096;     // candidates the fast path can hold (32 KB of shared memory)
constexpr int KNN_SAMPLE = 8192;  // entries of the row sampled for the fast path's threshold

// order-preserving map of a float onto an unsigned 32-bit key; -0.0 takes the key of +0.0
__device__ __forceinline__ unsigned fkey(float v) {
    unsigned b = __float_as_uint(v);
    if (b == 0x80000000u) b = 0u;
    return (b >> 31) ? ~b : (b | 0x80000000u);
}
// the keys the selections rank by: NaN (either sign) last
__device__ __forceinline__ unsigned okey(float v) { return (v != v) ? 0xFFFFFFFFu : fkey(v); }
__device__ __forceinline__ unsigned long long okey(double v) { return (v != v) ? ~0ull : dkey(v); }

// an item of the exact path's sort, ordered by (key, column): one word for a 32-bit key, a pair for a 64-bit one
__device__ __forceinline__ unsigned long long knn_item(unsigned key, int64_t j) { return ((unsigned long long)key << 32) | (unsigned)j; }
__device__ __forceinline__ unsigned knn_col(unsigned long long it) { return (unsigned)(it & 0xFFFFFFFFull); }
struct KnnItem64 {
    unsigned long long key, col;
};
__device__ __forceinline__ KnnItem64 knn_item(unsigned long long key, int64_t j) { return {key, (unsigned long long)(unsigned)j}; }
__device__ __forceinline__ unsigned knn_col(KnnItem64 it) { return (unsigned)it.col; }
__device__ __forceinline__ bool operator>(KnnItem64 a, KnnItem64 b) { return a.key != b.key ? a.key > b.key : a.col > b.col; }
__device__ __forceinline__ bool operator==(KnnItem64 a, KnnItem64 b) { return a.key == b.key && a.col == b.col; }

// Radix select over order-preserving keys K (32 bits for float entries, 64 for double), 8 bits per pass from
// the top, each pass a shared-memory histogram of the still undecided prefix class: the key of the
// need-th smallest (1-based) key_of(j) over the columns j < ncols, j != self, and in *nties how many
// entries equal to it belong to the `need` smallest.  Called by every thread of the CTA.
template <typename K, typename KeyOf>
__device__ __forceinline__ K radix_select(KeyOf key_of, int64_t ncols, int64_t self, unsigned need, unsigned* hist, unsigned* nties) {
    __shared__ K r_prefix, r_mask;
    __shared__ unsigned r_need;
    const int tid = threadIdx.x;
    if (tid == 0) {
        r_prefix = 0;
        r_mask = 0;
        r_need = need;  // rank (1-based) of the wanted entry inside the current prefix class
    }
    __syncthreads();
    for (int pass = 0; pass < (int)sizeof(K); ++pass) {
        const int shift = 8 * ((int)sizeof(K) - 1 - pass);
        hist[tid] = 0u;
        __syncthreads();
        const K prefix = r_prefix, mask = r_mask;
        for (int64_t j0 = 0; j0 < ncols; j0 += KNN_THREADS) {
            const int64_t j = j0 + tid;
            unsigned bin = 0xFFFFFFFFu;
            if (j < ncols && j != self) {
                const K key = key_of(j);
                if ((key & mask) == prefix) bin = (unsigned)(key >> shift) & 255u;
            }
            // distances share their leading bits: aggregate equal bins inside the warp, one atomic per distinct bin
            const unsigned active = __ballot_sync(0xFFFFFFFFu, bin != 0xFFFFFFFFu);
            if (bin != 0xFFFFFFFFu) {
                const unsigned peers = __match_any_sync(active, bin);
                if ((tid & 31) == __ffs(peers) - 1) atomicAdd(&hist[bin], (unsigned)__popc(peers));
            }
        }
        __syncthreads();
        if (tid == 0) {
            unsigned need_ = r_need, acc = 0u;
            int b = 0;
            for (; b < 255; ++b) {
                if (acc + hist[b] >= need_) break;
                acc += hist[b];
            }
            r_need = need_ - acc;
            r_prefix = prefix | ((K)b << shift);
            r_mask = mask | ((K)255u << shift);
        }
        __syncthreads();
    }
    *nties = r_need;
    return r_prefix;
}

template <typename T>
__global__ void __launch_bounds__(KNN_THREADS) knn_kernel(const void* __restrict__ D, int64_t ld, int64_t ncols, int64_t self0, int k,
                                                          int kpad, int* __restrict__ out_idx, float* __restrict__ out_dist) {
    extern __shared__ unsigned long long knn_items[];  // fast path: candidates (distance key << 32 | column)
    __shared__ unsigned hist[256];
    __shared__ unsigned s_prefix, s_mask, s_need, s_below, s_ties;
    const int64_t i = blockIdx.x;
    const T* row = reinterpret_cast<const T*>(D) + i * ld;
    const int64_t self = self0 + i;
    const int tid = threadIdx.x;
    auto key_of = [&](int64_t j) { return okey(row[j]); };
    // ---------------- fast path (float32) ----------------
    if constexpr (sizeof(T) == 4) {
        unsigned* samp = reinterpret_cast<unsigned*>(knn_items);
        const int S = (int)min((int64_t)KNN_SAMPLE, ncols);
        const bool whole = (int64_t)S == ncols;
        const int64_t run_stride = ncols / 64;  // >= 128 when the row is longer than the sample
        for (int q = tid; q < S; q += KNN_THREADS) {
            const int64_t j = whole ? (int64_t)q : (int64_t)(q >> 7) * run_stride + (q & 127);
            samp[q] = (j == self) ? 0xFFFFFFFFu : key_of(j);
        }
        if (tid == 0) {
            s_prefix = 0u;
            s_mask = 0u;
            // rank in the sample: the k-th entry itself when the sample is the row, else twice the expected rank
            s_need = whole ? (unsigned)k : (unsigned)min(S, (int)((2.0 * (double)k * (double)S) / (double)ncols) + 17);
        }
        __syncthreads();
        for (int pass = 0; pass < 4; ++pass) {
            const int shift = 24 - 8 * pass;
            hist[tid] = 0u;
            __syncthreads();
            const unsigned prefix = s_prefix, mask = s_mask;
            for (int q0 = 0; q0 < S; q0 += KNN_THREADS) {
                const int q = q0 + tid;
                unsigned bin = 0xFFFFFFFFu;
                if (q < S) {
                    const unsigned key = samp[q];
                    if ((key & mask) == prefix) bin = (key >> shift) & 255u;
                }
                const unsigned active = __ballot_sync(0xFFFFFFFFu, bin != 0xFFFFFFFFu);
                if (bin != 0xFFFFFFFFu) {
                    const unsigned peers = __match_any_sync(active, bin);
                    if ((tid & 31) == __ffs(peers) - 1) atomicAdd(&hist[bin], (unsigned)__popc(peers));
                }
            }
            __syncthreads();
            if (tid == 0) {
                unsigned need = s_need, acc = 0u;
                int b = 0;
                for (; b < 255; ++b) {
                    if (acc + hist[b] >= need) break;
                    acc += hist[b];
                }
                s_need = need - acc;
                s_prefix = prefix | ((unsigned)b << shift);
                s_mask = mask | (255u << shift);
            }
            __syncthreads();
        }
        const unsigned tau = s_prefix;
        if (tid == 0) s_below = 0u;
        __syncthreads();  // everybody has read the threshold; the sample buffer becomes the candidate buffer
        // warp-collective append of the lanes' entries that pass the threshold (order in the buffer is irrelevant)
        auto push = [&](bool take, unsigned key, int64_t j) {
            const unsigned m = __ballot_sync(0xFFFFFFFFu, take);
            if (m) {
                unsigned base = 0u;
                if ((tid & 31) == __ffs(m) - 1) base = atomicAdd(&s_below, (unsigned)__popc(m));
                base = __shfl_sync(0xFFFFFFFFu, base, __ffs(m) - 1);
                const unsigned pos = base + __popc(m & ((1u << (tid & 31)) - 1u));
                if (take && pos < (unsigned)KNN_CAP) knn_items[pos] = ((unsigned long long)key << 32) | (unsigned)j;
            }
        };
        // 16-byte loads, four per thread in flight; the append runs only for the warps that saw a passing entry
        constexpr int VEC = 16 / (int)sizeof(T);
        constexpr int UN = 4;
        int64_t head = 0;
        if ((reinterpret_cast<uintptr_t>(row) & 15) == 0) {
            const int64_t nvec = ncols / VEC;
            const uint4* row4 = reinterpret_cast<const uint4*>(row);
            for (int64_t v0 = 0; v0 < nvec; v0 += (int64_t)KNN_THREADS * UN) {
                uint4 raw[UN];
#pragma unroll
                for (int u = 0; u < UN; ++u) {
                    const int64_t v = v0 + (int64_t)u * KNN_THREADS + tid;
                    raw[u] = (v < nvec) ? __ldg(row4 + v) : make_uint4(0u, 0u, 0u, 0u);
                }
#pragma unroll
                for (int u = 0; u < UN; ++u) {
                    const int64_t v = v0 + (int64_t)u * KNN_THREADS + tid;
                    const T* e = reinterpret_cast<const T*>(&raw[u]);
                    unsigned keys[VEC];
                    bool takes[VEC], any = false;
#pragma unroll
                    for (int c = 0; c < VEC; ++c) {
                        keys[c] = okey(e[c]);
                        takes[c] = v < nvec && keys[c] <= tau && v * VEC + c != self;
                        any |= takes[c];
                    }
                    if (__any_sync(0xFFFFFFFFu, any)) {
#pragma unroll
                        for (int c = 0; c < VEC; ++c) push(takes[c], keys[c], v * VEC + c);
                    }
                }
            }
            head = nvec * VEC;
        }
        for (int64_t j0 = head; j0 < ncols; j0 += KNN_THREADS) {
            const int64_t j = j0 + tid;
            unsigned key = 0xFFFFFFFFu;
            bool take = false;
            if (j < ncols && j != self) {
                key = key_of(j);
                take = key <= tau;
            }
            push(take, key, j);
        }
        __syncthreads();
        const unsigned count = s_below;
        if (count >= (unsigned)k && count <= (unsigned)KNN_CAP) {
            int sz = 2;
            while (sz < (int)count) sz <<= 1;
            for (int q = (int)count + tid; q < sz; q += KNN_THREADS) knn_items[q] = ~0ull;
            __syncthreads();
            for (int size = 2; size <= sz; size <<= 1) {
                for (int stride = size >> 1; stride > 0; stride >>= 1) {
                    for (int q = tid; q < sz; q += KNN_THREADS) {
                        const int partner = q ^ stride;
                        if (partner > q) {
                            const bool up = (q & size) == 0;
                            const unsigned long long a = knn_items[q], b = knn_items[partner];
                            if ((a > b) == up) {
                                knn_items[q] = b;
                                knn_items[partner] = a;
                            }
                        }
                    }
                    __syncthreads();
                }
            }
            for (int q = tid; q < k; q += KNN_THREADS) {
                const unsigned long long it = knn_items[q];
                const int col = (int)(unsigned)(it & 0xFFFFFFFFull);
                out_idx[i * k + q] = col;
                out_dist[i * k + q] = (float)row[col];
            }
            return;
        }
        __syncthreads();
    }
    // ---------------- exact path ----------------
    using K = decltype(okey(T()));
    using Item = decltype(knn_item(K(), 0));
    Item* items = reinterpret_cast<Item*>(knn_items);  // kpad
    const Item pad = knn_item(~K(0), 0xFFFFFFFFll);   // sorts after every entry, NaN included
    unsigned nties;  // how many entries equal to the k-th smallest belong to the k smallest
    const K kth = radix_select<K>(key_of, ncols, self, (unsigned)k, hist, &nties);  // key of the k-th smallest
    if (tid == 0) {
        s_below = 0u;
        s_ties = 0u;
    }
    for (int q = tid; q < kpad; q += KNN_THREADS) items[q] = pad;
    __syncthreads();
    // gather: entries below the threshold in any order (sorted afterwards); ties in column order, which a
    // strided sweep does not give -- so ties are taken by their rank among the ties (count of equal
    // entries at smaller columns), computed block by block of columns in order
    for (int64_t j0 = 0; j0 < ncols; j0 += KNN_THREADS) {
        const int64_t j = j0 + tid;
        K key = ~K(0);
        bool valid = j < ncols && j != self;
        if (valid) key = key_of(j);
        const bool below = valid && key < kth;
        const bool tie = valid && key == kth;
        if (below) items[atomicAdd(&s_below, 1u)] = knn_item(key, j);
        // rank of this tie among the ties: ties in earlier blocks (s_ties) + ties at smaller columns in this block
        const unsigned tmask = __ballot_sync(0xFFFFFFFFu, tie);
        __shared__ unsigned warp_ties[KNN_THREADS / 32];
        if ((tid & 31) == 0) warp_ties[tid >> 5] = __popc(tmask);
        __syncthreads();
        if (tie) {
            unsigned before = s_ties + __popc(tmask & ((1u << (tid & 31)) - 1u));
            for (int w = 0; w < (tid >> 5); ++w) before += warp_ties[w];
            if (before < nties) items[(unsigned)k - nties + before] = knn_item(key, j);
        }
        __syncthreads();
        if (tid == 0) {
            unsigned t = 0u;
            for (int w = 0; w < KNN_THREADS / 32; ++w) t += warp_ties[w];
            s_ties += t;
        }
        __syncthreads();
    }
    // bitonic sort of the kpad items (padding sorts last); the ties already sit in column order at the end
    for (int size = 2; size <= kpad; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int q = tid; q < kpad; q += KNN_THREADS) {
                const int partner = q ^ stride;
                if (partner > q) {
                    const bool up = (q & size) == 0;
                    const Item a = items[q], b = items[partner];
                    if ((a > b) == up) {
                        items[q] = b;
                        items[partner] = a;
                    }
                }
            }
            __syncthreads();
        }
    }
    for (int q = tid; q < k; q += KNN_THREADS) {
        const Item it = items[q];
        const int col = (int)knn_col(it);
        out_idx[i * k + q] = (it == pad) ? -1 : col;
        out_dist[i * k + q] = (it == pad) ? __int_as_float(0x7FC00000) : (float)row[col];
    }
}


// The k-th smallest entry (1-based, every column counted, the diagonal too) of every row, returned bit for
// bit in the matrix's dtype: the exact radix select of knn_kernel over the full-width key of the entry
// (4 passes for float, 8 for double), so that no two float64 entries that round to one float32 are
// confused.  NaN entries sort last; -0.0 equals +0.0 and comes back as +0.0.  One CTA per row.
__device__ __forceinline__ float from_okey(unsigned k) { return __uint_as_float((k >> 31) ? (k & 0x7FFFFFFFu) : ~k); }
__device__ __forceinline__ double from_okey(unsigned long long k) {
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k));
}

template <typename T>
__global__ void __launch_bounds__(KNN_THREADS) kth_kernel(const void* __restrict__ D, int64_t ld, int64_t ncols, int k, T* __restrict__ out) {
    __shared__ unsigned hist[256];
    const T* row = reinterpret_cast<const T*>(D) + (int64_t)blockIdx.x * ld;
    unsigned nties;
    const auto key = radix_select<decltype(okey(T()))>([&](int64_t j) { return okey(row[j]); }, ncols, (int64_t)-1, (unsigned)k, hist, &nties);
    if (threadIdx.x == 0) out[blockIdx.x] = from_okey(key);
}

}  // namespace po

using namespace po;

extern "C" {

int po_matrix_rowsums(const void* d_D, int64_t ld, int dtype, const int64_t* d_rows, int64_t n_rows, int64_t n_cols,
                      const int* d_labels, const int* d_row_labels, double* d_out, po_stream_t stream) {
    // a matrix without columns may have no storage: its sums are 0 and it is never read
    if ((!d_D && n_cols > 0) || !d_out || n_rows < 0 || n_cols < 0 || ld < n_cols || (dtype != PO_F32 && dtype != PO_F64) ||
        ((d_labels == nullptr) != (d_row_labels == nullptr)) || n_rows > 0x7FFFFFFFll) {
        set_error("po_matrix_rowsums: bad arguments");
        return PO_ERR_ARG;
    }
    if (n_rows == 0) return PO_OK;
    if (dtype == PO_F32)
        rowsums_kernel<float><<<(unsigned)n_rows, 256, 0, (cudaStream_t)stream>>>(d_D, ld, d_rows, n_cols, d_labels, d_row_labels, d_out);
    else
        rowsums_kernel<double><<<(unsigned)n_rows, 256, 0, (cudaStream_t)stream>>>(d_D, ld, d_rows, n_cols, d_labels, d_row_labels, d_out);
    count_launch(2);
    PO_LAUNCH_CHECK("rowsums_kernel");
    return PO_OK;
}

int po_matrix_argmin_rows(const void* d_D, int64_t ld, int dtype, const int64_t* d_rows, int k, int64_t n_cols, int* d_out,
                          po_stream_t stream) {
    if (!d_D || !d_rows || !d_out || k < 1 || n_cols < 0 || ld < n_cols || (dtype != PO_F32 && dtype != PO_F64)) {
        set_error("po_matrix_argmin_rows: bad arguments");
        return PO_ERR_ARG;
    }
    if (n_cols == 0) return PO_OK;
    const unsigned grid = (unsigned)((n_cols + 255) / 256);
    if (dtype == PO_F32)
        argmin_rows_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(d_D, ld, d_rows, k, n_cols, d_out);
    else
        argmin_rows_kernel<double><<<grid, 256, 0, (cudaStream_t)stream>>>(d_D, ld, d_rows, k, n_cols, d_out);
    count_launch(2);
    PO_LAUNCH_CHECK("argmin_rows_kernel");
    return PO_OK;
}

int po_cluster_argmin(const double* d_cost, const int* d_labels, int64_t n, int k, void* d_work, int64_t* d_best_idx,
                      double* d_best_cost, int64_t* d_count, po_stream_t stream) {
    // no points (n = 0) may come with no storage: every cluster is then empty
    if (((!d_cost || !d_labels) && n > 0) || !d_work || !d_best_idx || !d_best_cost || !d_count || n < 0 || k < 1) {
        set_error("po_cluster_argmin: bad arguments");
        return PO_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long* min_key = reinterpret_cast<unsigned long long*>(d_work);  // k keys, then k candidate indices
    long long* arg = reinterpret_cast<long long*>(min_key + k);
    const unsigned gk = (unsigned)((k + 255) / 256), gn = (unsigned)((n + 255) / 256);
    cluster_init_kernel<<<gk, 256, 0, st>>>(min_key, arg, reinterpret_cast<long long*>(d_count), k);
    if (n > 0) {
        cluster_min_kernel<<<gn, 256, 0, st>>>(d_cost, d_labels, n, k, min_key, reinterpret_cast<long long*>(d_count));
        cluster_argmin_kernel<<<gn, 256, 0, st>>>(d_cost, d_labels, n, k, min_key, arg);
    }
    cluster_finish_kernel<<<gk, 256, 0, st>>>(min_key, arg, d_cost, d_best_cost, reinterpret_cast<long long*>(d_best_idx), k);
    count_launch(2);
    PO_LAUNCH_CHECK("cluster_argmin kernels");
    return PO_OK;
}

int po_matrix_knn(const void* d_D, int64_t ld, int dtype, int64_t n_rows, int64_t n_cols, int64_t self0, int k, int* d_idx,
                  float* d_dist, po_stream_t stream) {
    if (!d_D || !d_idx || !d_dist || n_rows < 0 || n_cols < 1 || ld < n_cols || (dtype != PO_F32 && dtype != PO_F64) || k < 1 ||
        n_rows > 0x7FFFFFFFll || n_cols > 0x7FFFFFFFll) {
        set_error("po_matrix_knn: bad arguments");
        return PO_ERR_ARG;
    }
    if (k > KNN_MAX_K || k > n_cols - 1) {
        set_error("po_matrix_knn: k = %d outside [1, min(%d, columns - 1 = %lld)]", k, KNN_MAX_K, (long long)(n_cols - 1));
        return PO_ERR_UNSUPPORTED;
    }
    if (n_rows == 0) return PO_OK;
    int kpad = 2;
    while (kpad < k) kpad <<= 1;
    // float32: candidates of the fast path / items of the exact path; float64: the exact path's (key, column) pairs
    const size_t smem = dtype == PO_F32 ? (size_t)(kpad > KNN_CAP ? kpad : KNN_CAP) * 8 : (size_t)kpad * sizeof(KnnItem64);
    if (dtype == PO_F32)
        knn_kernel<float><<<(unsigned)n_rows, KNN_THREADS, smem, (cudaStream_t)stream>>>(d_D, ld, n_cols, self0, k, kpad, d_idx, d_dist);
    else
        knn_kernel<double><<<(unsigned)n_rows, KNN_THREADS, smem, (cudaStream_t)stream>>>(d_D, ld, n_cols, self0, k, kpad, d_idx, d_dist);
    count_launch(2);
    PO_LAUNCH_CHECK("knn_kernel");
    return PO_OK;
}

int po_matrix_kth(const void* d_D, int64_t ld, int dtype, int64_t n_rows, int64_t n_cols, int k, void* d_out, po_stream_t stream) {
    if (!d_D || !d_out || n_rows < 0 || n_cols < 1 || ld < n_cols || (dtype != PO_F32 && dtype != PO_F64) || k < 1 ||
        n_rows > 0x7FFFFFFFll) {
        set_error("po_matrix_kth: bad arguments");
        return PO_ERR_ARG;
    }
    if (k > n_cols) {
        set_error("po_matrix_kth: k = %d outside [1, columns = %lld]", k, (long long)n_cols);
        return PO_ERR_UNSUPPORTED;
    }
    if (n_rows == 0) return PO_OK;
    if (dtype == PO_F32)
        kth_kernel<float><<<(unsigned)n_rows, KNN_THREADS, 0, (cudaStream_t)stream>>>(d_D, ld, n_cols, k, (float*)d_out);
    else
        kth_kernel<double><<<(unsigned)n_rows, KNN_THREADS, 0, (cudaStream_t)stream>>>(d_D, ld, n_cols, k, (double*)d_out);
    count_launch(2);
    PO_LAUNCH_CHECK("kth_kernel");
    return PO_OK;
}

}  // extern "C"
