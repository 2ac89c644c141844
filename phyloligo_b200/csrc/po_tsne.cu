// phyloselect's t-SNE projection (reference bin/phyloselect.py:381-398) on the resident N x N matrix: what
// sklearn.manifold.TSNE(metric="precomputed", method="barnes_hut", angle=0.0, init="random") computes.  With
// angle 0 scikit-learn's Barnes-Hut gradient is the exact gradient of the sparse-P objective, so this file
// evaluates that gradient exactly:
//   check_array / check_non_negative       -> po_tsne_check
//   _utils._binary_search_perplexity       -> po_tsne_conditional (one warp per row, float64)
//   sum(P + P.T) in _joint_probabilities_nn -> po_tsne_sum (fixed-order float64 sum)
//   _barnes_hut_tsne.gradient, negative part -> po_tsne_repulsion (exact all-pairs pass: the hot path)
//   positive part, KL, _gradient_descent step -> po_tsne_attraction_step (CSR row walk, fused update)
// Every sum runs in a fixed order (no floating-point atomics), so two fits on one device are bitwise equal.
#include <cmath>
#include "po_common.cuh"

namespace po {

namespace {

typedef unsigned long long u64;

// ---------------------------------------------------------------------------------------------------
// input check: the smallest row-major index i * n_cols + j of a NaN, infinite or negative entry
// ---------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) check_kernel(const T* __restrict__ D, int64_t ld, int64_t n_cols, u64* __restrict__ first_bad) {
    const int64_t i = blockIdx.x;
    const T* row = D + i * ld;
    u64 bad = ~0ull;
    for (int64_t j = threadIdx.x; j < n_cols; j += blockDim.x) {
        const T x = row[j];
        if (!(x >= (T)0) || isinf(x)) {  // NaN fails x >= 0; -0.0 passes, as in check_non_negative
            bad = (u64)(i * n_cols + j);
            break;  // this thread's later columns are larger indices
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) bad = min(bad, __shfl_xor_sync(0xFFFFFFFFu, bad, o));
    if ((threadIdx.x & 31) == 0 && bad != ~0ull) atomicMin(first_bad, bad);
}

// ---------------------------------------------------------------------------------------------------
// conditional P: scikit-learn's _binary_search_perplexity, one warp per row.  The squared distances are
// float32 as scikit-learn's (distances.data **= 2 in the matrix's dtype, then astype(float32)); the search runs
// in float64 with the same bracketing, update rules, tolerance and step limit.
// ---------------------------------------------------------------------------------------------------
constexpr int COND_WARPS = 4;
constexpr int COND_SLOTS = 32;  // k <= 32 * 32 = 1024 (po_matrix_knn's limit)

template <typename T>
__global__ void __launch_bounds__(COND_WARPS * 32) conditional_kernel(const T* __restrict__ D, int64_t ld, int64_t n,
                                                                      const int* __restrict__ idx, int k, double desired_entropy,
                                                                      double* __restrict__ P) {
    const int64_t i = (int64_t)blockIdx.x * COND_WARPS + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= n) return;
    float d2[COND_SLOTS];
    double p[COND_SLOTS];
#pragma unroll
    for (int s = 0; s < COND_SLOTS; ++s) {
        const int t = s * 32 + lane;
        d2[s] = 0.f;
        p[s] = 0.0;
        if (t < k) {
            const T d = D[i * ld + idx[i * k + t]];
            d2[s] = (float)(d * d);
        }
    }
    double beta = 1.0, beta_min = -INFINITY, beta_max = INFINITY;
    for (int step = 0; step < 100; ++step) {
        double sum_p = 0.0;
#pragma unroll
        for (int s = 0; s < COND_SLOTS; ++s) {
            if (s * 32 + lane < k) {
                p[s] = exp(-(double)d2[s] * beta);
                sum_p += p[s];
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum_p += __shfl_xor_sync(0xFFFFFFFFu, sum_p, o);  // the same value in every lane
        if (sum_p == 0.0) sum_p = 1e-8;  // EPSILON_DBL
        double sum_dp = 0.0;
#pragma unroll
        for (int s = 0; s < COND_SLOTS; ++s) {
            if (s * 32 + lane < k) {
                p[s] /= sum_p;
                sum_dp += (double)d2[s] * p[s];
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) sum_dp += __shfl_xor_sync(0xFFFFFFFFu, sum_dp, o);
        const double diff = log(sum_p) + beta * sum_dp - desired_entropy;
        if (fabs(diff) <= 1e-5) break;
        if (diff > 0.0) {
            beta_min = beta;
            beta = beta_max == INFINITY ? beta * 2.0 : (beta + beta_max) / 2.0;
        } else {
            beta_max = beta;
            beta = beta_min == -INFINITY ? beta / 2.0 : (beta + beta_min) / 2.0;
        }
    }
#pragma unroll
    for (int s = 0; s < COND_SLOTS; ++s)
        if (s * 32 + lane < k) P[i * k + s * 32 + lane] = p[s];
}

// ---------------------------------------------------------------------------------------------------
// fixed-order float64 sums: one CTA, thread t adds elements t, t + 1024, ... in order, then a fixed tree
// ---------------------------------------------------------------------------------------------------
constexpr int SUM_THREADS = 1024;

__device__ __forceinline__ double block_sum(double v, double* sh) {
    sh[threadIdx.x] = v;
    __syncthreads();
    for (int h = SUM_THREADS / 2; h > 0; h >>= 1) {
        if ((int)threadIdx.x < h) sh[threadIdx.x] += sh[threadIdx.x + h];
        __syncthreads();
    }
    const double r = sh[0];
    __syncthreads();
    return r;
}

// out[a] = sum of x[a * n .. a * n + n - 1] for a < arrays
__global__ void __launch_bounds__(SUM_THREADS) sum_kernel(const double* __restrict__ x, int64_t n, int arrays, double* __restrict__ out) {
    __shared__ double sh[SUM_THREADS];
    for (int a = 0; a < arrays; ++a) {
        double s = 0.0;
        for (int64_t e = threadIdx.x; e < n; e += SUM_THREADS) s += x[a * n + e];
        s = block_sum(s, sh);
        if (threadIdx.x == 0) out[a] = s;
    }
}

int launch_sum(const double* d_x, int64_t n, int arrays, double* d_out, cudaStream_t st) {
    sum_kernel<<<1, SUM_THREADS, 0, st>>>(d_x, n, arrays, d_out);
    count_launch(2);
    PO_LAUNCH_CHECK("tsne sum_kernel");
    return PO_OK;
}

// ---------------------------------------------------------------------------------------------------
// repulsion: for every row i, sum_j q_ij^2 (y_i - y_j) and sum_j q_ij, q_ij = 1 / (1 + |y_i - y_j|^2), over all
// j (j = i adds exactly 1 to the second sum and nothing to the first; the fold removes it).
//
// A CTA owns REP_ROWS rows and one chunk of the columns; a thread keeps REP_RPT rows as two packed f32x2 row
// pairs, so every y_j staged in shared memory (as (x, x, y, y): one broadcast 16-byte load) serves four rows.
// Per pair: FADD2 dx, FADD2 dy, 2 FFMA2 for 1 + dx^2 + dy^2, MUFU.RCP, FMUL2 q^2, 2 FFMA2 for the forces, FADD2
// for Z -- 8 FP32 lane operations and one MUFU, i.e. the FP32 pipe (128 lanes / clk / SM) and the MUFU pipe (16 /
// clk / SM) bound the pair rate within 4 % of each other.  Sums: float32 runs of REP_SUB columns, those added in
// float32 over a REP_TILE, then folded into float64 accumulators; a chunk's float64 partials are added over the
// chunks in a fixed order.  The two float32 levels cost 3 FADD2 per 32 columns and cut the rounding of one flat
// float32 run of 256 several-fold, which matters near convergence, where attraction and repulsion cancel to a
// few digits.
// ---------------------------------------------------------------------------------------------------
constexpr int REP_THREADS = 128;
constexpr int REP_RPT = 4;
constexpr int REP_ROWS = REP_THREADS * REP_RPT;
constexpr int REP_TILE = 256;
constexpr int REP_SUB = 32;  // float32 runs of 32 columns, added in float32 over a tile, then folded into float64
constexpr int64_t REP_TARGET_CTAS = 4096;
constexpr float REP_FAR = 1e18f;  // padding columns: q ~ 5e-37, q^2 flushes to 0

__device__ __forceinline__ u64 pk2(float lo, float hi) {
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk2(u64 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
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
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

int64_t rep_chunks(int64_t n) {
    const int64_t row_ctas = (n + REP_ROWS - 1) / REP_ROWS, tiles = (n + REP_TILE - 1) / REP_TILE;
    int64_t s = (REP_TARGET_CTAS + row_ctas - 1) / row_ctas;
    return s < 1 ? 1 : (s > tiles ? tiles : s);
}
int64_t rep_chunk_cols(int64_t n, int64_t chunks) {
    const int64_t tiles = (n + REP_TILE - 1) / REP_TILE;
    return (tiles + chunks - 1) / chunks * REP_TILE;
}

// workspace: partial x, y, z [chunks][n]; rep x, y [n]; zrow [n]; kl_row, gn_row [n]; sums [4]
struct TWork {
    double *px, *py, *pz, *rx, *ry, *zrow, *kl_row, *gn_row, *sums;
};
TWork tcarve(void* d_work, int64_t n) {
    const int64_t s = rep_chunks(n);
    double* p = reinterpret_cast<double*>(d_work);
    TWork w;
    w.px = p;
    w.py = p + s * n;
    w.pz = p + 2 * s * n;
    w.rx = p + 3 * s * n;
    w.ry = w.rx + n;
    w.zrow = w.ry + n;
    w.kl_row = w.zrow + n;
    w.gn_row = w.kl_row + n;
    w.sums = w.gn_row + n;
    return w;
}
int64_t tworkspace(int64_t n) { return (3 * rep_chunks(n) * n + 5 * n + 4) * (int64_t)sizeof(double); }

__global__ void __launch_bounds__(REP_THREADS) repulsion_kernel(const float2* __restrict__ Y, int n, int chunk_cols, double* __restrict__ px,
                                                                double* __restrict__ py, double* __restrict__ pz) {
    __shared__ float4 sy[REP_TILE];
    const int r0 = blockIdx.x * REP_ROWS;
    const int c0 = blockIdx.y * chunk_cols, c1 = min(n, c0 + chunk_cols);
    u64 X2[2], Y2[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int ra = r0 + threadIdx.x + REP_THREADS * (2 * q), rb = ra + REP_THREADS;
        const float2 a = ra < n ? Y[ra] : make_float2(0.f, 0.f), b = rb < n ? Y[rb] : make_float2(0.f, 0.f);
        X2[q] = pk2(a.x, b.x);
        Y2[q] = pk2(a.y, b.y);
    }
    const u64 one2 = pk2(1.f, 1.f);
    double ax[REP_RPT] = {}, ay[REP_RPT] = {}, az[REP_RPT] = {};
    for (int t0 = c0; t0 < c1; t0 += REP_TILE) {
        __syncthreads();
        for (int u = threadIdx.x; u < REP_TILE; u += REP_THREADS) {
            const int j = t0 + u;
            const float2 v = j < c1 ? Y[j] : make_float2(REP_FAR, REP_FAR);
            sy[u] = make_float4(v.x, v.x, v.y, v.y);
        }
        __syncthreads();
        u64 mx[2] = {0, 0}, my[2] = {0, 0}, mz[2] = {0, 0};
        for (int u0 = 0; u0 < REP_TILE; u0 += REP_SUB) {
            u64 fx[2] = {0, 0}, fy[2] = {0, 0}, fz[2] = {0, 0};
#pragma unroll 4
            for (int u = u0; u < u0 + REP_SUB; ++u) {
                const float4 v = sy[u];
                const u64 xj = pk2(v.x, v.y), yj = pk2(v.z, v.w);
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const u64 dx = sub2(X2[q], xj), dy = sub2(Y2[q], yj);
                    const u64 d2 = fma2(dy, dy, fma2(dx, dx, one2));
                    float lo, hi;
                    upk2(d2, lo, hi);
                    const u64 w = pk2(rcp_approx(lo), rcp_approx(hi));
                    const u64 w2 = mul2(w, w);
                    fx[q] = fma2(w2, dx, fx[q]);
                    fy[q] = fma2(w2, dy, fy[q]);
                    fz[q] = add2(fz[q], w);
                }
            }
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                mx[q] = add2(mx[q], fx[q]);
                my[q] = add2(my[q], fy[q]);
                mz[q] = add2(mz[q], fz[q]);
            }
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            float a, b;
            upk2(mx[q], a, b);
            ax[2 * q] += a;
            ax[2 * q + 1] += b;
            upk2(my[q], a, b);
            ay[2 * q] += a;
            ay[2 * q + 1] += b;
            upk2(mz[q], a, b);
            az[2 * q] += a;
            az[2 * q + 1] += b;
        }
    }
    const int64_t off = (int64_t)blockIdx.y * n;
#pragma unroll
    for (int m = 0; m < REP_RPT; ++m) {
        const int r = r0 + threadIdx.x + REP_THREADS * m;
        if (r < n) {
            px[off + r] = ax[m];
            py[off + r] = ay[m];
            pz[off + r] = az[m];
        }
    }
}

// the chunks' partials of every row, added in chunk order; the row's own q_ii = 1 removed from Z's part
__global__ void fold_kernel(int64_t n, int chunks, const double* __restrict__ px, const double* __restrict__ py,
                            const double* __restrict__ pz, double* __restrict__ rx, double* __restrict__ ry, double* __restrict__ zrow) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double x = 0.0, y = 0.0, z = 0.0;
    for (int s = 0; s < chunks; ++s) {
        x += px[s * n + i];
        y += py[s * n + i];
        z += pz[s * n + i];
    }
    rx[i] = x;
    ry[i] = y;
    zrow[i] = z - 1.0;
}

// ---------------------------------------------------------------------------------------------------
// attraction + step, one warp per row: sum_j P_ij q_ij (y_i - y_j) over the row's CSR entries (P_ij read as
// scikit-learn's float32 val_P of the float64 P scaled as _tsne scales it in place: P * early_exaggeration in the
// first stage, then (P * ee) * (1 / ee) in the second, since scipy's P /= ee multiplies by the reciprocal), the gradient 4 (attraction - repulsion / Z), optionally the row's KL terms, then
// _gradient_descent's gains / momentum / position update into the other position buffer.
// ---------------------------------------------------------------------------------------------------
constexpr int STEP_WARPS = 8;

struct StepArgs {
    const int64_t* indptr;
    const int* indices;
    const double* P;
    double mul, rdiv;  // rdiv = 1.0 / div, rounded once on the host as scipy's 1.0 / other
    const float2* Y;
    float2* Y_next;   // NULL: gradient only
    double* update;   // float64 (scikit-learn's update is float64 when the learning rate is a float64 scalar)
    float* gains;
    float* grad_out;  // optional: the gradient before the gains, [n x 2]
    double momentum, lr;
    int update64;
    int compute_error;
};

__global__ void __launch_bounds__(STEP_WARPS * 32) step_kernel(StepArgs a, int64_t n, const double* __restrict__ rx,
                                                               const double* __restrict__ ry, const double* __restrict__ Zp,
                                                               double* __restrict__ kl_row, double* __restrict__ gn_row) {
    const int64_t i = (int64_t)blockIdx.x * STEP_WARPS + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= n) return;
    const double Z = *Zp;
    const float2 yi = a.Y[i];
    double sx = 0.0, sy = 0.0, kl = 0.0;
    const float tiny = 1.17549435e-38f;  // FLOAT32_TINY
    for (int64_t e = a.indptr[i] + lane; e < a.indptr[i + 1]; e += 32) {
        const int j = a.indices[e];
        const float p = (float)((a.P[e] * a.mul) * a.rdiv);
        const float2 yj = a.Y[j];
        const float bx = __fsub_rn(yi.x, yj.x), by = __fsub_rn(yi.y, yj.y);
        const float d = __fadd_rn(__fmul_rn(bx, bx), __fmul_rn(by, by));
        const float q = __fdiv_rn(1.0f, __fadd_rn(1.0f, d));
        const double pq = (double)p * (double)q;
        sx += pq * (double)bx;
        sy += pq * (double)by;
        if (a.compute_error) kl += (double)p * log(fmax((double)p, (double)tiny) / fmax((double)q / Z, (double)tiny));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sx += __shfl_xor_sync(0xFFFFFFFFu, sx, o);
        sy += __shfl_xor_sync(0xFFFFFFFFu, sy, o);
        kl += __shfl_xor_sync(0xFFFFFFFFu, kl, o);
    }
    if (lane != 0) return;
    float g[2] = {(float)(4.0 * (sx - rx[i] / Z)), (float)(4.0 * (sy - ry[i] / Z))};
    if (a.grad_out) {
        a.grad_out[2 * i] = g[0];
        a.grad_out[2 * i + 1] = g[1];
    }
    if (a.compute_error) kl_row[i] = kl;
    if (!a.Y_next) return;
    float yn[2] = {yi.x, yi.y};
    double gn = 0.0;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        const int64_t k = 2 * i + c;
        double u = a.update[k];
        float gain = a.gains[k];
        const bool inc = a.update64 ? u * (double)g[c] < 0.0 : __fmul_rn((float)u, g[c]) < 0.0f;
        gain = inc ? __fadd_rn(gain, 0.2f) : __fmul_rn(gain, 0.8f);
        gain = fmaxf(gain, 0.01f);
        const float gg = __fmul_rn(g[c], gain);
        if (a.update64) {
            u = __dsub_rn(__dmul_rn(a.momentum, u), __dmul_rn(a.lr, (double)gg));
            yn[c] = (float)__dadd_rn((double)yn[c], u);
        } else {
            const float uf = __fsub_rn(__fmul_rn((float)a.momentum, (float)u), __fmul_rn((float)a.lr, gg));
            u = uf;
            yn[c] = __fadd_rn(yn[c], uf);
        }
        a.update[k] = u;
        a.gains[k] = gain;
        gn += (double)gg * (double)gg;
    }
    a.Y_next[i] = make_float2(yn[0], yn[1]);
    if (a.compute_error) gn_row[i] = gn;
}

}  // namespace

}  // namespace po

using namespace po;

extern "C" {

int po_tsne_check(const void* d_D, int64_t ld, int dtype, int64_t n_rows, int64_t n_cols, int64_t row0, void* d_work,
                  po_stream_t stream) {
    if (!d_D || !d_work || n_rows < 0 || n_cols < 0 || row0 < 0 || ld < n_cols || (dtype != PO_F32 && dtype != PO_F64) ||
        n_rows > 0x7FFFFFFFll) {
        set_error("po_tsne_check: bad arguments");
        return PO_ERR_ARG;
    }
    if (n_rows == 0 || n_cols == 0) return PO_OK;
    cudaStream_t st = (cudaStream_t)stream;
    u64* first = reinterpret_cast<u64*>(d_work);
    PO_CUDA_CHECK(cudaMemsetAsync(first, 0xFF, sizeof(u64), st));
    if (dtype == PO_F32)
        check_kernel<float><<<(unsigned)n_rows, 256, 0, st>>>((const float*)d_D, ld, n_cols, first);
    else
        check_kernel<double><<<(unsigned)n_rows, 256, 0, st>>>((const double*)d_D, ld, n_cols, first);
    count_launch(2);
    PO_LAUNCH_CHECK("tsne check_kernel");
    u64 bad = 0;
    PO_CUDA_CHECK(cudaMemcpyAsync(&bad, first, sizeof(bad), cudaMemcpyDeviceToHost, st));
    PO_CUDA_CHECK(cudaStreamSynchronize(st));
    if (bad == ~0ull) return PO_OK;
    const int64_t i = (int64_t)(bad / (u64)n_cols), j = (int64_t)(bad % (u64)n_cols);
    const size_t es = dtype == PO_F32 ? 4 : 8;
    unsigned char raw[8];
    PO_CUDA_CHECK(cudaMemcpy(raw, reinterpret_cast<const char*>(d_D) + (i * ld + j) * (int64_t)es, es, cudaMemcpyDeviceToHost));
    double x;
    if (dtype == PO_F32) {
        float f;
        memcpy(&f, raw, 4);
        x = f;
    } else {
        memcpy(&x, raw, 8);
    }
    if (std::isnan(x))
        set_error("po_tsne_check: entry (%lld, %lld) is NaN", (long long)(row0 + i), (long long)j);
    else if (std::isinf(x))
        set_error("po_tsne_check: entry (%lld, %lld) is infinite (%g)", (long long)(row0 + i), (long long)j, x);
    else
        set_error("po_tsne_check: entry (%lld, %lld) is negative (%.17g); t-SNE needs non-negative distances", (long long)(row0 + i),
                  (long long)j, x);
    return PO_ERR_ARG;
}

int po_tsne_conditional(const void* d_D, int64_t ld, int dtype, int64_t n, const int* d_idx, int k, double perplexity, double* d_P,
                        po_stream_t stream) {
    if (!d_D || !d_idx || !d_P || n < 0 || ld < n || (dtype != PO_F32 && dtype != PO_F64) || k < 1 || k > COND_SLOTS * 32 ||
        !(perplexity > 0.0)) {
        set_error("po_tsne_conditional: bad arguments (k = %d, perplexity = %g)", k, perplexity);
        return PO_ERR_ARG;
    }
    if (n == 0) return PO_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = (unsigned)((n + COND_WARPS - 1) / COND_WARPS);
    const double h = std::log(perplexity);
    if (dtype == PO_F32)
        conditional_kernel<float><<<grid, COND_WARPS * 32, 0, st>>>((const float*)d_D, ld, n, d_idx, k, h, d_P);
    else
        conditional_kernel<double><<<grid, COND_WARPS * 32, 0, st>>>((const double*)d_D, ld, n, d_idx, k, h, d_P);
    count_launch(2);
    PO_LAUNCH_CHECK("tsne conditional_kernel");
    return PO_OK;
}

int po_tsne_sum(const double* d_x, int64_t n, double* d_out, po_stream_t stream) {
    if ((!d_x && n > 0) || !d_out || n < 0) {  // an empty vector may have no storage
        set_error("po_tsne_sum: bad arguments");
        return PO_ERR_ARG;
    }
    return launch_sum(d_x, n, 1, d_out, (cudaStream_t)stream);
}

int64_t po_tsne_workspace(int64_t n) { return n < 1 ? -1 : tworkspace(n); }

int po_tsne_repulsion(const float* d_Y, int64_t n, void* d_work, po_stream_t stream) {
    if (!d_Y || !d_work || n < 2 || n > 0x7FFFFFFFll / 2) {
        set_error("po_tsne_repulsion: bad arguments (n = %lld)", (long long)n);
        return PO_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    TWork w = tcarve(d_work, n);
    const int64_t chunks = rep_chunks(n), cols = rep_chunk_cols(n, chunks);
    const dim3 grid((unsigned)((n + REP_ROWS - 1) / REP_ROWS), (unsigned)chunks);
    repulsion_kernel<<<grid, REP_THREADS, 0, st>>>(reinterpret_cast<const float2*>(d_Y), (int)n, (int)cols, w.px, w.py, w.pz);
    fold_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(n, (int)chunks, w.px, w.py, w.pz, w.rx, w.ry, w.zrow);
    count_launch(2);
    count_launch(2);
    PO_LAUNCH_CHECK("tsne repulsion_kernel / fold_kernel");
    return launch_sum(w.zrow, n, 1, w.sums, st);  // Z
}

int po_tsne_attraction_step(const int64_t* d_indptr, const int* d_indices, const double* d_P, int64_t n, double mul, double div,
                            const float* d_Y, void* d_work, float* d_Y_next, double* d_update, float* d_gains, float* d_grad,
                            double momentum, double learning_rate, int update64, double* h_kl_gradnorm2, po_stream_t stream) {
    if (!d_indptr || !d_indices || !d_P || !d_Y || !d_work || n < 2 || !(div != 0.0) ||
        (d_Y_next && (!d_update || !d_gains || d_Y_next == d_Y))) {
        set_error("po_tsne_attraction_step: bad arguments");
        return PO_ERR_ARG;
    }
    cudaStream_t st = (cudaStream_t)stream;
    TWork w = tcarve(d_work, n);
    StepArgs a;
    a.indptr = d_indptr;
    a.indices = d_indices;
    a.P = d_P;
    a.mul = mul;
    a.rdiv = 1.0 / div;
    a.Y = reinterpret_cast<const float2*>(d_Y);
    a.Y_next = reinterpret_cast<float2*>(d_Y_next);
    a.update = d_update;
    a.gains = d_gains;
    a.grad_out = d_grad;
    a.momentum = momentum;
    a.lr = learning_rate;
    a.update64 = update64 ? 1 : 0;
    a.compute_error = h_kl_gradnorm2 ? 1 : 0;
    step_kernel<<<(unsigned)((n + STEP_WARPS - 1) / STEP_WARPS), STEP_WARPS * 32, 0, st>>>(a, n, w.rx, w.ry, w.sums, w.kl_row,
                                                                                          w.gn_row);
    count_launch(2);
    PO_LAUNCH_CHECK("tsne step_kernel");
    if (!h_kl_gradnorm2) return PO_OK;
    // kl_row and gn_row are adjacent: sums[1] = KL, sums[2] = |grad * gains|^2 (0 without a step)
    if (!d_Y_next) PO_CUDA_CHECK(cudaMemsetAsync(w.gn_row, 0, n * sizeof(double), st));
    const int rc = launch_sum(w.kl_row, n, 2, w.sums + 1, st);
    if (rc != PO_OK) return rc;
    PO_CUDA_CHECK(cudaMemcpyAsync(h_kl_gradnorm2, w.sums + 1, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
    PO_CUDA_CHECK(cudaStreamSynchronize(st));
    return PO_OK;
}

}  // extern "C"
