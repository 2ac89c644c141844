// Shared helpers for the phyloligo_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include "../../include/phyloligo_b200.h"

namespace po {

void set_error(const char* fmt, ...);
void count_launch(int family);

// Event-based timing of kernel families (enabled by po_timing_enable).
struct LaunchTimer {
    cudaStream_t stream;
    int family;
    cudaEvent_t e0, e1;
    bool active;
    LaunchTimer(int family, cudaStream_t s);
    ~LaunchTimer();
};

#define PO_CUDA_CHECK(expr)                                                              \
    do {                                                                                 \
        cudaError_t _e = (expr);                                                         \
        if (_e != cudaSuccess) {                                                         \
            po::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),        \
                          __FILE__, __LINE__);                                           \
            (void)cudaGetLastError(); /* reported here: do not leave it for the next launch check */ \
            return PO_ERR_CUDA;                                                          \
        }                                                                                \
    } while (0)

#define PO_LAUNCH_CHECK(name)                                                            \
    do {                                                                                 \
        cudaError_t _e = cudaGetLastError();                                             \
        if (_e != cudaSuccess) {                                                         \
            po::set_error("launch of %s failed: %s", name, cudaGetErrorString(_e));      \
            return PO_ERR_CUDA;                                                          \
        }                                                                                \
    } while (0)

// Geometry of a spaced pattern, passed by value to the profiling kernel.
// A pattern is decomposed into runs of consecutive '1's; every run is one
// shift+mask of the rolling window register.
struct PatternGeom {
    int width;           // len(pattern)
    int k;               // number of '1'
    int nruns;           // runs of consecutive '1's
    int palindromic;     // pattern == reversed(pattern)
    unsigned char shift[16];  // bit shift of run r inside the window register
    unsigned char dst[16];    // bit position of run r inside the word code
    unsigned int mask[16];    // 4^len - 1 of run r
};

int parse_pattern(const char* pattern, PatternGeom* g);

// launchers implemented in the .cu files
int launch_profile(const uint8_t* d_text, const int64_t* d_begin, const int64_t* d_end, int64_t n,
                   const PatternGeom& g, int strand, uint32_t* d_counts, uint64_t* d_totals,
                   double* d_freq64, float* d_freq32, cudaStream_t stream);

int launch_prepare(int metric, const void* d_X, int dtype, int64_t n, int64_t dim, int64_t ldx,
                   void* d_P, double* d_aux, cudaStream_t stream);

int launch_rank_transform(const void* d_X, int dtype, int64_t n, int64_t dim, int64_t ldx, double* d_R, int64_t ldr,
                          cudaStream_t stream);

int launch_distance(int metric, const void* d_P, const double* d_aux, int64_t n, int64_t dim,
                    int64_t row0, int64_t row1, int64_t col0, int64_t col1,
                    void* d_out, int64_t ld_out, int64_t out_row0, int64_t out_col0,
                    void* d_mir, int64_t ld_mir, int64_t mir_row0, int64_t mir_col0,
                    int out_dtype, unsigned flags, cudaStream_t stream);

// Euclidean distances on the tensor cores (po_gram.cu)
bool eucl_use_gram(int metric, int64_t dim);
int64_t gram_prepared_bytes(int64_t n, int64_t dim);
int launch_gram_prepare(const void* d_X, int dtype, int64_t n, int64_t dim, int64_t ldx, void* d_P, double* d_aux,
                        cudaStream_t stream);
bool sc_use_gram(int metric, int64_t dim);
int64_t sc_gram_prepared_bytes(int64_t n, int64_t dim);
int launch_sc_gram_prepare(const void* d_X, int dtype, int64_t n, int64_t dim, int64_t ldx, void* d_P, double* d_aux,
                           cudaStream_t stream);
int launch_gram(int metric, const void* d_P, const double* d_aux, int64_t n, int64_t dim, int64_t row0, int64_t row1, int64_t col0,
                int64_t col1, void* d_out, int64_t ld_out, int64_t out_row0, int64_t out_col0, void* d_mir,
                int64_t ld_mir, int64_t mir_row0, int64_t mir_col0, int out_dtype, unsigned flags, cudaStream_t stream);

// number of 32-bit elements of one prepared row (JSD: of one operand copy)
int64_t prepared_row_elems(int metric, int64_t dim);
// total bytes of the prepared operand buffer of n rows
int64_t prepared_bytes(int metric, int64_t n, int64_t dim);

int launch_jsd(const void* d_P, int64_t n, int64_t dim, int64_t row0, int64_t row1, int64_t col0, int64_t col1,
               void* d_out, int64_t ld_out, int64_t out_row0, int64_t out_col0, void* d_mir, int64_t ld_mir,
               int64_t mir_row0, int64_t mir_col0, int out_dtype, unsigned flags, cudaStream_t stream);

// microseconds per grid.sync() of the linkage kernels' grid (po_linkage.cu; po_microbench kind 4)
int barrier_latency_us(double* result);

}  // namespace po
