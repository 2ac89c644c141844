// extern "C" entry points of libphyloligo_b200.so (see include/phyloligo_b200.h).
#include <stdarg.h>
#include <atomic>
#include <thread>
#include <vector>
#include "po_common.cuh"

namespace po {

static thread_local char g_error[512] = "";
static std::atomic<long long> g_launches{0};
static std::atomic<int> g_timing{0};

struct FamilyTiming {
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending;
    double total_ms = 0.0;
    long long launches = 0;
};
static FamilyTiming g_fam[4];

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

void count_launch(int) { g_launches.fetch_add(1, std::memory_order_relaxed); }

LaunchTimer::LaunchTimer(int fam, cudaStream_t s) : stream(s), family(fam), active(false) {
    if (g_timing.load(std::memory_order_relaxed) && fam >= 0 && fam < 4) {
        if (cudaEventCreate(&e0) == cudaSuccess && cudaEventCreate(&e1) == cudaSuccess) {
            cudaEventRecord(e0, stream);
            active = true;
        }
    }
}
LaunchTimer::~LaunchTimer() {
    if (active) {
        cudaEventRecord(e1, stream);
        g_fam[family].pending.emplace_back(e0, e1);
    }
}

int parse_pattern(const char* pattern, PatternGeom* g) {
    if (!pattern) {
        set_error("pattern is NULL");
        return PO_ERR_ARG;
    }
    const int width = (int)strlen(pattern);
    if (width < 1 || width > PO_MAX_PATTERN) {
        set_error("pattern length %d outside [1, %d]", width, PO_MAX_PATTERN);
        return PO_ERR_UNSUPPORTED;
    }
    memset(g, 0, sizeof(*g));
    g->width = width;
    int k = 0;
    for (int i = 0; i < width; ++i) k += (pattern[i] == '1');
    if (k > PO_MAX_K) {
        set_error("pattern has %d ones, more than the supported %d", k, PO_MAX_K);
        return PO_ERR_UNSUPPORTED;
    }
    g->k = k;
    // runs of consecutive '1': window offset o holds bits [2(width-1-o), +2) of the
    // rolling register; the j-th '1' (from the left) is digit 4^(k-1-j) of the word.
    int j = 0, nruns = 0;
    for (int o = 0; o < width;) {
        if (pattern[o] != '1') { ++o; continue; }
        int o2 = o;
        while (o2 + 1 < width && pattern[o2 + 1] == '1') ++o2;
        const int len = o2 - o + 1;
        const int j2 = j + len - 1;
        g->shift[nruns] = (unsigned char)(2 * (width - 1 - o2));
        g->dst[nruns] = (unsigned char)(2 * (k - 1 - j2));
        g->mask[nruns] = (len >= 16) ? 0xFFFFFFFFu : ((1u << (2 * len)) - 1u);
        ++nruns;
        j += len;
        o = o2 + 1;
    }
    g->nruns = nruns;
    int pal = 1;
    for (int i = 0; i < width; ++i) pal &= ((pattern[i] == '1') == (pattern[width - 1 - i] == '1'));
    g->palindromic = pal;
    return PO_OK;
}

}  // namespace po

using namespace po;

extern "C" {

const char* po_version(void) { return "phyloligo_b200 0.1.0 (sm_100a)"; }
const char* po_last_error(void) { return g_error; }

int po_device_info(int* sm_count, int* cc_major, int* cc_minor) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) {
        set_error("no CUDA device");
        return PO_ERR_NODEVICE;
    }
    cudaDeviceProp prop;
    PO_CUDA_CHECK(cudaGetDeviceProperties(&prop, dev));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    return PO_OK;
}

int po_pattern_info(const char* pattern, int* width, int* k, int64_t* dim) {
    PatternGeom g;
    int rc = parse_pattern(pattern, &g);
    if (rc != PO_OK) return rc;
    if (width) *width = g.width;
    if (k) *k = g.k;
    if (dim) *dim = (int64_t)1 << (2 * g.k);
    return PO_OK;
}

int64_t po_fasta_index_host(const uint8_t* h_text, int64_t len, int64_t* h_begin, int64_t* h_end,
                            int64_t cap, int threads) {
    if (!h_text || len < 0) {
        set_error("po_fasta_index_host: bad buffer");
        return PO_ERR_ARG;
    }
    if (threads <= 0) {
        threads = (int)std::thread::hardware_concurrency();
        if (threads <= 0) threads = 1;
        if (threads > 32) threads = 32;
    }
    if (len < (1 << 20)) threads = 1;
    // pass 1 (parallel): positions of every '>' that starts a line
    std::vector<std::vector<int64_t>> found((size_t)threads);
    auto scan = [&](int t) {
        const int64_t lo = len * t / threads, hi = len * (t + 1) / threads;
        const uint8_t* p = h_text + lo;
        const uint8_t* e = h_text + hi;
        while (p < e) {
            const uint8_t* q = (const uint8_t*)memchr(p, '>', (size_t)(e - p));
            if (!q) break;
            const int64_t pos = q - h_text;
            // a line starts after LF, or after a CR (CRLF, or the lone CR of old Mac files: Python's universal
            // newlines, which the reference's SeqIO.parse reads with, break lines there too)
            if (pos == 0 || h_text[pos - 1] == '\n' || h_text[pos - 1] == '\r') found[(size_t)t].push_back(pos);
            p = q + 1;
        }
    };
    if (threads == 1) {
        scan(0);
    } else {
        std::vector<std::thread> pool;
        for (int t = 0; t < threads; ++t) pool.emplace_back(scan, t);
        for (auto& th : pool) th.join();
    }
    // pass 2: header line end -> sequence begin; next header -> sequence end
    int64_t nrec = 0;
    int64_t prev_begin = -1;
    for (int t = 0; t < threads; ++t) {
        for (int64_t pos : found[(size_t)t]) {
            if (prev_begin >= 0 && nrec - 1 < cap && h_end) h_end[nrec - 1] = pos;
            const uint8_t* nl = (const uint8_t*)memchr(h_text + pos, '\n', (size_t)(len - pos));
            int64_t b = nl ? (nl - h_text) + 1 : len;
            // a CR before that LF which is not its CRLF partner ends the header line earlier
            const uint8_t* cr = (const uint8_t*)memchr(h_text + pos, '\r', (size_t)(b - pos));
            if (cr && !(nl && cr + 1 == nl)) b = (cr - h_text) + 1;
            if (nrec < cap && h_begin) h_begin[nrec] = b;
            prev_begin = b;
            ++nrec;
        }
    }
    if (nrec > 0 && nrec - 1 < cap && h_end) h_end[nrec - 1] = len;
    return nrec;
}

int po_profile_batch(const uint8_t* d_text, const int64_t* d_begin, const int64_t* d_end, int64_t n,
                     const char* pattern, int strand, uint32_t* d_counts, uint64_t* d_totals,
                     double* d_freq64, float* d_freq32, po_stream_t stream) {
    PatternGeom g;
    int rc = parse_pattern(pattern, &g);
    if (rc != PO_OK) return rc;
    if (strand != PO_STRAND_PLUS && strand != PO_STRAND_MINUS && strand != PO_STRAND_BOTH) {
        set_error("strand must be 0 (plus), 1 (minus) or 2 (both), got %d", strand);
        return PO_ERR_ARG;
    }
    if (n < 0) {
        set_error("negative record count");
        return PO_ERR_ARG;
    }
    if (n > 0 && (!d_text || !d_begin || !d_end)) {
        set_error("po_profile_batch: NULL input pointer");
        return PO_ERR_ARG;
    }
    if (((uintptr_t)d_text & 15u) != 0) {
        set_error("d_text must be 16-byte aligned");
        return PO_ERR_ARG;
    }
    return launch_profile(d_text, d_begin, d_end, n, g, strand, d_counts, d_totals, d_freq64, d_freq32,
                          (cudaStream_t)stream);
}

int64_t po_prepared_row_bytes(int metric, int64_t dim) {
    if (metric < PO_EUCL || metric > PO_EUCL_GRAM || dim < 1) {
        set_error("po_prepared_row_bytes: bad metric/dim");
        return PO_ERR_ARG;
    }
    return prepared_row_elems(metric, dim) * 4 * (metric == PO_JSD ? 2 : 1);
}

int64_t po_prepared_bytes(int metric, int64_t n, int64_t dim) {
    if (metric < PO_EUCL || metric > PO_EUCL_GRAM || dim < 1 || n < 0) {
        set_error("po_prepared_bytes: bad metric/n/dim");
        return PO_ERR_ARG;
    }
    return prepared_bytes(metric, n, dim);
}

int po_prepare_profiles(int metric, const void* d_X, int dtype, int64_t n, int64_t dim, int64_t ldx,
                        void* d_P, double* d_aux, po_stream_t stream) {
    if (metric < PO_EUCL || metric > PO_EUCL_GRAM) {
        set_error("unknown metric %d", metric);
        return PO_ERR_ARG;
    }
    if (n < 0 || dim < 1 || ldx < dim || (n > 0 && (!d_X || !d_P))) {
        set_error("po_prepare_profiles: bad arguments");
        return PO_ERR_ARG;
    }
    return launch_prepare(metric, d_X, dtype, n, dim, ldx, d_P, d_aux, (cudaStream_t)stream);
}

int po_rank_transform(const void* d_X, int dtype, int64_t n, int64_t dim, int64_t ldx, double* d_ranks, int64_t ldr,
                      po_stream_t stream) {
    if (n < 0 || dim < 1 || ldx < dim || ldr < dim || (dtype != PO_F32 && dtype != PO_F64) || (n > 0 && (!d_X || !d_ranks))) {
        set_error("po_rank_transform: bad arguments");
        return PO_ERR_ARG;
    }
    return launch_rank_transform(d_X, dtype, n, dim, ldx, d_ranks, ldr, (cudaStream_t)stream);
}

static int distance_block_checked(int metric, const void* d_P, const double* d_aux, int64_t n, int64_t dim,
                                  int64_t row0, int64_t row1, int64_t col0, int64_t col1, void* d_out,
                                  int64_t ld_out, int64_t out_row0, int64_t out_col0, void* d_mir, int64_t ld_mir,
                                  int64_t mir_row0, int64_t mir_col0, int out_dtype, unsigned flags,
                                  po_stream_t stream) {
    if (metric < PO_EUCL || metric > PO_EUCL_GRAM) {
        set_error("unknown metric %d", metric);
        return PO_ERR_ARG;
    }
    if (out_dtype != PO_F32 && out_dtype != PO_F64) {
        set_error("unknown output dtype %d", out_dtype);
        return PO_ERR_ARG;
    }
    if (n < 1 || dim < 1 || row0 < 0 || col0 < 0 || row1 > n || col1 > n || !d_P || !d_out || !d_mir) {
        set_error("po_distance_block: bad arguments (n=%lld rows [%lld,%lld) cols [%lld,%lld))", (long long)n,
                  (long long)row0, (long long)row1, (long long)col0, (long long)col1);
        return PO_ERR_ARG;
    }
    if ((metric == PO_SC || metric == PO_KT || metric == PO_BC) && !d_aux) {
        set_error("metric %d needs d_aux from po_prepare_profiles", metric);
        return PO_ERR_ARG;
    }
    if (((uintptr_t)d_P & 15u) != 0) {
        set_error("d_P must be 16-byte aligned");
        return PO_ERR_ARG;
    }
    return launch_distance(metric, d_P, d_aux, n, dim, row0, row1, col0, col1, d_out, ld_out, out_row0, out_col0,
                           d_mir, ld_mir, mir_row0, mir_col0, out_dtype, flags, (cudaStream_t)stream);
}

int po_distance_block(int metric, const void* d_P, const double* d_aux, int64_t n, int64_t dim,
                      int64_t row0, int64_t row1, int64_t col0, int64_t col1, void* d_out, int64_t ld_out,
                      int64_t out_row0, int64_t out_col0, int out_dtype, unsigned flags, po_stream_t stream) {
    return distance_block_checked(metric, d_P, d_aux, n, dim, row0, row1, col0, col1, d_out, ld_out, out_row0,
                                  out_col0, d_out, ld_out, out_row0, out_col0, out_dtype, flags, stream);
}

int po_distance_block_ex(int metric, const void* d_P, const double* d_aux, int64_t n, int64_t dim,
                         int64_t row0, int64_t row1, int64_t col0, int64_t col1, void* d_out, int64_t ld_out,
                         int64_t out_row0, int64_t out_col0, void* d_mirror, int64_t ld_mirror,
                         int64_t mirror_row0, int64_t mirror_col0, int out_dtype, unsigned flags,
                         po_stream_t stream) {
    return distance_block_checked(metric, d_P, d_aux, n, dim, row0, row1, col0, col1, d_out, ld_out, out_row0,
                                  out_col0, d_mirror, ld_mirror, mirror_row0, mirror_col0, out_dtype, flags, stream);
}

int po_ipc_export(const void* d_ptr, void* h_handle64, int64_t* offset) {
    if (!d_ptr || !h_handle64 || !offset) {
        set_error("po_ipc_export: NULL argument");
        return PO_ERR_ARG;
    }
    // base of the allocation that contains d_ptr (cuMemGetAddressRange, through the runtime's entry-point lookup)
    typedef int (*get_range_fn)(unsigned long long*, size_t*, unsigned long long);
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    PO_CUDA_CHECK(cudaGetDriverEntryPoint("cuMemGetAddressRange", &fn, cudaEnableDefault, &qres));
    if (!fn || qres != cudaDriverEntryPointSuccess) {
        set_error("po_ipc_export: cuMemGetAddressRange is not available");
        return PO_ERR_CUDA;
    }
    unsigned long long base = 0;
    size_t size = 0;
    const int rc = reinterpret_cast<get_range_fn>(fn)(&base, &size, (unsigned long long)(uintptr_t)d_ptr);
    if (rc != 0) {
        set_error("po_ipc_export: cuMemGetAddressRange failed (%d)", rc);
        return PO_ERR_CUDA;
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t h;
    PO_CUDA_CHECK(cudaIpcGetMemHandle(&h, reinterpret_cast<void*>((uintptr_t)base)));
    memcpy(h_handle64, &h, 64);
    *offset = (int64_t)((unsigned long long)(uintptr_t)d_ptr - base);
    return PO_OK;
}

int po_ipc_open(const void* h_handle64, void** d_base) {
    if (!h_handle64 || !d_base) {
        set_error("po_ipc_open: NULL argument");
        return PO_ERR_ARG;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, h_handle64, 64);
    PO_CUDA_CHECK(cudaIpcOpenMemHandle(d_base, h, cudaIpcMemLazyEnablePeerAccess));
    return PO_OK;
}

int po_ipc_close(void* d_base) {
    if (d_base) PO_CUDA_CHECK(cudaIpcCloseMemHandle(d_base));
    return PO_OK;
}

int po_copy2d_async(void* dst, int64_t dst_pitch, const void* src, int64_t src_pitch, int64_t width, int64_t rows,
                    po_stream_t stream) {
    if (width < 0 || rows < 0 || dst_pitch < width || src_pitch < width) {
        set_error("po_copy2d_async: bad geometry (width %lld, rows %lld, pitches %lld / %lld)", (long long)width,
                  (long long)rows, (long long)dst_pitch, (long long)src_pitch);
        return PO_ERR_ARG;
    }
    if (width == 0 || rows == 0) return PO_OK;
    if (!dst || !src) {
        set_error("po_copy2d_async: NULL pointer");
        return PO_ERR_ARG;
    }
    PO_CUDA_CHECK(cudaMemcpy2DAsync(dst, (size_t)dst_pitch, src, (size_t)src_pitch, (size_t)width, (size_t)rows,
                                    cudaMemcpyDefault, (cudaStream_t)stream));
    return PO_OK;
}

int64_t po_launch_count(void) { return g_launches.load(); }

int po_timing_enable(int on) {
    g_timing.store(on ? 1 : 0);
    return PO_OK;
}

static void drain(FamilyTiming& f) {
    for (auto& pr : f.pending) {
        float ms = 0.f;
        if (cudaEventSynchronize(pr.second) == cudaSuccess && cudaEventElapsedTime(&ms, pr.first, pr.second) == cudaSuccess) {
            f.total_ms += ms;
            f.launches += 1;
        }
        cudaEventDestroy(pr.first);
        cudaEventDestroy(pr.second);
    }
    f.pending.clear();
}

int po_timing_reset(void) {
    for (auto& f : g_fam) {
        drain(f);
        f.total_ms = 0.0;
        f.launches = 0;
    }
    return PO_OK;
}

int po_timing_read(int family, double* total_ms, int64_t* launches) {
    if (family < 0 || family >= 4) {
        set_error("bad timing family %d", family);
        return PO_ERR_ARG;
    }
    drain(g_fam[family]);
    if (total_ms) *total_ms = g_fam[family].total_ms;
    if (launches) *launches = g_fam[family].launches;
    return PO_OK;
}

}  // extern "C"
