/*
 * phyloligo_b200 -- C ABI of the B200-native PhylOligo hot path.
 *
 * The reference (itsmeludo/PhylOligo) is pure Python: it has no FFI layer.  The
 * seam this library sits behind is the set of worker functions that the
 * reference's scoop / joblib back-ends call (SURVEY.md section 8b).  Each entry
 * point below names the reference worker(s) it replaces, with file:line into
 * /root/reference/phylopackage.  INTEGRATION.md shows the ctypes stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - plain C: pointers and sizes only, no C++/torch types.
 *   - every function returns 0 (PO_OK) or a negative po_status; the message of
 *     the last failure on the calling thread is available from po_last_error().
 *   - pointers named d_* are DEVICE pointers on the current CUDA device, owned
 *     and allocated by the caller (the Python host uses torch for that).
 *     Pointers named h_* are host pointers.
 *   - `stream` is a cudaStream_t passed as void*; all device work is enqueued
 *     on it and nothing synchronises unless stated.
 */
#ifndef PHYLOLIGO_B200_H
#define PHYLOLIGO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* po_stream_t; /* cudaStream_t */

enum po_status {
    PO_OK = 0,
    PO_ERR_ARG = -1,         /* invalid argument (bad strand / metric / pattern / alignment) */
    PO_ERR_CUDA = -2,        /* a CUDA runtime call or kernel launch failed */
    PO_ERR_UNSUPPORTED = -3, /* valid request outside the implemented envelope */
    PO_ERR_NODEVICE = -4     /* no CUDA device / not an sm_100 device */
};

/* select_strand(), bin/phyloligo.py:124-149 */
enum po_strand { PO_STRAND_PLUS = 0, PO_STRAND_MINUS = 1, PO_STRAND_BOTH = 2 };

/* -d/--distance choices, bin/phyloligo.py:1010; unpack_distances, bin/phyloligo.py:159-164 */
enum po_metric {
    PO_EUCL = 0, PO_JSD = 1, PO_KT = 2, PO_BC = 3, PO_SC = 4,
    /* Eucl in the Gram form ||x||^2 + ||y||^2 - 2 x.y on the tensor cores: what the reference's
     * --large workers compute through sklearn euclidean_distances (bin/phyloligo.py:200-202,
     * 238-246), stated tolerance 1e-4 relative.  PO_EUCL is the direct sum (a-b)^2 of
     * phylodist.Eucl (core/phylodist.py:36-41).  Below 256 dimensions, or with
     * PO_EUCL_EXACT=1 in the environment, PO_EUCL_GRAM runs the PO_EUCL kernel. */
    PO_EUCL_GRAM = 5
};

enum po_dtype { PO_F32 = 0, PO_F64 = 1 };

/* flags of po_distance_block */
#define PO_FLAG_SKIP_LOWER 1u /* skip the kernel tiles that lie wholly below the diagonal       */
#define PO_FLAG_MIRROR     2u /* tiles wholly above the diagonal are also written transposed  */
#define PO_FLAG_MIRROR_ONLY 4u /* with PO_FLAG_MIRROR: store only the transposed tiles (into the mirror
                                  buffer) and nothing into d_out -- the part of a row panel left of its
                                  diagonal square, computed from the block rows above it */

#define PO_MAX_PATTERN 32 /* longest spaced pattern (window width) */
#define PO_MAX_K       10 /* most '1's in a pattern (4^10 bins)     */
#define PO_TILE        64 /* tile edge of the CUDA-core distance kernels                       */
#define PO_TILE_ALIGN 128 /* largest tile granule of any distance kernel (32x64 JSD, 64x64 CUDA-core
                             metrics, 128x128 groups on the tensor cores): block boundaries that are
                             multiples of it never split a tile between two calls */

const char* po_version(void);
const char* po_last_error(void);

/* Number of SMs and compute capability of the current device. */
int po_device_info(int* sm_count, int* cc_major, int* cc_minor);

/*
 * Pattern geometry.  `pattern` is the '0'/'1' string of -p/--pattern (or "1"*k for
 * -k, bin/phyloligo.py:1040-1041).  Characters other than '1' are don't-care
 * positions, exactly as target_index at bin/phyloligo.py:622 treats them.
 * width = len(pattern), k = number of '1', dim = 4^k.
 */
int po_pattern_info(const char* pattern, int* width, int* k, int64_t* dim);

/*
 * FASTA record index on the host -- replaces the SeqIO.parse(genome, "fasta")
 * iteration at bin/phyloligo.py:87,114,154,869,914,959 (Biopython semantics:
 * a record starts at a line beginning with '>', text before the first '>' is
 * ignored, the sequence is every later line up to the next header with
 * whitespace removed).  Writes, for each record, the byte range [begin, end) of
 * its sequence lines inside `h_text`.  Returns the number of records found (it
 * may exceed `cap`, in which case only `cap` entries were written), or a
 * negative po_status.  `threads` <= 0 picks a default.
 */
int64_t po_fasta_index_host(const uint8_t* h_text, int64_t len,
                            int64_t* h_begin, int64_t* h_end, int64_t cap, int threads);

/*
 * Composition profiling of n records -- replaces compute_frequency
 * (bin/phyloligo.py:663-691), compute_frequency_memmap (:693-720) and
 * compute_frequency_h5py_chunk (:756-792), i.e. select_strand (:124-149) +
 * .upper() (:683) + cut_sequence_and_count_pattern (:601-631) + count2freq
 * (:633-661) for every record of a batch.
 *
 *   d_text            raw FASTA text (or bare sequence bytes); 16-byte aligned
 *   d_begin, d_end    per record, byte range of its sequence inside d_text;
 *                     bytes '\n', '\r' and ' ' inside a range are skipped
 *   pattern, strand   as on the command line; strand is a po_strand
 *   d_counts          [n x dim] uint32 word counts in C,G,A,T product order
 *                     (bin/phyloligo.py:653), or NULL
 *   d_totals          [n] uint64 number of counted words (kword_count), or NULL
 *   d_freq64          [n x dim] float64 count/total, correctly rounded -- the
 *                     --large None dtype (bin/phyloligo.py:656), or NULL
 *   d_freq32          [n x dim] float32 cast of that float64 quotient -- the
 *                     memmap / h5py dtype (bin/phyloligo.py:720,777-786), or NULL
 * A record with no countable word gives an all-zero row (bin/phyloligo.py:660).
 */
int po_profile_batch(const uint8_t* d_text, const int64_t* d_begin, const int64_t* d_end,
                     int64_t n, const char* pattern, int strand,
                     uint32_t* d_counts, uint64_t* d_totals,
                     double* d_freq64, float* d_freq32, po_stream_t stream);

/*
 * Size in bytes of the prepared operand buffer (the layout po_distance_block consumes)
 * of n profiles of dimension `dim` for `metric`; the caller allocates it.
 *   Eucl / BC : n rows of dim rounded up to a multiple of 4, float32
 *   EuclGram  : centred operand blocks for the tensor-core kernel (n rounded up to 128, dim to 64,
 *               4 bytes per element: the float16 hi part, and hi and lo once more as e4m3 for the
 *               cross terms -- or float16 hi and lo below 1024 dimensions / with PO_EUCL_CROSS=f16), float64 column sums, a
 *               float32 copy of the profiles for the exact recomputation of cancelling entries, and
 *               the e4m3 scales
 *   SC        : 64 <= dim <= 4096: the centred doubled average ranks 2 rank - (dim+1) as two int8
 *               digits (r = 128 h + l; PO_SC_DIGITS=f16: two float16 digits, r = 64 h + l) in the
 *               tensor-core block layout (n rounded up to 128, dim to 64; the buffer is sized for the
 *               float16 form, 4 bytes per element) -- Spearman runs on the tensor cores, exactly;
 *               otherwise n rows of dim (rounded up to 4) int32 ranks for the CUDA-core kernel
 *   KT        : n rows of packed order-relation bit masks, 2 * ceil(dim(dim-1)/2 / 128) * 16 bytes
 *   JSD       : float32 with exact zeros biased to 1e-30, dim rounded up to a multiple of 32
 *               and n to a multiple of 64, stored as bulk-copy blocks: [n/64][dim/32] blocks
 *               of [32 dims][64 profiles], then [n/32][dim/32] blocks of
 *               [32 dims][32 profiles]
 * po_prepared_row_bytes is the per-profile figure of the row-major layouts (Eucl, BC, KT, and
 * the CUDA-core SC layout); the blocked layouts (JSD, EuclGram, tensor-core SC) are padded to
 * whole groups of profiles -- use po_prepared_bytes.
 */
int64_t po_prepared_bytes(int metric, int64_t n, int64_t dim);
int64_t po_prepared_row_bytes(int metric, int64_t dim);

/*
 * Prepare the operand matrix for a metric from raw profiles.
 *   d_X       [n x ldx] profiles, float32 or float64 (`dtype`), ldx in elements
 *   d_P       po_prepared_bytes(metric, n, dim) bytes of prepared operands (written), 16-byte aligned
 *   d_aux     [n] float64 per-row constant (written):
 *               Eucl (tensor-core path): squared norm of the centred, scaled row
 *               SC: sum of squares of the centred doubled ranks (0 = constant row)
 *               KT: number of element pairs that are not tied in the row
 *               others: unused (may be NULL)
 * Eucl/JSD/BC: a float32 copy, zero padded.  SC: rank transform with average
 * ranks for ties -- the scipy.stats.spearmanr step of phylodist.SC
 * (core/phylodist.py:82-85).  KT: the per-row half of Bio.Cluster's kendall()
 * loop (core/phylodist.py:71-74): which element pairs are ordered up / down.
 */
int po_prepare_profiles(int metric, const void* d_X, int dtype, int64_t n, int64_t dim, int64_t ldx,
                        void* d_P, double* d_aux, po_stream_t stream);

/*
 * Rank transform of every profile: average ranks 1..dim, ties sharing the mean of their positions --
 * the scipy.stats.spearmanr / rankdata step of phylodist.SC (core/phylodist.py:82-85) as a stand-alone
 * call.  d_X is [n x dim] float32 / float64 with row pitch ldx, d_ranks [n x dim] float64 with row
 * pitch ldr.  (po_prepare_profiles(PO_SC) runs the same transform and stores it in the layout the
 * tile kernels read.)
 */
int po_rank_transform(const void* d_X, int dtype, int64_t n, int64_t dim, int64_t ldx, double* d_ranks,
                      int64_t ldr, po_stream_t stream);

/*
 * One block of the all-by-all distance matrix -- replaces the slice workers
 * distances_loc / *_loc (bin/phyloligo.py:195-222), distances_h5py / *_h5py
 * (:233-301), compute_unpack (:166-171) and the phylodist pair functions Eucl,
 * JSD, KT, BC, SC (core/phylodist.py:36-85):
 *
 *   out[(r - out_row0) * ld_out + (c - out_col0)] = metric(profile r, profile c)
 *   for r in [row0, row1), c in [col0, col1).
 *
 *   d_P, d_aux   prepared operands of all n rows (po_prepare_profiles)
 *   out_dtype    PO_F32 (the --large dtypes) or PO_F64 (the --large None dtype)
 *   flags        PO_FLAG_SKIP_LOWER / PO_FLAG_MIRROR exploit symmetry when the
 *                caller's `out` addresses the full matrix (mirrored entries
 *                (c, r) must be addressable).
 * Values: Eucl = sqrt(sum (a-b)^2) (PO_EUCL_GRAM: Gram form on the tensor cores, exact 0 on the
 * diagonal, stated tolerance 1e-4 relative, measured <= 5e-6); JSD in nats (core/phylodist.py:22), 0 for
 * identical rows, ln(2)/2 against an all-zero row; BC = sum|a-b| / sum|a+b|;
 * KT = 1 - (1 - tau_b) (tau_b itself; 0 when a row is constant); SC = 1 - rho
 * (NaN when a row is constant).
 */
int po_distance_block(int metric, const void* d_P, const double* d_aux, int64_t n, int64_t dim,
                      int64_t row0, int64_t row1, int64_t col0, int64_t col1,
                      void* d_out, int64_t ld_out, int64_t out_row0, int64_t out_col0,
                      int out_dtype, unsigned flags, po_stream_t stream);

/*
 * The same block with the mirrored tiles written to a second buffer instead of `d_out`:
 *   mirror[(c - mirror_row0) * ld_mirror + (r - mirror_col0)] = metric(profile r, profile c)
 * for every tile that PO_FLAG_MIRROR mirrors.  This is the multi-GPU form of the
 * reference's block-row split (gen_even_slices over rows, bin/phyloligo.py:424,516): a
 * rank computes only the part of its block row that lies right of the diagonal and
 * hands the transposed blocks to the ranks that own those columns as rows.
 */
int po_distance_block_ex(int metric, const void* d_P, const double* d_aux, int64_t n, int64_t dim,
                         int64_t row0, int64_t row1, int64_t col0, int64_t col1,
                         void* d_out, int64_t ld_out, int64_t out_row0, int64_t out_col0,
                         void* d_mirror, int64_t ld_mirror, int64_t mirror_row0, int64_t mirror_col0,
                         int out_dtype, unsigned flags, po_stream_t stream);

/*
 * Peer memory for the multi-GPU distance stage (one process per GPU on one node).  A rank
 * exports the buffer that holds its block rows; the other ranks open it and pass the peer
 * address as `d_mirror` of po_distance_block_ex, so that the transposed off-diagonal tiles are
 * stored straight into their owner's rows over NVLink while the tile kernel runs -- the exchange
 * step costs no staging buffer and no separate transfer.
 *   po_ipc_export : 64-byte CUDA IPC handle of the allocation containing d_ptr, and d_ptr's offset in it
 *   po_ipc_open   : map a peer's allocation into this process (peer access is enabled lazily)
 *   po_ipc_close  : unmap it
 */
int po_ipc_export(const void* d_ptr, void* h_handle64, int64_t* offset);
int po_ipc_open(const void* h_handle64, void** d_base);
int po_ipc_close(void* d_base);

/*
 * Kount.py's sliding-window stage (bin/Kount.py:274-453).  Every window of every contig is a
 * virtual record of po_profile_batch (d_begin / d_end = the window's byte range in a text whose
 * sequences carry no line breaks).  Two small per-window kernels complete it:
 *   po_window_count_byte  occurrences of one byte value in every window -- the
 *                         seq.count('N') / len(seq) <= n_max_freq_in_windows filter (:294)
 *   po_window_distances   distance of every window profile (float64 [n x dim], row pitch ld) to ONE
 *                         reference profile d_ref[dim], float64 out[n]: the 1-D forms dispatched by
 *                         compute_distance_joblib (:317-324).  metric 0 = JSD (:94-123, x1000),
 *                         1 = KL (:71-86), 2 = Eucl (:88-92, x1000); NaN / Inf terms are zeroed
 *                         term by term (posdef_check_value, :67-69).
 */
enum po_window_metric { PO_W_JSD = 0, PO_W_KL = 1, PO_W_EUCL = 2 };
int po_window_count_byte(const uint8_t* d_text, const int64_t* d_begin, const int64_t* d_end, int64_t n,
                         int value, int64_t* d_counts, po_stream_t stream);
int po_window_distances(int metric, const double* d_freq, int64_t n, int64_t dim, int64_t ld,
                        const double* d_ref, double* d_out, po_stream_t stream);

/*
 * Strided block copy between any two of device / pinned host memory (one DMA, no staging):
 * `rows` rows of `width` bytes, row pitches in bytes.  This is how finished parts of the matrix
 * leave the device -- the row slices output[s] = ... of the reference's block-row workers
 * (bin/phyloligo.py:202, 207, 212, 217, 222) -- without waiting for whole rows: a row panel's
 * part right of the diagonal and the mirrored column block below it are both final as soon as
 * the panel's tiles are done.  Asynchronous on `stream` when the host side is pinned.
 */
int po_copy2d_async(void* dst, int64_t dst_pitch, const void* src, int64_t src_pitch, int64_t width,
                    int64_t rows, po_stream_t stream);

/*
 * Text matrix writer on the host -- replaces np.savetxt(path, M, delimiter="\t") at
 * bin/phyloligo.py:1059-1066 (the -o distance matrix and the -q frequency file): "%.18e"
 * fields of the float64 value of every entry, tab separated, '\n' rows, no header; nan / inf /
 * -inf spelled as Python spells them.  h_data is a host matrix [rows x cols], row pitch ld
 * elements, dtype PO_F32 or PO_F64.  Row blocks are formatted by `threads` host threads
 * (<= 0 picks the hardware concurrency) and written in order.
 */
int po_savetxt_host(const char* path, const void* h_data, int64_t rows, int64_t cols, int64_t ld,
                    int dtype, int threads);

/*
 * The host end of the output path.  The reference's --large workers assign their block row into
 * the caller's mapping of the output file (output[s] = ..., bin/phyloligo.py:202-222 into the
 * np.memmap of :413-425, or the 'distances' dataset of the HDF5 file, :471-478).  Here block
 * rows leave the device by DMA (po_copy2d_async), and these calls make the caller's mapping a
 * DMA target or move finished panels into it with host threads.  All pointers are HOST pointers;
 * `threads` <= 0 picks the hardware concurrency.
 *   po_host_prefault      instantiate the pages of [h_ptr, h_ptr + bytes) for writing (parallel
 *                         madvise(MADV_POPULATE_WRITE); touches every page on kernels without it)
 *   po_host_premap        map the pages of a shared mapping of an EXISTING file (descriptor fd) ahead of the
 *                         writes: on tmpfs by populating for reading (fault-around maps 16 up-to-date pages per
 *                         fault and the entries are writable at once: 27-43 GB/s against 2-3 GB/s per thread),
 *                         elsewhere like po_host_prefault
 *   po_host_register      page-lock an existing mapping (cudaHostRegister, portable) so that
 *                         po_copy2d_async DMAs straight into it; fails with PO_ERR_CUDA when the
 *                         kernel refuses to pin the pages (file systems with dirty tracking)
 *   po_host_unregister    undo it (before munmap)
 *   po_host_copy2d        strided block copy host -> host on `threads` threads (pinned panel ->
 *                         mapping of the output file)
 *   po_host_pwrite2d      the same through pwrite(fd, ...) at file_offset with row pitch file_pitch
 *                         (no page faults, no mapping needed)
 *   po_host_pread         read `bytes` bytes at file_offset of fd into h_dst with `threads` parallel
 *                         pread calls: how the FASTA text reaches the pinned staging ring (the
 *                         SeqIO.parse(genome, "fasta") reads of bin/phyloligo.py:869, 914, 959)
 *   po_host_transpose_f32 h_dst[c * ld_dst + r] = h_src[r * ld_src + c], float32: the mirrored block
 *                         of a block that has already arrived (the matrix is symmetric), so that only
 *                         the part on and right of the diagonal needs to cross PCIe
 *   po_host_mirror_*      the same, asynchronous and in stream order: _open starts a pool of host threads
 *                         (NULL on failure); _submit queues one block -- with after_stream != 0 the block is
 *                         released to the pool by a host callback once everything enqueued on `stream`
 *                         before the call (the DMA that brings h_src) has completed, with 0 at once; _wait
 *                         blocks until every submitted block is written; _close waits, then joins the pool.
 *                         The reference assigns every entry of its block row (output[s] = ...,
 *                         bin/phyloligo.py:202-222); this is how the entries left of the diagonal get there
 *                         without crossing PCIe.
 */
int po_host_prefault(void* h_ptr, int64_t bytes, int threads);
int po_host_premap(int fd, void* h_ptr, int64_t bytes, int threads);
int po_host_register(void* h_ptr, int64_t bytes);
int po_host_unregister(void* h_ptr);
int po_host_copy2d(void* h_dst, int64_t dst_pitch, const void* h_src, int64_t src_pitch, int64_t width,
                   int64_t rows, int threads);
int po_host_pwrite2d(int fd, int64_t file_offset, int64_t file_pitch, const void* h_src, int64_t src_pitch,
                     int64_t width, int64_t rows, int threads);
int po_host_pread(int fd, int64_t file_offset, void* h_dst, int64_t bytes, int threads);
int po_host_transpose_f32(float* h_dst, int64_t ld_dst, const float* h_src, int64_t ld_src, int64_t rows,
                          int64_t cols, int threads);
void* po_host_mirror_open(int threads);
int po_host_mirror_submit(void* h_pool, po_stream_t stream, int after_stream, float* h_dst, int64_t ld_dst,
                          const float* h_src, int64_t ld_src, int64_t rows, int64_t cols);
int po_host_mirror_wait(void* h_pool);
int po_host_mirror_close(void* h_pool);

/*
 * The front half of phyloselect.py (bin/phyloselect.py) on the device: what its K-medoids loop and
 * its nearest-neighbour consumers read out of the N x N matrix, while the matrix (or a block row of it,
 * [n_rows x n_cols] with row pitch ld, PO_F32 or PO_F64) is resident in device memory.
 *   po_matrix_rowsums      d_out[i] = sum_j D[row(i), j] in float64 -- np.sum(D, axis=1) of the medoid
 *                          heuristic (:291-309); row(i) = d_rows[i] or i when d_rows is NULL.  With
 *                          d_labels (int32 per column) and d_row_labels (int32 per output row) the sum
 *                          runs over the columns j with d_labels[j] == d_row_labels[i] only: the
 *                          within-cluster cost of every member and of the current medoids (:197-240)
 *   po_matrix_argmin_rows  d_out[j] = argmin_c D[d_rows[c], j], first minimum on ties --
 *                          np.argmin(D[medoid_ics, :], axis=0) (:187-195)
 *   po_cluster_argmin      per cluster c < k: d_count[c] members, d_best_cost[c] = the smallest d_cost
 *                          among them and d_best_idx[c] = the first member that has it (-1 for an empty
 *                          cluster) -- np.argmin(all_costs) over the members in index order (:224-227);
 *                          d_work: 16 k bytes of scratch
 *   po_matrix_knn          the k (<= 1024) nearest neighbours of every row, ascending distance, ties by
 *                          column, the row's own column (self0 + i) excluded -- what sklearn's
 *                          kneighbors_graph(mode="distance") gives TSNE / HDBSCAN on a precomputed matrix
 *                          (:381-428); d_idx int32 [n_rows x k], d_dist float32 [n_rows x k]
 */
int po_matrix_rowsums(const void* d_D, int64_t ld, int dtype, const int64_t* d_rows, int64_t n_rows, int64_t n_cols,
                      const int* d_labels, const int* d_row_labels, double* d_out, po_stream_t stream);
int po_matrix_argmin_rows(const void* d_D, int64_t ld, int dtype, const int64_t* d_rows, int k, int64_t n_cols, int* d_out,
                          po_stream_t stream);
int po_cluster_argmin(const double* d_cost, const int* d_labels, int64_t n, int k, void* d_work, int64_t* d_best_idx,
                      double* d_best_cost, int64_t* d_count, po_stream_t stream);
int po_matrix_knn(const void* d_D, int64_t ld, int dtype, int64_t n_rows, int64_t n_cols, int64_t self0, int k, int* d_idx,
                  float* d_dist, po_stream_t stream);

/*
 * HDBSCAN on the resident matrix: what find_clusters (:403-428) gets from
 * hdbscan.HDBSCAN(min_cluster_size, min_samples, metric="precomputed"), every other argument at its default.
 * MST edges compare by the triple (mutual reachability, min(i, j), max(i, j)); the MST is then unique.
 *   po_hdbscan_check         refuses (PO_ERR_ARG) a matrix that is not square, not bitwise symmetric or holds a
 *                            NaN or an infinite entry; the message names the first offending entry in row-major
 *                            order.  d_work: 8 bytes.  Synchronises `stream`.  With ld_cols = 0 (row0 = 0, d_cols
 *                            NULL), d_D is the whole matrix.  With ld_cols > 0, d_D is the row panel [row0, row0 +
 *                            n_rows) x [0, n_cols) of an n_cols x n_cols matrix, and entry (i, j) is compared with
 *                            (j, i) taken from d_cols, the column strip [0, n_cols) x [row0, row0 + n_rows) with row
 *                            pitch ld_cols; with d_cols NULL (a source symmetric by construction) only the panel's
 *                            diagonal square is tested for symmetry.  Checked panel by panel in row order, the first
 *                            panel that fails names the entry the whole-matrix check names.
 *   po_matrix_kth            d_out[i] = the k-th smallest (1-based) entry of row i, every column counted (the
 *                            diagonal too), bit for bit in the matrix's dtype: the core distances, k =
 *                            min_samples + 1 (contrib's np.partition(D, min_samples, axis=0)[min_samples] in
 *                            mutual_reachability)
 *   po_hdbscan_mst_workspace bytes of d_work the three entries below need for n points
 *   po_hdbscan_mst_init      n singleton components in d_work
 *   po_hdbscan_mst_scan      the pass of one Boruvka round over the rows [row0, row0 + n_rows) of the matrix, held in
 *                            d_D (row pitch ld, n columns): every row's lightest edge to another component under
 *                            mr(i, j) = max(core_i, core_j, D[i, j]), computed on the fly and never stored
 *                            (replaces contrib's mutual_reachability and mst_linkage_core).  A round scans every
 *                            row once, in one call or in row panels, then merges.
 *   po_hdbscan_mst_merge     the rest of the round: per-component reduction, hooking and pointer jumping.  Appends
 *                            the new edges to d_u, d_v (int64) and d_w (dtype), n - 1 entries each over all rounds,
 *                            in no particular order; *h_components = components left (1 when done).  Reads two
 *                            counters to the host (synchronises `stream`).
 *   po_hdbscan_tree          host: sorts the n - 1 MST edges in place by the tie rule (u < v), then contrib's
 *                            label (single-linkage rows sl_*: left, right, distance, size), condense_tree
 *                            (ct_*: parent, child, lambda_val, child_size; up to 2 n rows, *ct_rows written),
 *                            compute_stability, get_clusters (excess of mass, allow_single_cluster=False) and
 *                            get_probabilities: labels (-1 = noise; clusters numbered in ascending condensed-tree
 *                            id) and probabilities.  O(N log N).
 */
int po_hdbscan_check(const void* d_D, int64_t ld, int dtype, int64_t n_rows, int64_t n_cols, int64_t row0, const void* d_cols,
                     int64_t ld_cols, void* d_work, po_stream_t stream);
int po_matrix_kth(const void* d_D, int64_t ld, int dtype, int64_t n_rows, int64_t n_cols, int k, void* d_out, po_stream_t stream);
int64_t po_hdbscan_mst_workspace(int64_t n);
int po_hdbscan_mst_init(int64_t n, void* d_work, po_stream_t stream);
int po_hdbscan_mst_scan(const void* d_D, int64_t ld, int dtype, int64_t row0, int64_t n_rows, int64_t n, const void* d_core,
                        void* d_work, po_stream_t stream);
int po_hdbscan_mst_merge(int64_t n, int dtype, const void* d_core, void* d_work, int64_t* d_u, int64_t* d_v, void* d_w,
                         int64_t* h_components, po_stream_t stream);
int po_hdbscan_tree(int64_t n, int64_t min_cluster_size, int64_t* u, int64_t* v, double* w, int64_t* sl_left, int64_t* sl_right,
                    double* sl_dist, int64_t* sl_size, int64_t* ct_parent, int64_t* ct_child, double* ct_lambda, int64_t* ct_size,
                    int64_t* ct_rows, int64_t* labels, double* probabilities);

/*
 * t-SNE on the resident matrix: what sklearn.manifold.TSNE(metric="precomputed", method="barnes_hut", angle=0.0)
 * computes for the reference's -t projection (:381-398).  With angle 0 scikit-learn's Barnes-Hut gradient is the
 * exact gradient of the sparse-P objective; these entries evaluate it exactly.  Sums run in a fixed order.
 *   po_tsne_check            refuses (PO_ERR_ARG) a matrix holding a NaN, an infinite or a negative entry
 *                            (check_array / check_non_negative); the message names the first in row-major order.
 *                            d_D holds the rows [row0, row0 + n_rows) (row0 = 0: the whole matrix); the message
 *                            names the absolute entry.  d_work: 8 bytes.  Synchronises `stream`.
 *   po_tsne_conditional      _binary_search_perplexity over the k neighbours d_idx [n x k] (po_matrix_knn) of
 *                            every row: squared distances D[i, idx]^2 in the matrix's dtype, then float32; the
 *                            search in float64 (tolerance 1e-5 on the entropy, at most 100 steps).  d_P float64
 *                            [n x k], each row summing to 1 (0 where every exp underflows)
 *   po_tsne_sum              *d_out = sum of d_x[0 .. n) in float64 in a fixed order (one CTA)
 *   po_tsne_workspace        bytes of d_work the two entries below need for n points
 *   po_tsne_repulsion        the exact all-pairs pass over the positions d_Y (float32 [n x 2]): per row
 *                            sum_j q_ij^2 (y_i - y_j) and Z = sum_{i != j} q_ij, q_ij = 1 / (1 + |y_i - y_j|^2),
 *                            kept in d_work for the step
 *   po_tsne_attraction_step  per row the CSR walk sum_j p_ij q_ij (y_i - y_j), p_ij = float32((P_ij * mul) * r),
 *                            r = 1.0 / div (scipy's in-place P /= div multiplies by the reciprocal), and the gradient 4 (attraction - repulsion / Z) of the positions the last
 *                            po_tsne_repulsion saw.  d_grad (optional, float32 [n x 2]) receives it.  With d_Y_next
 *                            one _gradient_descent step: gains (+0.2 / x0.8, at least 0.01, float32), update =
 *                            momentum update - learning_rate grad gains (float64 when update64, else float32 as
 *                            scikit-learn's arithmetic with a float32 learning rate), d_Y_next = d_Y + update.
 *                            With h_kl_gradnorm2 the KL divergence sum p_ij log(max(p_ij, tiny) / max(q_ij / Z,
 *                            tiny)) and |grad gains|^2 are reduced and copied to h_kl_gradnorm2[0..1]
 *                            (synchronises `stream`).
 */
int po_tsne_check(const void* d_D, int64_t ld, int dtype, int64_t n_rows, int64_t n_cols, int64_t row0, void* d_work,
                  po_stream_t stream);
int po_tsne_conditional(const void* d_D, int64_t ld, int dtype, int64_t n, const int* d_idx, int k, double perplexity, double* d_P,
                        po_stream_t stream);
int po_tsne_sum(const double* d_x, int64_t n, double* d_out, po_stream_t stream);
int64_t po_tsne_workspace(int64_t n);
int po_tsne_repulsion(const float* d_Y, int64_t n, void* d_work, po_stream_t stream);
int po_tsne_attraction_step(const int64_t* d_indptr, const int* d_indices, const double* d_P, int64_t n, double mul, double div,
                            const float* d_Y, void* d_work, float* d_Y_next, double* d_update, float* d_gains, float* d_grad,
                            double momentum, double learning_rate, int update64, double* h_kl_gradnorm2, po_stream_t stream);

/*
 * Hierarchical clustering of the resident matrix: the tree phyloselect.R builds with hclust (:22-35), computed
 * as scipy.cluster.hierarchy.linkage(squareform(D, checks=False), method) computes it, bit for bit.
 * method: 0 single, 1 complete, 2 average, 3 weighted, 4 ward.
 *   po_linkage_workspace     bytes of d_work po_linkage_run needs for n points
 *   po_linkage_run           one persistent cooperative launch (one CTA per SM at most, steps separated by
 *                            grid.sync()).  single: scipy's mst_single_linkage (Prim from vertex 0) on d_D in
 *                            place, n - 1 steps.  Otherwise scipy's nn_chain on d_W, a float64 n x n working copy
 *                            of d_D (row stride n) that this call fills: every scan takes the minimum of the tip's
 *                            row (smallest index on ties; the chain's previous entry when it holds the minimum),
 *                            every merge applies the Lance-Williams update to row y and column y in float64 without
 *                            FMA contraction.  At most 3 (n - 1) scans: past that bound the launch stops and the
 *                            call fails.  Writes the n - 1 raw merges (d_zx, d_zy, d_zh: x, y, height) in merge
 *                            order and *h_phases = the number of grid barriers.  d_D is read only; it must be
 *                            finite and symmetric (po_hdbscan_check).  Synchronises `stream`.
 *   po_linkage_tree          host: the stable sort of the raw merges by height (NaN last; numpy's mergesort
 *                            argsort) and scipy's label (union-find, new clusters n, n + 1, ...) into Z, the
 *                            row-major (n - 1) x 4 float64 linkage matrix
 */
int64_t po_linkage_workspace(int64_t n);
int po_linkage_run(const void* d_D, int64_t ld, int dtype, int64_t n, int method, double* d_W, void* d_work, int64_t* d_zx,
                   int64_t* d_zy, double* d_zh, int64_t* h_phases, po_stream_t stream);
int po_linkage_tree(int64_t n, const int64_t* zx, const int64_t* zy, const double* zh, double* Z);

/*
 * Neighbour-joining trees of the resident matrix: the NJ and BIONJ trees phyloselect.R builds with ape's nj / bionj
 * (:22-35), bit for bit in the order of float64 operations DESIGN.md section 4.11 fixes (agreement with ape itself
 * is not pinned).
 * method: 0 NJ, 1 BIONJ.
 *   po_nj_capacity     C, the slots per side of the working state for n points (n plus a front headroom, rounded up
 *                      to 32)
 *   po_nj_workspace    bytes of d_work po_nj_run needs for n points
 *   po_nj_stage_bytes  bytes of d_stage po_nj_run needs for n points (the compaction's staging rows, <= 256 MB)
 *   po_nj_run          n - 3 joins, each four launches on `stream` (row sums, Q scan, decision, update) with no host
 *                      synchronisation in between, then the three root edges.  d_W is the float64 C x C working state
 *                      (8 C^2 bytes) that this call fills from d_D: D above the diagonal, BIONJ's variance below it.
 *                      Writes d_edge (int64, (2n - 3) x 2, (parent, child)) and d_length (float64, 2n - 3) in ape's
 *                      numbering from 0 (leaves 0 .. n-1, root n, the node of join t 2n - 3 - t), the rows in join
 *                      order, and *h_compactions = how often the live block was packed.  d_D is read only; it must be
 *                      finite and symmetric (po_hdbscan_check).  Fails with PO_ERR_ARG when a join finds no pair whose
 *                      Q is below 1e50.  Synchronises `stream`.
 */
int64_t po_nj_capacity(int64_t n);
int64_t po_nj_workspace(int64_t n);
int64_t po_nj_stage_bytes(int64_t n);
int po_nj_run(const void* d_D, int64_t ld, int dtype, int64_t n, int method, double* d_W, void* d_stage, void* d_work,
              int64_t* d_edge, double* d_length, int64_t* h_compactions, po_stream_t stream);

/* Number of kernels this library has launched since load (for bench.py's gpu_launches). */
int64_t po_launch_count(void);

/* Average device time (ms) of the launches of one kernel family since the last
 * po_timing_reset(): CUDA events recorded on the launching stream around each
 * launch while timing is enabled.  family: 0 = profiling, 1 = distance tile, 2 = the linkage kernels'
 * cooperative launch (po_linkage_run), 3 = the launches of one po_nj_run, first to last. */
int po_timing_enable(int on);
int po_timing_reset(void);
int po_timing_read(int family, double* total_ms, int64_t* launches);

/* Pipe-peak microbenchmark for roofline denominators that MEASURED_PEAKS.json lacks.
 * kind 0: FP32 FFMA TFLOP/s, 1: MUFU.LG2 1e12 op/s, 2: POPC 1e12 op/s, 3: MUFU.RCP 1e12 op/s (best of 4 timed runs),
 * 4: microseconds per grid.sync() of the linkage kernels' grid (least of 4 timed runs),
 * 5..12: warp-instructions per SM per clock of packed-f32x2 operand forms (csrc/po_microbench.cu; best of 4). */
int po_microbench(int kind, double* result);

#ifdef __cplusplus
}
#endif
#endif /* PHYLOLIGO_B200_H */
