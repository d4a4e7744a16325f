/*
 * spmm_b200.h — C-ABI of the B200-native sparse-matrix x fat-vector path.
 *
 * Drop-in boundary for AlexisBalayre/SparseMatrixMultiplicationMPI's one hot
 * path (C = A*B, A CSR FP64/int32, B dense N x k FP64). Plain pointers and
 * sizes only; every function returns an spmm_status and records a message
 * readable through spmm_last_error() (thread-local). No function falls back
 * to the CPU: without a CUDA device they fail with SPMM_ERR_CUDA.
 *
 * Each entry cites the reference interface it replaces; paths are relative to
 * /root/reference/"Source Code"/. Dense operands are flat row-major, the
 * layout of the reference's serialize() (utils.cpp:216-228). "d_" arguments
 * are device pointers on the handle's device; all others are host pointers.
 * `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 * Device multiplies of one handle may be enqueued on different streams: the scratch a launch writes on the handle (the
 * merge kernel's carry rows) is ordered across streams by the library; the operands B and C are the caller's to order.
 * One handle must not be used from several host threads at once (AUTO's lazy tile layout and the CTA-cut cache are
 * updated without a lock); the host-buffer forms alone serialize themselves.
 */
#ifndef SPMM_B200_H
#define SPMM_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct spmm_csr_s *spmm_csr_t; /* device-resident SparseMatrix (MatrixDefinitions.h:14-19) */

enum spmm_status
{
    SPMM_OK = 0,
    SPMM_ERR_INVALID = 1,     /* bad argument (the reference checks nothing; we do) */
    SPMM_ERR_CUDA = 2,        /* CUDA runtime error or no device */
    SPMM_ERR_NOMEM = 3,
    SPMM_ERR_UNSUPPORTED = 4
};

/* Kernel families (DESIGN.md §kernels). AUTO picks from the handle's row-length schedule. */
enum spmm_kernel
{
    SPMM_KERNEL_AUTO = 0,
    SPMM_KERNEL_ROWS = 1,  /* (sub-)warp-per-row teams over contiguous row chunks */
    SPMM_KERNEL_MERGE = 2, /* nnz-balanced merge-path with deterministic carry fix-up */
    /* ids 3, 4, 5 and 7 belonged to experimental layouts that never won a regime (profiles/r1_union.md); retired */
    SPMM_KERNEL_TILED = 6,    /* row tiles whose B rows are staged in shared memory by TMA (needs spmm_csr_build_tiles; even k) */
    SPMM_KERNEL_STREAM = 8,   /* k = 1, 2, 4, 8: CSR arrays streamed in nnz order, rows reduced from shared memory; bit-identical to the reference's mul-then-add (spmm_stream.cu) */
    SPMM_KERNEL_BSR = 9       /* b x b dense blocks: a team per block row loads each B row piece once for the b rows (needs spmm_csr_build_bsr; spmm_bsr.cu) */
};

const char *spmm_last_error(void);
/* Name of the kernel family the calling thread's last multiply launched ("spmm_tiled_kernel", "spmm_rows_kernel",
 * "spmm_merge_kernel", "spmm_stream_kernel", "spmm_bsr_kernel"; "" before the first launch): what AUTO chose, for
 * measurement reports. */
const char *spmm_last_kernel_name(void);
int spmm_version(void);
int spmm_device_count(int *count);
/* multiProcessorCount, L2 bytes, total global memory of `device` */
int spmm_device_info(int device, int *sm_count, long long *l2_bytes, long long *hbm_bytes);

/* ---- a1: SparseMatrix in HBM ------------------------------------------------------ */

/* Upload a host CSR (the SparseMatrix fields values/colIndices/rowPtr + numRows/numCols,
 * MatrixDefinitions.h:14-19, utils.cpp:180-181) to `device` and build its row-length
 * schedule. Arrays are copied bit-for-bit; the host arrays are not retained. */
int spmm_csr_create_host(int device, int n_rows, int n_cols, long long nnz,
                         const int *rowptr, const int *colidx, const double *vals,
                         spmm_csr_t *out);

/* Same from arrays already on `device`. copy=0 borrows them (caller keeps them alive). */
int spmm_csr_create_device(int device, int n_rows, int n_cols, long long nnz,
                           const int *d_rowptr, const int *d_colidx, const double *d_vals,
                           int copy, spmm_csr_t *out);

/* More than 2^31 - 1 stored entries: 64-bit row offsets (rowptr[n_rows+1] as long long); colidx / vals as above.
 * Not part of the reference's data model (its rowPtr is int32); every other call keeps its int32 meaning.
 * Checks as the 32-bit entries: rowptr[0] == 0, rowptr[n_rows] == nnz, non-NULL arrays (else SPMM_ERR_INVALID); a row of
 * more than 2^31 - 1 entries (possible only with duplicates) is SPMM_ERR_UNSUPPORTED. The rows are cut into segments of at
 * most 2^30 non-zeros each (a longer row is a segment of its own), found on the device when the handle is created; each
 * segment keeps a rebased int32 copy of its row pointer (4 bytes per row in all) and borrows its slices of colidx / vals.
 * _device64 with copy=0 borrows the three arrays as spmm_csr_create_device does; a caller who changes the pattern must
 * create the handle again.
 * On such a handle (DESIGN.md section 4.8):
 *   - every device multiply form runs the int32 kernels segment after segment on the caller's stream, and so do the host
 *     forms built on them; AUTO decides per segment from that segment's schedule (merge-path, the stream kernel at k = 1
 *     from stream.min_nnz non-zeros, else the row kernel) and never builds a tile layout;
 *   - ROWS, MERGE and STREAM run on every segment (STREAM checks its shape per segment, before anything is launched, and
 *     stays bit-identical to the reference); TILED and BSR are SPMM_ERR_UNSUPPORTED; other ids as on int32 handles;
 *   - spmm_csr_build_tiles(_for_k), spmm_csr_build_bsr, spmm_csr_column_block, spmm_csr_device_ptrs and
 *     spmm_csr_download are SPMM_ERR_UNSUPPORTED (the last two: use the 64-bit forms below);
 *   - spmm_csr_info, spmm_csr_schedule (bins summed over the segments, global maximum and mean, auto_kernel merge-path if
 *     any segment picked it), spmm_csr_column_span, spmm_nnz_range_rows, spmm_csr_update_values_host / _device and
 *     spmm_csr_destroy work as on int32 handles. */
int spmm_csr_create_host64(int device, int n_rows, int n_cols, long long nnz,
                           const long long *rowptr, const int *colidx, const double *vals,
                           spmm_csr_t *out);
int spmm_csr_create_device64(int device, int n_rows, int n_cols, long long nnz,
                             const long long *d_rowptr, const int *d_colidx, const double *d_vals,
                             int copy, spmm_csr_t *out);
/* The device arrays and the host copy of a handle with 64-bit row offsets (an int32 handle: SPMM_ERR_UNSUPPORTED). */
int spmm_csr_device_ptrs64(spmm_csr_t A, const long long **d_rowptr, const int **d_colidx, const double **d_vals);
int spmm_csr_download64(spmm_csr_t A, long long *rowptr, int *colidx, double *vals);

/* a7: the CSR assembly of readMatrixMarketFile (utils.cpp:124-181) on the device.
 * Input = the file's coordinate records in file order, 0-based. Semantics reproduced
 * bit-exactly: symmetric!=0 mirrors off-diagonal records (:146-152), each row is ordered
 * by (column, value) ascending (:156-159), duplicates are kept, rowPtr is the prefix sum
 * (:162-179). *_host copies the records up first; *_device reads device arrays. */
int spmm_csr_from_coo_host(int device, int n_rows, int n_cols, long long n_entries,
                           const int *rows, const int *cols, const double *vals,
                           int symmetric, spmm_csr_t *out);
int spmm_csr_from_coo_device(int device, int n_rows, int n_cols, long long n_entries,
                             const int *d_rows, const int *d_cols, const double *d_vals,
                             int symmetric, spmm_csr_t *out);

/* Text half of readMatrixMarketFile (utils.cpp:70-153) in native code: comment lines, the size line, then the body as a
 * stream of whitespace-separated tokens (line breaks mean nothing, as with the reference's operator>>), converted by all
 * host threads. Returns malloc'ed 0-based records (free them with spmm_mm_free); *symmetric is set when a comment line
 * contains "symmetric" (:88-91), a "pattern" file gets 1.0 values (:130-133). Errors: the reference's messages
 * "Unable to open file: ", "Failed to read matrix dimensions from file: ", "Failed to read data from file: " (:77,:114,:140)
 * through spmm_last_error(); records outside the declared size (undefined behaviour in the reference) are an error. */
int spmm_mm_read(const char *path, int *n_rows, int *n_cols, long long *n_entries, int *symmetric,
                 int **rows, int **cols, double **vals);
void spmm_mm_free(int *rows, int *cols, double *vals);
/* readMatrixMarketFile end to end: spmm_mm_read + spmm_csr_from_coo_host (utils.cpp:70-185). */
int spmm_csr_from_matrix_market(int device, const char *path, spmm_csr_t *out);

int spmm_csr_destroy(spmm_csr_t A);
int spmm_csr_info(spmm_csr_t A, int *n_rows, int *n_cols, long long *nnz, int *device);
/* Writing through the returned value pointer requires spmm_csr_update_values_device(A, that pointer, stream) before the
 * next multiply: without it the tiled kernel uses the old values (its layout holds a copy of them). The BSR view reads
 * d_vals itself and needs no refresh. A borrowed handle (copy=0) whose caller later changes the column ids keeps a stale
 * tile layout and a stale BSR view: build them again (or drop them) after such a change. */
int spmm_csr_device_ptrs(spmm_csr_t A, const int **d_rowptr, const int **d_colidx, const double **d_vals);
/* New values for the same pattern: vals[nnz] in the handle's CSR order. The schedule, the CTA cuts and the tile
 * layout are kept; the values inside the tile layout are refreshed. Bits are copied (-0.0, NaN payloads survive).
 * Whether the pattern is the same is not checked. nnz == 0: no-op; a NULL pointer otherwise: SPMM_ERR_INVALID.
 * _device: enqueued on `stream`, returns without waiting. d_vals may be A's own value array (the pointer from
 * spmm_csr_device_ptrs, or the caller's array behind a borrowed handle) after it was edited in place: then only the
 * layout is refreshed. A borrowed handle (spmm_csr_create_device with copy=0) accepts no other pointer: the library
 * never writes into memory lent to it as const. Multiplies enqueued later on other streams, the host-buffer forms
 * included, must be ordered after `stream` by the caller; so must the update after earlier multiplies on other streams.
 * _host: through the handle's pinned staging and host threads, on the handle's own stream (one host-buffer call per
 * handle at a time); returns when the update is done, so `vals` may be reused. Not for borrowed handles. */
int spmm_csr_update_values_device(spmm_csr_t A, const double *d_vals, void *stream);
int spmm_csr_update_values_host(spmm_csr_t A, const double *vals);
/* Copy the device CSR back (rowptr n_rows+1, colidx nnz, vals nnz) for memcmp-style checks. */
int spmm_csr_download(spmm_csr_t A, int *rowptr, int *colidx, double *vals);
/* Row-length schedule: bins[0..7] = rows with length 0, 1-2, 3-4, 5-8, 9-16, 17-32, 33-256, >256. */
int spmm_csr_schedule(spmm_csr_t A, long long bins[8], int *max_row_len, double *mean_row_len,
                      int *auto_kernel);
/* Optional second layout next to the CSR, the one AUTO prefers for even k >= 4 when neighbouring rows share columns:
 * tiles of rows_per_tile consecutive rows walked in order by one CTA that keeps a window of B-row
 * boxes (box_rows consecutive rows of B each, brought in by one TMA box copy) in shared memory;
 * non-zeros re-encoded as 16-byte records addressing that window, stragglers staged row by row
 * (spmm_tiled.cu, DESIGN.md section 4.5). rows_per_tile: 0 drops it, -1 picks the tile height
 * that stages the fewest B rows among those that fit shared memory (none if no shape fits: the
 * call still succeeds and the CSR kernels stay in charge), else a multiple of 4 in [4,256].
 * box_rows: 0 (= 16), 4, 8, 16 or 32. The CSR arrays are untouched. The reference has no derived
 * layouts; this serves SparseMatrixFatVectorMultiply.cpp:17-28. */
int spmm_csr_build_tiles(spmm_csr_t A, int rows_per_tile, int box_rows);
/* The same, cut for multiplies with k columns the way AUTO does it (8-column k-tile for k <= 8; from k = 32 / 64 the
 * chunks are longer and shared by 2 / 4 CTAs that take one group of k-tiles each). k = 0: as spmm_csr_build_tiles. */
int spmm_csr_build_tiles_for_k(spmm_csr_t A, int rows_per_tile, int box_rows, int k);
/* reuse = non-zeros per B row staged in shared memory (per pass over the matrix); single_fraction =
 * share of the non-zeros whose B row is staged on its own. Zeros when no layout is built. */
int spmm_csr_tile_info(spmm_csr_t A, int *rows_per_tile, int *box_rows, int *window_slots, int *max_records,
                       double *reuse, double *single_fraction);
/* b x b dense blocks (block sparse row) read straight from the CSR arrays: no copy, values are always the handle's d_vals.
 * block_dim: 0 drops the view; 2..6 checks that the pattern is exactly b-blocked (else SPMM_ERR_UNSUPPORTED, message names
 * the first block row that breaks it and why); -1 takes the largest b in 6..2 that fits (none: succeeds with *out_dim = 0).
 * *out_dim (may be NULL) receives the block size in force.
 * Exactly b-blocked: n_rows % b == 0; the b rows of block row R have one length L with L % b == 0; and for every q, t, i
 * colidx[rowptr[R*b+i] + q*b + t] == c_q + t with c_q = colidx[rowptr[R*b] + q*b] and c_q % b == 0 (duplicates, missing
 * entries and unaligned groups fail; empty block rows pass; columns need not be sorted: storage order is kept). Checked
 * by one pass over the CSR on the device. A failed check leaves the view in force unchanged. With a view, AUTO takes
 * SPMM_KERNEL_BSR in spmm_multiply_device / spmm_multiply_strided_device (and the host forms built on them) where it
 * measured faster (DESIGN.md section 4.7) unless the schedule picked merge-path; the row-range, non-zero-range, window and
 * scatter forms refuse SPMM_KERNEL_BSR with SPMM_ERR_UNSUPPORTED. */
int spmm_csr_build_bsr(spmm_csr_t A, int block_dim, int *out_dim);
/* Sub-matrix A[:, col_begin:col_end) with local column ids (column-block strategy,
 * north_star reading of sparseMatrixFatVectorMultiplyColumnWise). Built on the device. */
int spmm_csr_column_block(spmm_csr_t A, int col_begin, int col_end, spmm_csr_t *out);

/* Smallest and largest column id stored in the handle (-> the rows of B a shard reads; 0, -1 when empty). */
int spmm_csr_column_span(spmm_csr_t A, int *min_col, int *max_col);

/* ---- a3: sparseMatrixFatVectorMultiply (SparseMatrixFatVectorMultiply.cpp:11-31) ---- */

/* C[n_rows x k] = A * B[n_cols x k], everything resident on the device.
 * kernel: AUTO, ROWS, MERGE, TILED, STREAM or BSR; any other id is SPMM_ERR_INVALID. */
int spmm_multiply_device(spmm_csr_t A, const double *d_B, int k, double *d_C, int kernel, void *stream);

/* Row-wise strategy with the gather fused into the multiply (RowWise.cpp:36-50 + the MPI_Gatherv of :85-87,
 * or an all-gather): the C rows of this shard (n_rows x k, contiguous) are stored from registers to every one of
 * the n_dst (1..8) destinations — d_C_list[0] usually the local copy, the others peer GPUs' buffers mapped into
 * this process over NVLink (CUDA IPC / symmetric memory), each already offset to the shard's first row.
 * kernel: AUTO, ROWS, MERGE or TILED (BSR: SPMM_ERR_UNSUPPORTED, other ids: SPMM_ERR_INVALID). No NCCL call, no
 * staging copy; the caller synchronises the ranks afterwards (a barrier) before anybody reads its buffer. */
int spmm_multiply_scatter_device(spmm_csr_t A, const double *d_B, int k, int n_dst, double *const *d_C_list,
                                 int kernel, void *stream);

/* Row-wise strategy without replicating B (RowWise.cpp:36-50 reads fatVector[colIndices[j]] only): d_B_window holds the
 * rows [window_first_row, window_first_row + window_rows) of B — the rows this shard's column ids name (see
 * spmm_csr_column_span), e.g. the rank's own rows plus a halo fetched from its neighbours. kernel: AUTO, ROWS or MERGE (BSR:
 * SPMM_ERR_UNSUPPORTED, other ids: SPMM_ERR_INVALID). */
int spmm_multiply_window_device(spmm_csr_t A, const double *d_B_window, int window_first_row, int window_rows, int k,
                                double *d_C, int kernel, void *stream);

/* Strided form: B has leading dimension ldb, C has ldc; columns [k_begin, k_begin+k_count)
 * of B/C are computed (the k-slab split of ColumnWise.cpp:25-48). kernel: as spmm_multiply_device. */
int spmm_multiply_strided_device(spmm_csr_t A, const double *d_B, int ldb, double *d_C, int ldc,
                                 int k_begin, int k_count, int kernel, void *stream);

/* Host-buffer form, the call the C++ entry points make: copies B up, multiplies, copies C back.
 * B: n_cols*k doubles, C: n_rows*k doubles. Operands of 16 MB and more with k >= 32 go in two
 * k-slabs so that the upload of the second overlaps the download of the first (PCIe is full duplex). */
int spmm_multiply_host(spmm_csr_t A, const double *B, int k, double *C, int kernel);

/* a2: the same with the operands in the memory shape of a FatVector (MatrixDefinitions.h:22): B_rows[i] / C_rows[i]
 * point at row i (k doubles each, separately allocated). Pack (serialize(), utils.cpp:216-228) and unpack
 * (deserialize(), :237-253) run on the library's host threads straight into / out of pinned staging memory, chunk by
 * chunk, overlapped with the copies. C_rows must already point at n_rows buffers of k doubles. */
int spmm_multiply_host_rows(spmm_csr_t A, const double *const *B_rows, int k, double *const *C_rows, int kernel);
/* The same, with the result handed to the caller chunk by chunk while later chunks are still on their way down:
 * sink(row_begin, row_end, rows, ctx) receives rows [row_begin, row_end) of C (row-major, leading dimension k) and is
 * called from the library's host threads on disjoint row ranges — the C++ entry points construct the rows of the
 * result FatVector in it (allocation and copy in one pass, SparseMatrixFatVectorMultiply.cpp:15). */
typedef void (*spmm_rows_sink)(int row_begin, int row_end, const double *rows, void *ctx);
int spmm_multiply_host_sink(spmm_csr_t A, const double *const *B_rows, int k, spmm_rows_sink sink, void *ctx, int kernel);
int spmm_host_threads(void); /* size of that host thread pool (env SPMM_HOST_THREADS, default min(cores, 32)) */
/* fn(i, ctx) for i in [0, n) on that pool, the caller taking part; returns when all are done (the entry points use it to
 * allocate the rows of the result FatVector in parallel). */
void spmm_host_parallel_for(int n, void (*fn)(int, void *), void *ctx);

/* ---- a4: row block [row_begin,row_end) (RowWise.cpp:26-50). d_C_local holds
 * (row_end-row_begin) x k, i.e. the rank's localResult before the Gatherv.
 * kernel: AUTO, ROWS or MERGE as named, BSR SPMM_ERR_UNSUPPORTED, any other id runs the row kernel. ---- */
int spmm_multiply_rows_device(spmm_csr_t A, int row_begin, int row_end, const double *d_B, int k,
                              double *d_C_local, int kernel, void *stream);

int spmm_multiply_rows_host(spmm_csr_t A, int row_begin, int row_end, const double *B, int k, double *C_local,
                            int kernel);

/* ---- a6: non-zero range [nnz_begin,nnz_end) (NonZeroElement.cpp:24-67).
 * Rows touched by the range are first_row..last_row; d_C_local holds
 * (last_row-first_row+1) x k and receives, for each of those rows, the sum over
 * the range's elements only (boundary rows are therefore partial sums, to be
 * combined across ranks in rank order). Rows strictly inside get their full value;
 * empty rows inside get zeros. kernel: as spmm_multiply_rows_device. ---- */
int spmm_nnz_range_rows(spmm_csr_t A, long long nnz_begin, long long nnz_end, int *first_row, int *last_row);
int spmm_multiply_nnz_range_device(spmm_csr_t A, long long nnz_begin, long long nnz_end, int first_row, int last_row,
                                   const double *d_B, int k, double *d_C_local, int kernel, void *stream);

int spmm_multiply_nnz_range_host(spmm_csr_t A, long long nnz_begin, long long nnz_end, int first_row, int last_row,
                                 const double *B, int k, double *C_local, int kernel);

/* ---- a5, column-block strategy (north_star reading of ColumnWise.cpp, SURVEY F2): the reduce of the partial C
 * blocks without NCCL. d_out[0..n_elems) = sum over i of d_src_list[i][0..n_elems), added in list order (pass the
 * ranks' partial blocks in ascending rank order: the sum is then reproducible and equals the oracle's rank-order
 * reduce bit for bit). The sources may be peer GPUs' buffers mapped over NVLink; n_elems even; more than 8 sources
 * are added in passes of 8 that continue the same left-to-right sum. ---- */
int spmm_reduce_blocks_device(int device, int n_src, const double *const *d_src_list, long long n_elems,
                              double *d_out, void *stream);

/* ---- strategies whose ranks share one process (compat MPI rank-threads, one GPU per rank): the collectives of
 * RowWise.cpp:85-87, ColumnWise.cpp:82-84 and NonZeroElement.cpp:88 without host buffers. A rank stages only the rows of
 * B its shard reads, multiplies with spmm_multiply_scatter_device storing C rows straight into the root rank's device
 * buffer over NVLink, and the root brings the finished C down once. ---- */
/* Rows [row_begin,row_end) of B (row pointers as in a FatVector) -> the handle's device image of B (n_cols x k, the other
 * rows are left as they are); the copies are enqueued on the handle's own stream, returned in *stream. */
int spmm_stage_b_rows(spmm_csr_t A, const double *const *B_rows, int row_begin, int row_end, int k, const double **d_B,
                      void **stream);
/* A flat row-major host block <-> a device buffer through the handle's pinned staging and the host threads (a pinned
 * block goes straight to the copy engine). Enqueued on `stream` (a stream of A's device); both return when done. */
int spmm_upload_dense(spmm_csr_t A, const double *src, long long n_rows, int k, double *d_dst, void *stream);
int spmm_download_dense(spmm_csr_t A, const double *d_src, long long n_rows, int k, double *dst, void *stream);
int spmm_csr_stream_sync(spmm_csr_t A); /* wait for everything enqueued on the handle's stream */
/* n_rows x k doubles at d_C (on A's device) -> C_rows[i], through A's pinned staging, unpacked by the host threads. */
int spmm_fetch_c_rows(spmm_csr_t A, const double *d_C, int n_rows, int k, double *const *C_rows);
int spmm_fetch_c_sink(spmm_csr_t A, const double *d_C, int n_rows, int k, spmm_rows_sink sink, void *ctx);
/* A device buffer of at least `bytes` that lives until spmm_device_scratch_release (one per (device, slot)). */
int spmm_device_scratch(int device, int slot, long long bytes, void **out);
int spmm_device_scratch_release(void);
/* Let kernels on `device` load from / store to memory of `peer` (cudaDeviceEnablePeerAccess; idempotent). */
int spmm_peer_enable(int device, int peer);
/* d_dst[i] += d_src[i] on `device` (d_src may be peer memory): cut rows of the non-zero strategy, added in rank order. */
int spmm_add_device(int device, double *d_dst, const double *d_src, long long n_elems, void *stream);
/* Device-to-device copy enqueued on a stream of `device`; the two buffers may live on any GPUs of the box (rows a rank
 * owns -> the root's C). */
int spmm_copy_device(int device, void *d_dst, const void *d_src, long long bytes, void *stream);
int spmm_fill_zero_device(int device, void *d_dst, long long bytes, void *stream);
int spmm_device_sync(int device); /* wait for all work enqueued on `device` */
/* Create the CUDA context of every visible device, start the host threads and (enable_peers != 0) enable peer access between
 * all pairs of devices now instead of inside the first multiply: the one-off cost (seconds on an 8-GPU box) belongs to
 * program start (the reference's MPI_Init, main.cpp:14), not to a timed call. Called by libspmm_entry.so when it is loaded. */
int spmm_devices_init(int enable_peers);
/* The same for ONE device (a process that was given one GPU of a multi-process launch leaves the others alone): context, host
 * threads, the page-locked staging arena, and one tiny multiply per kernel module (CUDA loads a module at its first launch). */
int spmm_device_init(int device);

/* ---- partition formulas (bit-for-bit the reference's integer arithmetic) ---- */
void spmm_partition_rows(int n_rows, int n_ranks, int rank, int *begin, int *end);           /* RowWise.cpp:26-29 */
void spmm_partition_cols(int k, int n_ranks, int rank, int *begin, int *end);                /* ColumnWise.cpp:25-28 */
void spmm_partition_nnz(long long nnz, int n_ranks, int rank, long long *begin, long long *end); /* NonZeroElement.cpp:24-39 */

/* ---- a8: host utilities ---- */
/* generateLargeFatVector (utils.cpp:193-209): rand()%100+1 from the never-seeded libc state. */
void spmm_generate_fat_vector(int n, int k, double *out);
/* areMatricesEqual (utils.cpp:38-63): 1 when every |a-b| <= tol. */
int spmm_are_equal(const double *a, const double *b, long long n, double tol);

/* ---- synthetic workloads generated in HBM (bench / large parity cases) ---- */
/* Banded: every row has nnz_per_row distinct ascending columns inside a window of
 * 2*half_bandwidth+1 columns around the diagonal; values in [0.5,1.5). */
int spmm_gen_banded(int device, int n, int nnz_per_row, int half_bandwidth, unsigned long long seed,
                    spmm_csr_t *out);
/* Rows [row_begin,row_end) of the same matrix as a local CSR (row_end-row_begin rows x n
 * columns): bit-identical to those rows of spmm_gen_banded, so every rank of the row-block
 * strategy can generate just its own block (RowWise.cpp:26-29 partition). */
int spmm_gen_banded_rows(int device, int n, int row_begin, int row_end, int nnz_per_row, int half_bandwidth,
                         unsigned long long seed, spmm_csr_t *out);
/* R-MAT (a,b,c,d) edge list of n_edges over 2^scale vertices, duplicates kept, built
 * into CSR by the device CSR build. */
int spmm_gen_rmat(int device, int scale, long long n_edges, double a, double b, double c,
                  unsigned long long seed, spmm_csr_t *out);
/* Dense fill with integers 1..100 (the value range of generateLargeFatVector, utils.cpp:203).
 * Element i of d_out is a function of (seed, first_elem + i) only, so slabs generated
 * separately agree with the whole. */
int spmm_gen_fat_vector_device(int device, double *d_out, long long n_elems, long long first_elem,
                               unsigned long long seed, void *stream);

/* Measurement knob (not needed for correct results): override the automatic team shape.
 * keys: rows.kl rows.nv rows.np rows.unroll rows.vec rows.ctas_per_sm rows.tile rows.prefetch merge.items merge.wave
 *       tiled tiled.thr tiled.chunk tiled.depth tiled.pool tiled.ns tiled.ksplit tiled.group tiled.stride tiled.pdl
 *       tiled.auto_after stream stream.tile stream.kmax stream.min_nnz host.slabs seg.max_nnz reset
 * seg.max_nnz: non-zeros per segment of the handles with 64-bit row offsets created after it is set (tests; default 2^30).
 * An unknown key fails with SPMM_ERR_INVALID. */
int spmm_tune_set(const char *key, int value);

#ifdef __cplusplus
}
#endif
#endif
