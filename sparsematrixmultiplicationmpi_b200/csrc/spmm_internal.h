// spmm_internal.h — host-side structures shared by the translation units of libspmm_b200.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "spmm_b200.h"

namespace spmm
{

void set_error(const std::string &msg);
void note_kernel(const char *name); // kernel family of the calling thread's last launch (spmm_last_kernel_name)
int cuda_fail(cudaError_t e, const char *what, const char *file, int line);

#define SPMM_CUDA(call)                                                        \
    do                                                                         \
    {                                                                          \
        cudaError_t e__ = (call);                                              \
        if (e__ != cudaSuccess)                                                \
            return ::spmm::cuda_fail(e__, #call, __FILE__, __LINE__);          \
    } while (0)

#define SPMM_REQUIRE(cond, msg)                                                \
    do                                                                         \
    {                                                                          \
        if (!(cond))                                                           \
        {                                                                      \
            ::spmm::set_error(std::string("invalid argument: ") + (msg));     \
            return SPMM_ERR_INVALID;                                           \
        }                                                                      \
    } while (0)

// Row-length schedule of a CSR handle (built once on the device).
struct Schedule
{
    long long bins[8] = {0, 0, 0, 0, 0, 0, 0, 0}; // 0, 1-2, 3-4, 5-8, 9-16, 17-32, 33-256, >256
    int max_len = 0;
    double mean_len = 0.0;
    int auto_kernel = SPMM_KERNEL_ROWS;
};

// Tuning knobs (0 = choose automatically). Set through spmm_tune_set for experiments.
struct Tuning
{
    int rows_kl = 0;        // lanes across the columns of a B row
    int rows_nv = 0;        // accesses per lane (1, 2, 4)
    int rows_np = 0;        // concurrent non-zeros of one row per team
    int rows_unroll = 0;    // steps in flight per team
    int rows_vec = 0;       // 1 forces 8-byte accesses
    int rows_ctas_per_sm = 0;
    int merge_items = 0;    // merge-path items per team
    int merge_wave = 0;     // merge-path: warps per SM the item count is shrunk for on small shards (0 = 64)
    int rows_tile = 0;      // 0 auto, > 0 rows per round-robin tile, -1 never tile (one chunk per CTA)
    int rows_prefetch = -1; // -1 auto; bit0 A chunk, bit1 B share: TMA prefetch into L2 at kernel start
    int tiled = -1;         // -1 auto, 0 never use the tile layout, 1 always when built
    int tiled_thr = 0;      // build: non-zeros a box needs in a tile to be loaded as a box (else single rows)
    int tiled_chunk = 0;    // build: tiles per chunk
    int tiled_depth = 0;    // build: work items in flight (2..8)
    int tiled_pool = 0;     // build: rows of the singles pool
    int tiled_ns = 0;       // build: cap on the window slots
    int tiled_ksplit = 0;   // build: CTAs that share one chunk, each taking a group of k-tiles (0/1 none)
    int host_slabs = 0;     // host-buffer multiply: k-slabs in the PCIe pipeline (0 auto, 1 none)
    int tiled_auto_after = 8; // AUTO builds the tile layout on the multiply after this many whole-matrix multiplies of a handle
                              // (the build costs 4-7 ms of wall clock on cfg2 at k = 16 and 14-25 ms at k = 64 — five device passes of 1.9 ms
                              // plus allocations, tools/build_tiles_probe.py — and saves ~50 us per multiply)
    int tiled_pdl = 1;      // launch: programmatic dependent launch of the tiled kernel (0 off)
    int tiled_group = 0;    // build: tiles one far-band apart walked in turn, this many bands per group (0 auto = 2, 1 off)
    int tiled_stride = 0;   // build: far-band distance in rows (0 = detect from the matrix)
    int stream = -1;        // -1 auto, 0 AUTO never uses the stream kernel (k = 1, 2, 4, 8)
    int stream_auto_kmax = 1; // AUTO takes the stream kernel up to this k ...
    int stream_auto_min_nnz = 4 << 20; // ... from this many non-zeros (measured: equal to the row kernel at 2.6 M non-zeros, 43 against 56 us at 10.5 M; profiles/r1_stream.md)
    int stream_tile = 0;    // stream kernel: non-zeros per tile (0 = 4096 / k)
    int seg_max_nnz = 1 << 30; // 64-bit handles: non-zeros per segment (a longer row is a segment of its own); read at creation
};
Tuning &tuning();

struct DeviceProps
{
    int sm_count = 0;
    long long l2_bytes = 0;
};
const DeviceProps &device_props(int device);
// fn(i) for i in [0, n) on the library's host threads, the caller taking part (spmm_host.cu)
void host_parallel_for(int n, const std::function<void(int)> &fn);

} // namespace spmm

struct spmm_csr_s
{
    int device = 0;
    int n_rows = 0, n_cols = 0;
    long long nnz = 0;
    int *d_rowptr = nullptr;
    int *d_colidx = nullptr;
    double *d_vals = nullptr;
    bool owns = false;
    spmm::Schedule sched;
    // staging of the host-buffer entry points (spmm_host.cu): pinned mirrors of B and C, their device images, streams
    std::mutex host_mu; // one host-buffer call per handle at a time
    double *d_B = nullptr, *d_C = nullptr;
    size_t d_B_elems = 0, d_C_elems = 0;
    cudaStream_t stream = nullptr; // compute
    cudaStream_t stream_up = nullptr, stream_down = nullptr; // the two PCIe directions
    std::vector<cudaEvent_t> events;
    // B-staged row tiles (spmm_tiled.cu), optional
    int tl_T = 0, tl_BR = 0, tl_tiles = 0, tl_NS = 0, tl_POOL = 0, tl_max_recs = 0, tl_max_blob = 0, tl_chunk = 0, tl_kt = 0, tl_depth = 0, tl_drains = 0, tl_ksplit = 0;
    long long tl_box_rows_loaded = 0, tl_single_rows = 0; // B rows staged per pass over the matrix
    int auto_calls = 0;                                   // whole-matrix AUTO multiplies seen before the lazy build
    bool tl_tried = false;                                // AUTO already attempted the lazy build
    bool tl_auto = false;                                 // the layout was built by AUTO (it may rebuild it for another k)
    unsigned char *d_tblob = nullptr;
    void *d_tdesc = nullptr, *d_tloads = nullptr;
    int *d_tsingles = nullptr;
    int *d_torder = nullptr;          // walking order of the tiles (nullptr: as they lie)
    int tl_stride = 0, tl_group = 0;  // detected far-band distance in rows, planes interleaved per super-group
    mutable bool tl_refreshed = false; // blob values rewritten since the last tiled launch (that launch is not programmatic)
    int bsr_b = 0; // block size of the BSR view of the CSR arrays (spmm_bsr.cu), 0 = none
    // precomputed CTA cuts per (kind, grid size): kind 0 = rows of the CSR, 3 = stream-kernel tiles, 9 = block rows of the BSR view
    mutable std::map<long long, int *> bounds;
    // merge-path scratch (carry rows), grown on demand; one set per handle, so merge multiplies enqueued on different streams
    // are ordered through carry_done (recorded after each fix-up) whenever the stream changes
    double *d_carry = nullptr;
    int *d_carry_row = nullptr;
    size_t carry_elems = 0, carry_rows = 0;
    cudaEvent_t carry_done = nullptr;
    cudaStream_t carry_stream = nullptr; // stream of the last merge launch (carry_done was recorded there)
    // 64-bit row offsets (spmm_csr64.cu): d_rowptr stays nullptr; the rows are cut into segments, ordinary handles that
    // borrow their slices of d_colidx / d_vals and own nothing but their place in d_seg_rowptr (rebased int32 row pointers)
    long long *d_rowptr64 = nullptr;
    std::vector<spmm_csr_s *> segs;
    int *d_seg_rowptr = nullptr;
    int seg_row0 = 0;       // on a segment: its first row and first non-zero in the 64-bit handle
    long long seg_nnz0 = 0;
};

namespace spmm
{
// The device multiply forms: the whole matrix (spmm_multiply_device, _strided_device), scatter, a window of B rows (nothing
// beyond them may be read), a row range and a non-zero range; each accepts its own kernel ids (DESIGN.md section 4.3)
enum class Form { whole, scatter, window, rows, nnz_range };

// One device multiply: rows [row_begin,row_end), each clipped to the non-zero range [nnz_lo,nnz_hi); row c_row0 is
// stored at C[0]; kc columns of B and C
struct Request
{
    Form form;
    int row_begin, row_end;
    long long nnz_lo, nnz_hi;
    int c_row0;
    const double *B;
    long long ldb;
    double *C;
    long long ldc;
    int kc;
    const struct ExtraDst *extra; // scatter: the further copies of C (nullptr: none)
};

// The kernel `form` runs for the id `kernel` (AUTO stays AUTO), or the status that refuses the id (spmm_dispatch.cu)
int resolve_kernel(Form form, int kernel, int *effective);
// The one place that picks the kernel for a request; `kernel` as resolve_kernel returned it for req.form
int multiply(spmm_csr_s *A, const Request &req, int kernel, cudaStream_t stream);

// launchers implemented in the kernel translation units
int launch_rows(const spmm_csr_s *A, const Request &req, cudaStream_t stream);
int launch_merge(spmm_csr_s *A, const Request &req, cudaStream_t stream);
// tile layout (spmm_tiled.cu): what an explicit TILED request needs (status), when AUTO builds the layout, when AUTO uses it
int tiled_check(const spmm_csr_s *A, const Request &req);
void auto_tile_layout(spmm_csr_s *A, int k);
bool tiled_auto_ok(const spmm_csr_s *A, const Request &req);
int launch_tiled(const spmm_csr_s *A, const Request &req, cudaStream_t stream);
void free_tiles(spmm_csr_s *A);
// new values (d_src[nnz], CSR order, on A's device) into A->d_vals (skipped when d_src is A->d_vals) and into the value
// streams of the tile layout, enqueued on `stream`; the schedule, the CTA cuts and the rest of the layout are kept
int update_values(spmm_csr_s *A, const double *d_src, cudaStream_t stream);
int build_tiles(spmm_csr_s *A, int rows_per_tile, int box_rows, int kt_want, int ksplit_want);
// what AUTO cuts the tile layout for: 64-byte window rows for k <= 8; chunks shared by 2 / 4 CTAs (one k-tile group each) from k = 32 / 64
inline int tiles_kt_for(int k) { return k <= 8 ? 8 : 16; }
inline int tiles_ksplit_for(int k) { return k >= 64 ? 4 : (k >= 32 ? 2 : 1); }
// BSR view (spmm_bsr.cu): A->bsr_b != 0; every (row, column) is one FMA chain in storage order, as in the CSR kernels
int launch_bsr(const spmm_csr_s *A, const double *d_B, long long ldb, double *d_C, long long ldc, int kc, cudaStream_t stream);
bool stream_shape_ok(const spmm_csr_s *A, const double *d_B, long long ldb, const double *d_C, long long ldc, int kc);
int launch_stream(const spmm_csr_s *A, const double *d_B, long long ldb, double *d_C, long long ldc, int kc,
                  cudaStream_t stream);
// CTA cuts cached on the handle; `fill` launches the kernel that computes grid+1 cuts into its argument
int cached_bounds(const spmm_csr_s *A, int kind, int grid, cudaStream_t stream, const int **out,
                  const std::function<void(int *)> &fill);
void drop_bounds(spmm_csr_s *A, int kind); // kind < 0: all
// handle plumbing shared by spmm_capi.cu, csr_build.cu and spmm_csr64.cu; offsets64: nnz may exceed 2^31 - 1
int make_handle(int device, int n_rows, int n_cols, long long nnz, spmm_csr_s **out, bool offsets64 = false);
int alloc_arrays(spmm_csr_s *A);
int build_schedule(spmm_csr_s *A, cudaStream_t stream);
// 64-bit handles (spmm_csr64.cu): SPMM_ERR_UNSUPPORTED for a call that needs int32 row offsets, naming what to use instead
int refuse_offsets64(const char *call, const char *instead);
int nnz_range_rows64(const spmm_csr_s *A, long long nnz_begin, long long nnz_end, int *first_row, int *last_row);
} // namespace spmm
