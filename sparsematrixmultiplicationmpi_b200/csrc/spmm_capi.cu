// spmm_capi.cu — the extern "C" boundary declared in include/spmm_b200.h.
//
// Thin by design: argument checks, device memory and the row-length schedule; the kernel
// is picked in spmm_dispatch.cu. All arithmetic of the path lives in the CUDA kernels
// (spmm_kernels.cuh, spmm_tiled.cu, spmm_stream.cu, spmm_bsr.cu, csr_build.cu).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>

#include "spmm_internal.h"
#include "spmm_kernels.cuh"

namespace spmm
{

static thread_local std::string g_last_error;

void set_error(const std::string &msg) { g_last_error = msg; }

static thread_local const char *g_last_kernel = "";
void note_kernel(const char *name) { g_last_kernel = name; }

int cuda_fail(cudaError_t e, const char *what, const char *file, int line)
{
    const char *base = std::strrchr(file, '/');
    g_last_error = std::string("CUDA error: ") + cudaGetErrorString(e) + " in " + what + " (" +
                   (base ? base + 1 : file) + ":" + std::to_string(line) + ")";
    return e == cudaErrorMemoryAllocation ? SPMM_ERR_NOMEM : SPMM_ERR_CUDA;
}

Tuning &tuning()
{
    static Tuning t;
    return t;
}

const DeviceProps &device_props(int device)
{
    static std::mutex mu;
    static std::map<int, DeviceProps> cache;
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(device);
    if (it != cache.end())
        return it->second;
    DeviceProps p;
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) == cudaSuccess)
        p.sm_count = v;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrL2CacheSize, device) == cudaSuccess)
        p.l2_bytes = v;
    if (p.sm_count <= 0)
        p.sm_count = 148;
    return cache[device] = p;
}

int cached_bounds(const spmm_csr_s *A, int kind, int grid, cudaStream_t stream, const int **out,
                  const std::function<void(int *)> &fill)
{
    const long long key = ((long long)kind << 32) | (unsigned)grid;
    auto it = A->bounds.find(key);
    if (it == A->bounds.end())
    {
        int *d = nullptr;
        SPMM_CUDA(cudaMalloc(&d, sizeof(int) * ((size_t)grid + 1)));
        fill(d);
        cudaError_t e = cudaGetLastError();
        // one-off per (matrix, grid): finished before the caller launches anything — kernels launched with programmatic
        // dependent launch read their cuts before they wait for the kernels ahead of them in the stream
        if (e == cudaSuccess)
            e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess)
        {
            cudaFree(d);
            return cuda_fail(e, "CTA cut kernel", __FILE__, __LINE__);
        }
        it = A->bounds.emplace(key, d).first;
    }
    *out = it->second;
    return SPMM_OK;
}

void drop_bounds(spmm_csr_s *A, int kind)
{
    for (auto it = A->bounds.begin(); it != A->bounds.end();)
    {
        if (kind < 0 || (int)(it->first >> 32) == kind)
        {
            cudaFree(it->second);
            it = A->bounds.erase(it);
        }
        else
            ++it;
    }
}

// ---- row-length schedule ----------------------------------------------------------
__global__ void schedule_kernel(const int *__restrict__ rowptr, int n_rows, unsigned long long *bins, int *max_len)
{
    __shared__ unsigned int s_bins[8];
    __shared__ int s_max;
    if (threadIdx.x < 8)
        s_bins[threadIdx.x] = 0;
    if (threadIdx.x == 0)
        s_max = 0;
    __syncthreads();
    int local_max = 0;
    for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < n_rows;
         r += (long long)gridDim.x * blockDim.x)
    {
        const int len = rowptr[r + 1] - rowptr[r];
        local_max = max(local_max, len);
        int b;
        if (len == 0) b = 0;
        else if (len <= 2) b = 1;
        else if (len <= 4) b = 2;
        else if (len <= 8) b = 3;
        else if (len <= 16) b = 4;
        else if (len <= 32) b = 5;
        else if (len <= 256) b = 6;
        else b = 7;
        atomicAdd(&s_bins[b], 1u);
    }
    atomicMax(&s_max, local_max);
    __syncthreads();
    if (threadIdx.x < 8 && s_bins[threadIdx.x])
        atomicAdd(&bins[threadIdx.x], (unsigned long long)s_bins[threadIdx.x]);
    if (threadIdx.x == 0)
        atomicMax(max_len, s_max);
}

int build_schedule(spmm_csr_s *A, cudaStream_t stream)
{
    Schedule s;
    if (A->n_rows > 0)
    {
        unsigned long long *d_bins = nullptr;
        SPMM_CUDA(cudaMalloc(&d_bins, 9 * sizeof(unsigned long long)));
        if (cudaError_t me = cudaMemsetAsync(d_bins, 0, 9 * sizeof(unsigned long long), stream); me != cudaSuccess)
        {
            cudaFree(d_bins);
            SPMM_CUDA(me);
        }
        const int threads = 256;
        const int blocks = (int)std::min<long long>(((long long)A->n_rows + threads - 1) / threads,
                                                    (long long)device_props(A->device).sm_count * 8);
        schedule_kernel<<<blocks, threads, 0, stream>>>(A->d_rowptr, A->n_rows, d_bins, (int *)(d_bins + 8));
        unsigned long long h[9];
        cudaError_t e = cudaMemcpyAsync(h, d_bins, sizeof h, cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess)
            e = cudaStreamSynchronize(stream);
        cudaFree(d_bins);
        SPMM_CUDA(e);
        for (int i = 0; i < 8; ++i)
            s.bins[i] = (long long)h[i];
        s.max_len = (int)(h[8] & 0xffffffffu);
        s.mean_len = (double)A->nnz / (double)A->n_rows;
    }
    // Power-law rows: one row far longer than an equal-cost chunk would make the
    // row-chunk kernel serialise on it -> nnz-balanced merge-path instead.
    const double chunk = (double)A->nnz / (double)(device_props(A->device).sm_count * 8) + 1.0;
    s.auto_kernel = (s.max_len > 4096 && (double)s.max_len > 0.25 * chunk) ? SPMM_KERNEL_MERGE : SPMM_KERNEL_ROWS;
    A->sched = s;
    return SPMM_OK;
}

int make_handle(int device, int n_rows, int n_cols, long long nnz, spmm_csr_s **out, bool offsets64)
{
    SPMM_REQUIRE(out != nullptr, "out handle is NULL");
    SPMM_REQUIRE(n_rows >= 0 && n_cols >= 0 && nnz >= 0, "negative size");
    SPMM_REQUIRE(offsets64 || nnz <= 2147483647LL, "nnz exceeds the int32 rowPtr of the reference data model");
    int count = 0;
    SPMM_CUDA(cudaGetDeviceCount(&count));
    SPMM_REQUIRE(device >= 0 && device < count, "no such CUDA device");
    SPMM_CUDA(cudaSetDevice(device));
    spmm_csr_s *A = new spmm_csr_s();
    A->device = device;
    A->n_rows = n_rows;
    A->n_cols = n_cols;
    A->nnz = nnz;
    *out = A;
    return SPMM_OK;
}

int alloc_arrays(spmm_csr_s *A)
{
    SPMM_CUDA(cudaMalloc(&A->d_rowptr, sizeof(int) * ((size_t)A->n_rows + 1)));
    // + 8 elements: vector loads of the last ids / values may touch the padding past nnz
    SPMM_CUDA(cudaMalloc(&A->d_colidx, sizeof(int) * ((size_t)std::max<long long>(A->nnz, 1) + 8)));
    SPMM_CUDA(cudaMalloc(&A->d_vals, sizeof(double) * ((size_t)std::max<long long>(A->nnz, 1) + 8)));
    A->owns = true;
    return SPMM_OK;
}

} // namespace spmm

using namespace spmm;

extern "C"
{

const char *spmm_last_error(void) { return g_last_error.c_str(); }
const char *spmm_last_kernel_name(void) { return g_last_kernel; }
int spmm_version(void) { return 100; }

int spmm_device_count(int *count)
{
    SPMM_REQUIRE(count != nullptr, "count is NULL");
    SPMM_CUDA(cudaGetDeviceCount(count));
    return SPMM_OK;
}

int spmm_device_info(int device, int *sm_count, long long *l2_bytes, long long *hbm_bytes)
{
    cudaDeviceProp p;
    SPMM_CUDA(cudaGetDeviceProperties(&p, device));
    if (sm_count)
        *sm_count = p.multiProcessorCount;
    if (l2_bytes)
        *l2_bytes = p.l2CacheSize;
    if (hbm_bytes)
        *hbm_bytes = (long long)p.totalGlobalMem;
    return SPMM_OK;
}

// experiment knob, not part of the stable ABI header
int spmm_tune_set(const char *key, int value)
{
    Tuning &t = tuning();
    std::string k = key ? key : "";
    if (k == "rows.np") t.rows_np = value;
    else if (k == "rows.kl") t.rows_kl = value;
    else if (k == "rows.nv") t.rows_nv = value;
    else if (k == "rows.prefetch") t.rows_prefetch = value;
    else if (k == "rows.tile") t.rows_tile = value;
    else if (k == "tiled") t.tiled = value;
    else if (k == "tiled.thr") t.tiled_thr = value;
    else if (k == "tiled.chunk") t.tiled_chunk = value;
    else if (k == "tiled.depth") t.tiled_depth = value;
    else if (k == "tiled.pool") t.tiled_pool = value;
    else if (k == "tiled.ns") t.tiled_ns = value;
    else if (k == "tiled.ksplit") t.tiled_ksplit = value;
    else if (k == "host.slabs") t.host_slabs = value;
    else if (k == "tiled.group") t.tiled_group = value;
    else if (k == "tiled.pdl") t.tiled_pdl = value;
    else if (k == "tiled.auto_after") t.tiled_auto_after = value;
    else if (k == "tiled.stride") t.tiled_stride = value;
    else if (k == "stream") t.stream = value;
    else if (k == "stream.tile") t.stream_tile = value;
    else if (k == "stream.kmax") t.stream_auto_kmax = value;
    else if (k == "stream.min_nnz") t.stream_auto_min_nnz = value;
    else if (k == "rows.unroll") t.rows_unroll = value;
    else if (k == "rows.vec") t.rows_vec = value;
    else if (k == "rows.ctas_per_sm") t.rows_ctas_per_sm = value;
    else if (k == "merge.items") t.merge_items = value;
    else if (k == "merge.wave") t.merge_wave = value;
    else if (k == "seg.max_nnz") t.seg_max_nnz = value;
    else if (k == "reset") t = Tuning();
    else
    {
        set_error("unknown tuning key: " + k);
        return SPMM_ERR_INVALID;
    }
    return SPMM_OK;
}

int spmm_csr_create_host(int device, int n_rows, int n_cols, long long nnz, const int *rowptr, const int *colidx,
                         const double *vals, spmm_csr_t *out)
{
    SPMM_REQUIRE(rowptr != nullptr, "rowptr is NULL");
    SPMM_REQUIRE(nnz == 0 || (colidx && vals), "colidx/vals are NULL");
    SPMM_REQUIRE(rowptr[0] == 0 && rowptr[n_rows] == nnz, "rowptr[0] must be 0 and rowptr[n_rows] must equal nnz");
    spmm_csr_s *A = nullptr;
    int rc = make_handle(device, n_rows, n_cols, nnz, &A);
    if (rc)
        return rc;
    rc = alloc_arrays(A);
    if (!rc)
    {
        cudaError_t e = cudaMemcpy(A->d_rowptr, rowptr, sizeof(int) * ((size_t)n_rows + 1), cudaMemcpyHostToDevice);
        if (e == cudaSuccess && nnz)
            e = cudaMemcpy(A->d_colidx, colidx, sizeof(int) * (size_t)nnz, cudaMemcpyHostToDevice);
        if (e == cudaSuccess && nnz)
            e = cudaMemcpy(A->d_vals, vals, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice);
        if (e != cudaSuccess)
            rc = cuda_fail(e, "cudaMemcpy(H2D CSR)", __FILE__, __LINE__);
    }
    if (!rc)
        rc = build_schedule(A, nullptr);
    if (rc)
    {
        spmm_csr_destroy(A);
        return rc;
    }
    *out = A;
    return SPMM_OK;
}

int spmm_csr_create_device(int device, int n_rows, int n_cols, long long nnz, const int *d_rowptr,
                           const int *d_colidx, const double *d_vals, int copy, spmm_csr_t *out)
{
    SPMM_REQUIRE(d_rowptr != nullptr, "d_rowptr is NULL");
    SPMM_REQUIRE(nnz == 0 || (d_colidx && d_vals), "d_colidx/d_vals are NULL");
    spmm_csr_s *A = nullptr;
    int rc = make_handle(device, n_rows, n_cols, nnz, &A);
    if (rc)
        return rc;
    if (copy)
    {
        rc = alloc_arrays(A);
        if (!rc)
        {
            cudaError_t e = cudaMemcpy(A->d_rowptr, d_rowptr, sizeof(int) * ((size_t)n_rows + 1), cudaMemcpyDeviceToDevice);
            if (e == cudaSuccess && nnz)
                e = cudaMemcpy(A->d_colidx, d_colidx, sizeof(int) * (size_t)nnz, cudaMemcpyDeviceToDevice);
            if (e == cudaSuccess && nnz)
                e = cudaMemcpy(A->d_vals, d_vals, sizeof(double) * (size_t)nnz, cudaMemcpyDeviceToDevice);
            if (e != cudaSuccess)
                rc = cuda_fail(e, "cudaMemcpy(D2D CSR)", __FILE__, __LINE__);
        }
    }
    else
    {
        A->d_rowptr = const_cast<int *>(d_rowptr);
        A->d_colidx = const_cast<int *>(d_colidx);
        A->d_vals = const_cast<double *>(d_vals);
        A->owns = false;
    }
    if (!rc)
        rc = build_schedule(A, nullptr);
    if (rc)
    {
        spmm_csr_destroy(A);
        return rc;
    }
    *out = A;
    return SPMM_OK;
}

int spmm_csr_destroy(spmm_csr_t A)
{
    if (!A)
        return SPMM_OK;
    cudaSetDevice(A->device);
    if (A->owns)
    {
        cudaFree(A->d_rowptr);
        cudaFree(A->d_rowptr64);
        cudaFree(A->d_colidx);
        cudaFree(A->d_vals);
    }
    for (spmm_csr_s *S : A->segs)
        spmm_csr_destroy(S);
    cudaFree(A->d_seg_rowptr);
    free_tiles(A);
    drop_bounds(A, -1);
    cudaFree(A->d_B);
    cudaFree(A->d_C);
    cudaFree(A->d_carry);
    cudaFree(A->d_carry_row);
    if (A->carry_done)
        cudaEventDestroy(A->carry_done);
    if (A->stream)
        cudaStreamDestroy(A->stream);
    if (A->stream_up)
    {
        cudaStreamDestroy(A->stream_up);
        cudaStreamDestroy(A->stream_down);
    }
    for (cudaEvent_t e : A->events)
        cudaEventDestroy(e);
    delete A;
    return SPMM_OK;
}

int spmm_csr_info(spmm_csr_t A, int *n_rows, int *n_cols, long long *nnz, int *device)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    if (n_rows) *n_rows = A->n_rows;
    if (n_cols) *n_cols = A->n_cols;
    if (nnz) *nnz = A->nnz;
    if (device) *device = A->device;
    return SPMM_OK;
}

int spmm_csr_device_ptrs(spmm_csr_t A, const int **d_rowptr, const int **d_colidx, const double **d_vals)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    if (A->d_rowptr64)
        return refuse_offsets64("spmm_csr_device_ptrs", "spmm_csr_device_ptrs64");
    if (d_rowptr) *d_rowptr = A->d_rowptr;
    if (d_colidx) *d_colidx = A->d_colidx;
    if (d_vals) *d_vals = A->d_vals;
    return SPMM_OK;
}

int spmm_csr_update_values_device(spmm_csr_t A, const double *d_vals, void *stream)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    if (A->nnz == 0)
        return SPMM_OK;
    SPMM_REQUIRE(d_vals != nullptr, "d_vals is NULL");
    SPMM_REQUIRE(A->owns || d_vals == A->d_vals,
                 "a borrowed handle reads the caller's value array: edit that array and pass it, the library does not write into it");
    SPMM_CUDA(cudaSetDevice(A->device));
    return update_values(A, d_vals, (cudaStream_t)stream);
}

int spmm_csr_download(spmm_csr_t A, int *rowptr, int *colidx, double *vals)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    if (A->d_rowptr64)
        return refuse_offsets64("spmm_csr_download", "spmm_csr_download64");
    SPMM_CUDA(cudaSetDevice(A->device));
    if (rowptr)
        SPMM_CUDA(cudaMemcpy(rowptr, A->d_rowptr, sizeof(int) * ((size_t)A->n_rows + 1), cudaMemcpyDeviceToHost));
    if (colidx && A->nnz)
        SPMM_CUDA(cudaMemcpy(colidx, A->d_colidx, sizeof(int) * (size_t)A->nnz, cudaMemcpyDeviceToHost));
    if (vals && A->nnz)
        SPMM_CUDA(cudaMemcpy(vals, A->d_vals, sizeof(double) * (size_t)A->nnz, cudaMemcpyDeviceToHost));
    return SPMM_OK;
}

int spmm_csr_schedule(spmm_csr_t A, long long bins[8], int *max_row_len, double *mean_row_len, int *auto_kernel)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    if (bins)
        for (int i = 0; i < 8; ++i)
            bins[i] = A->sched.bins[i];
    if (max_row_len) *max_row_len = A->sched.max_len;
    if (mean_row_len) *mean_row_len = A->sched.mean_len;
    if (auto_kernel) *auto_kernel = A->sched.auto_kernel;
    return SPMM_OK;
}

// ---- multiply ---------------------------------------------------------------------

int spmm_multiply_strided_device(spmm_csr_t A, const double *d_B, int ldb, double *d_C, int ldc, int k_begin,
                                 int k_count, int kernel, void *stream)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    SPMM_REQUIRE(k_begin >= 0 && k_count >= 0, "negative column range");
    SPMM_REQUIRE(ldb >= k_begin + k_count && ldc >= k_begin + k_count, "leading dimension smaller than column range");
    if (int rc = resolve_kernel(Form::whole, kernel, &kernel))
        return rc;
    if (A->n_rows == 0 || k_count == 0)
        return SPMM_OK;
    SPMM_REQUIRE(d_C != nullptr, "d_C is NULL");
    SPMM_REQUIRE(d_B != nullptr || A->nnz == 0, "d_B is NULL");
    const Request r = {Form::whole, 0, A->n_rows, 0, A->nnz, 0, d_B + k_begin, ldb, d_C + k_begin, ldc, k_count, nullptr};
    return multiply(A, r, kernel, (cudaStream_t)stream);
}

int spmm_multiply_scatter_device(spmm_csr_t A, const double *d_B, int k, int n_dst, double *const *d_C_list, int kernel,
                                 void *stream)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    SPMM_REQUIRE(k >= 0, "k is negative");
    if (int rc = resolve_kernel(Form::scatter, kernel, &kernel))
        return rc;
    SPMM_REQUIRE(n_dst >= 1 && n_dst <= 1 + SPMM_MAX_EXTRA, "n_dst must be between 1 and 8");
    SPMM_REQUIRE(d_C_list != nullptr, "d_C_list is NULL");
    if (A->n_rows == 0 || k == 0)
        return SPMM_OK;
    ExtraDst x;
    for (int i = 0; i < n_dst; ++i)
    {
        SPMM_REQUIRE(d_C_list[i] != nullptr, "a destination pointer is NULL");
        SPMM_REQUIRE(((uintptr_t)d_C_list[i] - (uintptr_t)d_C_list[0]) % 16 == 0,
                     "destinations must be congruent modulo 16 bytes (same vector width for every copy)");
        if (i)
            x.off[x.n++] = (long long)(((intptr_t)d_C_list[i] - (intptr_t)d_C_list[0]) / (intptr_t)sizeof(double));
    }
    SPMM_REQUIRE(d_B != nullptr || A->nnz == 0, "d_B is NULL");
    const Request r = {Form::scatter, 0, A->n_rows, 0, A->nnz, 0, d_B, k, d_C_list[0], k, k, &x};
    return multiply(A, r, kernel, (cudaStream_t)stream);
}

int spmm_multiply_device(spmm_csr_t A, const double *d_B, int k, double *d_C, int kernel, void *stream)
{
    SPMM_REQUIRE(k >= 0, "k is negative");
    return spmm_multiply_strided_device(A, d_B, k, d_C, k, 0, k, kernel, stream);
}

int spmm_multiply_window_device(spmm_csr_t A, const double *d_B_window, int window_first_row, int window_rows, int k,
                                double *d_C, int kernel, void *stream)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    SPMM_REQUIRE(k >= 0 && window_first_row >= 0 && window_rows >= 0 && (long long)window_first_row + window_rows <= A->n_cols,
                 "window outside B");
    if (int rc = resolve_kernel(Form::window, kernel, &kernel))
        return rc;
    if (A->n_rows == 0 || k == 0)
        return SPMM_OK;
    SPMM_REQUIRE(d_C != nullptr && (d_B_window != nullptr || A->nnz == 0), "d_B_window / d_C is NULL");
    // virtual base: row j of B sits at d_B_window + (j - window_first_row) * k; only rows named by column ids are read
    const double *base = d_B_window - (long long)window_first_row * k;
    const Request r = {Form::window, 0, A->n_rows, 0, A->nnz, 0, base, k, d_C, k, k, nullptr};
    return multiply(A, r, kernel, (cudaStream_t)stream);
}

int spmm_multiply_rows_device(spmm_csr_t A, int row_begin, int row_end, const double *d_B, int k,
                              double *d_C_local, int kernel, void *stream)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    SPMM_REQUIRE(k >= 0, "k is negative");
    SPMM_REQUIRE(0 <= row_begin && row_begin <= row_end && row_end <= A->n_rows, "row range outside the matrix");
    if (int rc = resolve_kernel(Form::rows, kernel, &kernel))
        return rc;
    if (row_begin == row_end || k == 0)
        return SPMM_OK;
    SPMM_REQUIRE(d_C_local != nullptr, "d_C_local is NULL");
    SPMM_REQUIRE(d_B != nullptr || A->nnz == 0, "d_B is NULL");
    const Request r = {Form::rows, row_begin, row_end, 0, A->nnz, row_begin, d_B, k, d_C_local, k, k, nullptr};
    return multiply(A, r, kernel, (cudaStream_t)stream);
}

// Rows touched by a non-zero range: first = the row holding element nnz_begin,
// last = the row holding element nnz_end-1 (NonZeroElement.cpp:42-51 expands the same
// map element by element; here it is two binary searches on the device row pointer).
__global__ void nnz_range_rows_kernel(const int *__restrict__ rowptr, int n_rows, int nnz_begin, int nnz_end, int *out)
{
    // last row r with rowptr[r] <= x  (rows are non-decreasing; skips empty rows at x)
    auto find = [&](int x) {
        int lo = 0, hi = n_rows; // invariant: rowptr[lo] <= x < rowptr[hi] ... hi may be n_rows
        while (hi - lo > 1)
        {
            int mid = lo + ((hi - lo) >> 1);
            if (rowptr[mid] <= x)
                lo = mid;
            else
                hi = mid;
        }
        return lo;
    };
    out[0] = find(nnz_begin);
    out[1] = find(nnz_end - 1);
}

int spmm_nnz_range_rows(spmm_csr_t A, long long nnz_begin, long long nnz_end, int *first_row, int *last_row)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    SPMM_REQUIRE(first_row && last_row, "output pointer is NULL");
    SPMM_REQUIRE(0 <= nnz_begin && nnz_begin <= nnz_end && nnz_end <= A->nnz, "non-zero range outside the matrix");
    if (nnz_begin == nnz_end)
    {
        *first_row = 0;
        *last_row = -1; // empty range touches no row
        return SPMM_OK;
    }
    SPMM_CUDA(cudaSetDevice(A->device));
    if (A->d_rowptr64)
        return nnz_range_rows64(A, nnz_begin, nnz_end, first_row, last_row);
    int *d_out = nullptr;
    SPMM_CUDA(cudaMalloc(&d_out, 2 * sizeof(int)));
    nnz_range_rows_kernel<<<1, 1>>>(A->d_rowptr, A->n_rows, (int)nnz_begin, (int)nnz_end, d_out);
    int h[2] = {0, -1};
    cudaError_t e = cudaMemcpy(h, d_out, sizeof h, cudaMemcpyDeviceToHost);
    cudaFree(d_out);
    SPMM_CUDA(e);
    *first_row = h[0];
    *last_row = h[1];
    return SPMM_OK;
}

int spmm_multiply_nnz_range_device(spmm_csr_t A, long long nnz_begin, long long nnz_end, int first_row, int last_row,
                                   const double *d_B, int k, double *d_C_local, int kernel, void *stream)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    SPMM_REQUIRE(k >= 0, "k is negative");
    SPMM_REQUIRE(0 <= nnz_begin && nnz_begin <= nnz_end && nnz_end <= A->nnz, "non-zero range outside the matrix");
    if (int rc = resolve_kernel(Form::nnz_range, kernel, &kernel))
        return rc;
    if (nnz_begin == nnz_end || k == 0 || last_row < first_row)
        return SPMM_OK;
    SPMM_REQUIRE(0 <= first_row && last_row < A->n_rows, "row range outside the matrix");
    SPMM_REQUIRE(d_C_local != nullptr && d_B != nullptr, "d_B/d_C_local is NULL");
    const Request r = {Form::nnz_range, first_row, last_row + 1, nnz_begin, nnz_end, first_row, d_B, k, d_C_local, k, k, nullptr};
    return multiply(A, r, kernel, (cudaStream_t)stream);
}

} // extern "C"

// Column-block strategy without NCCL: this rank's block of C = sum over ranks of their partial blocks, read straight from
// the peers' buffers over NVLink (P2P loads) and added in ascending rank order — the order of the reference's MPI_Reduce on
// a single communicator walk and of the oracle, so the result is reproducible bit for bit.
struct ReduceSrc
{
    const double *p[8];
};
__global__ void __launch_bounds__(256) reduce_blocks_kernel(const ReduceSrc src, int n_src, double *__restrict__ out,
                                                            long long n_pairs)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_pairs; i += stride)
    {
        double2 acc = __ldcs(reinterpret_cast<const double2 *>(src.p[0]) + i);
        for (int r = 1; r < n_src; ++r)
        {
            const double2 v = __ldcs(reinterpret_cast<const double2 *>(src.p[r]) + i);
            acc.x += v.x;
            acc.y += v.y;
        }
        reinterpret_cast<double2 *>(out)[i] = acc;
    }
}

extern "C" int spmm_reduce_blocks_device(int device, int n_src, const double *const *d_src_list, long long n_elems,
                                         double *d_out, void *stream)
{
    SPMM_REQUIRE(n_src >= 1 && n_src <= 1024, "n_src must be between 1 and 1024");
    SPMM_REQUIRE(d_src_list != nullptr && d_out != nullptr, "source list / output is NULL");
    SPMM_REQUIRE(n_elems >= 0 && n_elems % 2 == 0, "n_elems must be even (16-byte accesses)");
    if (n_elems == 0)
        return SPMM_OK;
    for (int i = 0; i < n_src; ++i)
        SPMM_REQUIRE(d_src_list[i] != nullptr && (uintptr_t)d_src_list[i] % 16 == 0, "sources must be 16-byte aligned");
    SPMM_REQUIRE((uintptr_t)d_out % 16 == 0, "output must be 16-byte aligned");
    SPMM_CUDA(cudaSetDevice(device));
    const long long pairs = n_elems / 2;
    const int grid = (int)std::min<long long>((pairs + 255) / 256, (long long)device_props(device).sm_count * 8);
    // up to 8 sources per pass; further passes continue the same left-to-right sum from d_out
    for (int first = 0; first < n_src;)
    {
        ReduceSrc src = {};
        int n = 0;
        if (first > 0)
            src.p[n++] = d_out;
        while (n < 8 && first < n_src)
            src.p[n++] = d_src_list[first++];
        reduce_blocks_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, n, d_out, pairs);
        SPMM_CUDA(cudaGetLastError());
    }
    return SPMM_OK;
}

// dst[i] += src[i] (any n, any alignment): the non-zero strategy's cut rows, added on the root device in rank order
__global__ void __launch_bounds__(256) add_kernel(double *__restrict__ dst, const double *__restrict__ src, long long n)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        dst[i] += src[i];
}

extern "C" int spmm_add_device(int device, double *d_dst, const double *d_src, long long n_elems, void *stream)
{
    SPMM_REQUIRE(n_elems >= 0, "negative size");
    if (n_elems == 0)
        return SPMM_OK;
    SPMM_REQUIRE(d_dst != nullptr && d_src != nullptr, "d_dst / d_src is NULL");
    SPMM_CUDA(cudaSetDevice(device));
    const int grid = (int)std::min<long long>((n_elems + 255) / 256, (long long)device_props(device).sm_count * 8);
    add_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_dst, d_src, n_elems);
    SPMM_CUDA(cudaGetLastError());
    return SPMM_OK;
}

extern "C" int spmm_copy_device(int device, void *d_dst, const void *d_src, long long bytes, void *stream)
{
    SPMM_REQUIRE(bytes >= 0, "negative size");
    if (bytes == 0)
        return SPMM_OK;
    SPMM_REQUIRE(d_dst != nullptr && d_src != nullptr, "d_dst / d_src is NULL");
    SPMM_CUDA(cudaSetDevice(device));
    // unified addressing: the runtime routes the copy between whichever devices own the two buffers (NVLink when peers)
    SPMM_CUDA(cudaMemcpyAsync(d_dst, d_src, (size_t)bytes, cudaMemcpyDefault, (cudaStream_t)stream));
    return SPMM_OK;
}

extern "C" int spmm_fill_zero_device(int device, void *d_dst, long long bytes, void *stream)
{
    SPMM_REQUIRE(bytes >= 0 && (d_dst != nullptr || bytes == 0), "bad fill request");
    SPMM_CUDA(cudaSetDevice(device));
    if (bytes)
        SPMM_CUDA(cudaMemsetAsync(d_dst, 0, (size_t)bytes, (cudaStream_t)stream));
    return SPMM_OK;
}

extern "C" int spmm_device_sync(int device)
{
    SPMM_CUDA(cudaSetDevice(device));
    SPMM_CUDA(cudaDeviceSynchronize());
    return SPMM_OK;
}

// smallest and largest column id of a handle: the B rows a shard reads lie in [min, max]
__global__ void __launch_bounds__(256) column_span_kernel(const int *__restrict__ colidx, long long nnz, int *out)
{
    int lo = 0x7FFFFFFF, hi = -1;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += stride)
    {
        const int c = colidx[i];
        lo = min(lo, c);
        hi = max(hi, c);
    }
    lo = __reduce_min_sync(0xFFFFFFFFu, lo);
    hi = __reduce_max_sync(0xFFFFFFFFu, hi);
    if ((threadIdx.x & 31) == 0)
    {
        atomicMin(out, lo);
        atomicMax(out + 1, hi);
    }
}

extern "C" int spmm_csr_column_span(spmm_csr_t A, int *min_col, int *max_col)
{
    SPMM_REQUIRE(A != nullptr && min_col && max_col, "handle / output is NULL");
    *min_col = 0;
    *max_col = -1;
    if (A->nnz == 0)
        return SPMM_OK;
    SPMM_CUDA(cudaSetDevice(A->device));
    int *d = nullptr;
    SPMM_CUDA(cudaMalloc(&d, 2 * sizeof(int)));
    const int init[2] = {0x7FFFFFFF, -1};
    cudaError_t e = cudaMemcpy(d, init, sizeof init, cudaMemcpyHostToDevice);
    if (e == cudaSuccess)
    {
        const int grid = (int)std::min<long long>((A->nnz + 255) / 256, (long long)device_props(A->device).sm_count * 8);
        column_span_kernel<<<grid, 256>>>(A->d_colidx, A->nnz, d);
        e = cudaGetLastError();
    }
    int h[2] = {0, -1};
    if (e == cudaSuccess)
        e = cudaMemcpy(h, d, sizeof h, cudaMemcpyDeviceToHost);
    cudaFree(d);
    SPMM_CUDA(e);
    *min_col = h[0];
    *max_col = h[1];
    return SPMM_OK;
}

extern "C"
{

// ---- partition formulas -------------------------------------------------------------

void spmm_partition_rows(int n_rows, int n_ranks, int rank, int *begin, int *end)
{
    const int base = n_rows / n_ranks, extra = n_rows % n_ranks;
    const int b = rank * base + std::min(rank, extra);
    *begin = b;
    *end = b + base + (rank < extra ? 1 : 0);
}

void spmm_partition_cols(int k, int n_ranks, int rank, int *begin, int *end)
{
    const int base = k / n_ranks, extra = k % n_ranks;
    *begin = rank * base;
    *end = rank * base + base + (rank == n_ranks - 1 ? extra : 0);
}

void spmm_partition_nnz(long long nnz, int n_ranks, int rank, long long *begin, long long *end)
{
    const long long per = nnz / n_ranks, extra = nnz % n_ranks;
    if (rank < extra)
    {
        *begin = rank * (per + 1);
        *end = *begin + per + 1;
    }
    else
    {
        *begin = rank * per + extra;
        *end = *begin + per;
    }
}

// ---- host utilities -----------------------------------------------------------------

void spmm_generate_fat_vector(int n, int k, double *out)
{
    // The reference never seeds (utils.cpp:203): libc's default state == srand(1).
    srand(1);
    for (long long i = 0; i < (long long)n * k; ++i)
        out[i] = rand() % 100 + 1;
}

int spmm_are_equal(const double *a, const double *b, long long n, double tol)
{
    for (long long i = 0; i < n; ++i)
        if (std::fabs(a[i] - b[i]) > tol)
            return 0;
    return 1;
}

} // extern "C"
