// spmm_csr64.cu — handles with 64-bit row offsets: matrices of more than 2^31 - 1 stored entries.
//
// The handle keeps the caller's arrays (int64 rowptr, int32 colidx, f64 vals) and cuts the rows into segments, each an
// ordinary int32 handle of consecutive rows holding at most tuning().seg_max_nnz non-zeros (a longer row is a segment of
// its own). A segment borrows its slices of colidx / vals and reads a rebased int32 copy of its part of the row pointer,
// 4 bytes per row in all. multiply() (spmm_dispatch.cu) runs every request on the segments it touches with the int32
// kernels as they are; DESIGN.md section 4.8.
#include <algorithm>
#include <climits>
#include <string>
#include <vector>

#include "spmm_internal.h"

namespace spmm
{

namespace
{
// Segment cuts, greedy from the first row: segment s covers rows [cuts[s], cuts[s+1]), as many rows as keep it within
// max_nnz non-zeros and at least one. The cut steps back up to 32 rows to a row whose first non-zero is a multiple of 4,
// so that the segments' colidx and vals slices stay 16-byte aligned (the row kernel prefetches only aligned slices).
// One thread: a binary search on the 64-bit row pointer per segment. *n_segs = -1 when more than cap segments are needed.
__global__ void segment_cuts_kernel(const long long *__restrict__ rowptr, int n_rows, long long max_nnz, int cap,
                                    int *__restrict__ cuts, long long *__restrict__ cut_nnz, int *__restrict__ n_segs)
{
    int s = 0, r0 = 0;
    cuts[0] = 0;
    cut_nnz[0] = rowptr[0];
    while (r0 < n_rows && s < cap)
    {
        const long long limit = rowptr[r0] + max_nnz;
        int lo = r0 + 1, hi = n_rows; // the last row r in [r0 + 1, n_rows] with rowptr[r] <= limit, else r0 + 1
        while (lo < hi)
        {
            const int mid = lo + ((hi - lo + 1) >> 1);
            if (rowptr[mid] <= limit)
                lo = mid;
            else
                hi = mid - 1;
        }
        int r1 = lo;
        if (r1 < n_rows)
            for (int r = r1; r > r0 && r > r1 - 32; --r)
                if (rowptr[r] % 4 == 0)
                {
                    r1 = r;
                    break;
                }
        cuts[++s] = r1;
        cut_nnz[s] = rowptr[r1];
        r0 = r1;
    }
    *n_segs = r0 < n_rows ? -1 : s;
}

// The segments' row pointers one after another: segment s (rows [cuts[s], cuts[s+1])) starts at out[cuts[s] + s] and
// holds rowptr[r] - rowptr[cuts[s]] for r in [cuts[s], cuts[s+1]]
__global__ void segment_rowptr_kernel(const long long *__restrict__ rowptr, const int *__restrict__ cuts, int n_segs,
                                      long long n_out, int *__restrict__ out)
{
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < n_out; g += stride)
    {
        int lo = 0, hi = n_segs - 1; // the last s with cuts[s] + s <= g
        while (lo < hi)
        {
            const int mid = (lo + hi + 1) >> 1;
            if ((long long)cuts[mid] + mid <= g)
                lo = mid;
            else
                hi = mid - 1;
        }
        const long long r0 = cuts[lo];
        out[g] = (int)(rowptr[r0 + (g - r0 - lo)] - rowptr[r0]);
    }
}

// first = the row holding element nnz_begin, last = the row holding element nnz_end - 1 (as nnz_range_rows_kernel)
__global__ void nnz_range_rows64_kernel(const long long *__restrict__ rowptr, int n_rows, long long nnz_begin,
                                        long long nnz_end, int *out)
{
    auto find = [&](long long x) {
        int lo = 0, hi = n_rows;
        while (hi - lo > 1)
        {
            const int mid = lo + ((hi - lo) >> 1);
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

// RAII device buffer for the temporaries of segment_handles
struct Tmp
{
    void *p = nullptr;
    ~Tmp() { cudaFree(p); }
};

// Cut A (d_rowptr64, d_colidx, d_vals set) into segments, build each one's schedule and A's own from them
int segment_handles(spmm_csr_s *A)
{
    Schedule total;
    if (A->n_rows > 0)
    {
        const long long max_nnz = tuning().seg_max_nnz > 0 ? tuning().seg_max_nnz : (1LL << 30);
        // without the alignment step back, two neighbouring segments would hold more than max_nnz together, so fewer than
        // 2 nnz / max_nnz + 1 segments; should the step back need more, the cuts are found again with room for one per row
        int cap = (int)std::min<long long>(A->n_rows, 4 * (A->nnz / max_nnz) + 4), n_segs = -1;
        Tmp cuts, cut_nnz, count;
        SPMM_CUDA(cudaMalloc(&count.p, sizeof(int)));
        while (n_segs < 0)
        {
            cudaFree(cuts.p);
            cudaFree(cut_nnz.p);
            cuts.p = cut_nnz.p = nullptr;
            SPMM_CUDA(cudaMalloc(&cuts.p, sizeof(int) * ((size_t)cap + 1)));
            SPMM_CUDA(cudaMalloc(&cut_nnz.p, sizeof(long long) * ((size_t)cap + 1)));
            segment_cuts_kernel<<<1, 1>>>(A->d_rowptr64, A->n_rows, max_nnz, cap, (int *)cuts.p, (long long *)cut_nnz.p,
                                          (int *)count.p);
            SPMM_CUDA(cudaGetLastError());
            SPMM_CUDA(cudaMemcpy(&n_segs, count.p, sizeof(int), cudaMemcpyDeviceToHost));
            if (n_segs < 0)
            {
                SPMM_REQUIRE(cap < A->n_rows, "rowptr must not decrease");
                cap = A->n_rows;
            }
        }
        std::vector<int> h_cuts(n_segs + 1);
        std::vector<long long> h_nnz(n_segs + 1);
        SPMM_CUDA(cudaMemcpy(h_cuts.data(), cuts.p, sizeof(int) * h_cuts.size(), cudaMemcpyDeviceToHost));
        SPMM_CUDA(cudaMemcpy(h_nnz.data(), cut_nnz.p, sizeof(long long) * h_nnz.size(), cudaMemcpyDeviceToHost));
        for (int s = 0; s < n_segs; ++s)
        {
            const long long seg_nnz = h_nnz[s + 1] - h_nnz[s];
            SPMM_REQUIRE(seg_nnz >= 0, "rowptr must not decrease");
            if (seg_nnz > INT_MAX) // more than max_nnz: a single row
            {
                set_error("row " + std::to_string(h_cuts[s]) + " holds " + std::to_string(seg_nnz) +
                          " entries, more than the 2^31 - 1 the kernels address within one row");
                return SPMM_ERR_UNSUPPORTED;
            }
        }
        const long long n_out = (long long)A->n_rows + n_segs;
        SPMM_CUDA(cudaMalloc(&A->d_seg_rowptr, sizeof(int) * (size_t)n_out));
        const int grid = (int)std::min<long long>((n_out + 255) / 256, (long long)device_props(A->device).sm_count * 8);
        segment_rowptr_kernel<<<grid, 256>>>(A->d_rowptr64, (const int *)cuts.p, n_segs, n_out, A->d_seg_rowptr);
        SPMM_CUDA(cudaGetLastError());
        SPMM_CUDA(cudaDeviceSynchronize());
        for (int s = 0; s < n_segs; ++s)
        {
            spmm_csr_s *S = new spmm_csr_s();
            A->segs.push_back(S); // freed with A from here on
            S->device = A->device;
            S->n_rows = h_cuts[s + 1] - h_cuts[s];
            S->n_cols = A->n_cols;
            S->nnz = h_nnz[s + 1] - h_nnz[s];
            S->d_rowptr = A->d_seg_rowptr + h_cuts[s] + s;
            S->d_colidx = A->d_colidx + h_nnz[s];
            S->d_vals = A->d_vals + h_nnz[s];
            S->tl_tried = true; // AUTO never builds a tile layout on a segment
            S->seg_row0 = h_cuts[s];
            S->seg_nnz0 = h_nnz[s];
            if (int rc = build_schedule(S, nullptr))
                return rc;
            for (int i = 0; i < 8; ++i)
                total.bins[i] += S->sched.bins[i];
            total.max_len = std::max(total.max_len, S->sched.max_len);
            if (S->sched.auto_kernel == SPMM_KERNEL_MERGE)
                total.auto_kernel = SPMM_KERNEL_MERGE;
        }
        total.mean_len = (double)A->nnz / (double)A->n_rows;
    }
    A->sched = total;
    return SPMM_OK;
}

// The arrays are in place (copied or borrowed): the segments, then the handle goes out; on failure it is destroyed
int finish_handle(spmm_csr_s *A, spmm_csr_t *out)
{
    const int rc = segment_handles(A);
    if (rc)
    {
        spmm_csr_destroy(A);
        return rc;
    }
    *out = A;
    return SPMM_OK;
}
} // namespace

int refuse_offsets64(const char *call, const char *instead)
{
    set_error(std::string(call) + ": not available on a handle with 64-bit row offsets (spmm_csr_create_host64 / _device64); use " +
              instead);
    return SPMM_ERR_UNSUPPORTED;
}

int nnz_range_rows64(const spmm_csr_s *A, long long nnz_begin, long long nnz_end, int *first_row, int *last_row)
{
    Tmp d;
    SPMM_CUDA(cudaMalloc(&d.p, 2 * sizeof(int)));
    nnz_range_rows64_kernel<<<1, 1>>>(A->d_rowptr64, A->n_rows, nnz_begin, nnz_end, (int *)d.p);
    SPMM_CUDA(cudaGetLastError());
    int h[2] = {0, -1};
    SPMM_CUDA(cudaMemcpy(h, d.p, sizeof h, cudaMemcpyDeviceToHost));
    *first_row = h[0];
    *last_row = h[1];
    return SPMM_OK;
}

} // namespace spmm

using namespace spmm;

extern "C"
{

int spmm_csr_create_host64(int device, int n_rows, int n_cols, long long nnz, const long long *rowptr, const int *colidx,
                           const double *vals, spmm_csr_t *out)
{
    SPMM_REQUIRE(rowptr != nullptr, "rowptr is NULL");
    SPMM_REQUIRE(nnz == 0 || (colidx && vals), "colidx/vals are NULL");
    SPMM_REQUIRE(n_rows >= 0, "negative size");
    SPMM_REQUIRE(rowptr[0] == 0 && rowptr[n_rows] == nnz, "rowptr[0] must be 0 and rowptr[n_rows] must equal nnz");
    spmm_csr_s *A = nullptr;
    if (int rc = make_handle(device, n_rows, n_cols, nnz, &A, true))
        return rc;
    A->owns = true;
    cudaError_t e = cudaMalloc(&A->d_rowptr64, sizeof(long long) * ((size_t)n_rows + 1));
    // + 8 elements, as alloc_arrays: vector loads of the last ids / values may touch the padding past nnz
    if (e == cudaSuccess)
        e = cudaMalloc(&A->d_colidx, sizeof(int) * ((size_t)nnz + 8));
    if (e == cudaSuccess)
        e = cudaMalloc(&A->d_vals, sizeof(double) * ((size_t)nnz + 8));
    if (e == cudaSuccess)
        e = cudaMemcpy(A->d_rowptr64, rowptr, sizeof(long long) * ((size_t)n_rows + 1), cudaMemcpyHostToDevice);
    if (e == cudaSuccess && nnz)
        e = cudaMemcpy(A->d_colidx, colidx, sizeof(int) * (size_t)nnz, cudaMemcpyHostToDevice);
    if (e == cudaSuccess && nnz)
        e = cudaMemcpy(A->d_vals, vals, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice);
    if (e != cudaSuccess)
    {
        spmm_csr_destroy(A);
        return cuda_fail(e, "upload of the 64-bit CSR", __FILE__, __LINE__);
    }
    return finish_handle(A, out);
}

int spmm_csr_create_device64(int device, int n_rows, int n_cols, long long nnz, const long long *d_rowptr,
                             const int *d_colidx, const double *d_vals, int copy, spmm_csr_t *out)
{
    SPMM_REQUIRE(d_rowptr != nullptr, "d_rowptr is NULL");
    SPMM_REQUIRE(nnz == 0 || (d_colidx && d_vals), "d_colidx/d_vals are NULL");
    SPMM_REQUIRE(n_rows >= 0, "negative size");
    spmm_csr_s *A = nullptr;
    if (int rc = make_handle(device, n_rows, n_cols, nnz, &A, true))
        return rc;
    long long ends[2] = {-1, -1};
    cudaError_t e = cudaMemcpy(&ends[0], d_rowptr, sizeof(long long), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess)
        e = cudaMemcpy(&ends[1], d_rowptr + n_rows, sizeof(long long), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess || ends[0] != 0 || ends[1] != nnz)
    {
        spmm_csr_destroy(A);
        SPMM_CUDA(e);
        SPMM_REQUIRE(false, "rowptr[0] must be 0 and rowptr[n_rows] must equal nnz");
    }
    if (copy)
    {
        A->owns = true;
        e = cudaMalloc(&A->d_rowptr64, sizeof(long long) * ((size_t)n_rows + 1));
        if (e == cudaSuccess)
            e = cudaMalloc(&A->d_colidx, sizeof(int) * ((size_t)nnz + 8));
        if (e == cudaSuccess)
            e = cudaMalloc(&A->d_vals, sizeof(double) * ((size_t)nnz + 8));
        if (e == cudaSuccess)
            e = cudaMemcpy(A->d_rowptr64, d_rowptr, sizeof(long long) * ((size_t)n_rows + 1), cudaMemcpyDeviceToDevice);
        if (e == cudaSuccess && nnz)
            e = cudaMemcpy(A->d_colidx, d_colidx, sizeof(int) * (size_t)nnz, cudaMemcpyDeviceToDevice);
        if (e == cudaSuccess && nnz)
            e = cudaMemcpy(A->d_vals, d_vals, sizeof(double) * (size_t)nnz, cudaMemcpyDeviceToDevice);
        if (e != cudaSuccess)
        {
            spmm_csr_destroy(A);
            return cuda_fail(e, "copy of the 64-bit CSR", __FILE__, __LINE__);
        }
    }
    else
    {
        A->d_rowptr64 = const_cast<long long *>(d_rowptr);
        A->d_colidx = const_cast<int *>(d_colidx);
        A->d_vals = const_cast<double *>(d_vals);
    }
    return finish_handle(A, out);
}

int spmm_csr_device_ptrs64(spmm_csr_t A, const long long **d_rowptr, const int **d_colidx, const double **d_vals)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    if (!A->d_rowptr64)
    {
        set_error("spmm_csr_device_ptrs64: the handle has 32-bit row offsets; use spmm_csr_device_ptrs");
        return SPMM_ERR_UNSUPPORTED;
    }
    if (d_rowptr) *d_rowptr = A->d_rowptr64;
    if (d_colidx) *d_colidx = A->d_colidx;
    if (d_vals) *d_vals = A->d_vals;
    return SPMM_OK;
}

int spmm_csr_download64(spmm_csr_t A, long long *rowptr, int *colidx, double *vals)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    if (!A->d_rowptr64)
    {
        set_error("spmm_csr_download64: the handle has 32-bit row offsets; use spmm_csr_download");
        return SPMM_ERR_UNSUPPORTED;
    }
    SPMM_CUDA(cudaSetDevice(A->device));
    if (rowptr)
        SPMM_CUDA(cudaMemcpy(rowptr, A->d_rowptr64, sizeof(long long) * ((size_t)A->n_rows + 1), cudaMemcpyDeviceToHost));
    if (colidx && A->nnz)
        SPMM_CUDA(cudaMemcpy(colidx, A->d_colidx, sizeof(int) * (size_t)A->nnz, cudaMemcpyDeviceToHost));
    if (vals && A->nnz)
        SPMM_CUDA(cudaMemcpy(vals, A->d_vals, sizeof(double) * (size_t)A->nnz, cudaMemcpyDeviceToHost));
    return SPMM_OK;
}

} // extern "C"
