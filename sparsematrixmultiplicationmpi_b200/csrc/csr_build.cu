// csr_build.cu — device-resident CSR construction and the synthetic workloads.
//
//  * spmm_csr_from_coo_*: the CSR assembly of readMatrixMarketFile
//    (/root/reference "Source Code/utils.cpp":124-181) done in HBM: symmetric
//    mirroring (:146-152), per-row order by (column, value) ascending (:156-159,
//    std::sort on pair<int,double>), duplicates kept, rowPtr = prefix sum (:162-179).
//    The reference builds vector<vector<pair>> and sorts each row on the host; here
//    the records are ordered by two stable LSD radix sorts (value bits, then
//    row:col) and the row pointer is a binary search per row. Sorting/scanning is
//    plumbing, not the hot path: it uses CUB from the CUDA toolkit.
//  * spmm_csr_column_block: A[:, c0:c1) with local column ids (column-block strategy).
//  * spmm_gen_*: banded and R-MAT matrices and 1..100 fat vectors generated in HBM
//    from a counter-based hash, so that a row block generated on one GPU is
//    bit-identical to the same rows of the whole matrix generated on another.
#include <climits>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "spmm_internal.h"

namespace spmm
{

namespace
{

struct DevBuf
{
    void *p = nullptr;
    ~DevBuf() { cudaFree(p); }
    cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 1); }
    template <typename T>
    T *as() { return (T *)p; }
};

constexpr int TPB = 256;
inline unsigned blocks_for(long long n) { return (unsigned)std::max<long long>(1, (n + TPB - 1) / TPB); }

__host__ __device__ __forceinline__ unsigned long long splitmix64(unsigned long long x)
{
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}
__host__ __device__ __forceinline__ double u01(unsigned long long h) { return (double)(h >> 11) * (1.0 / 9007199254740992.0); }

// IEEE-754 double -> unsigned key with the same order as operator< (all -x < +x; -0 before +0).
__device__ __forceinline__ unsigned long long ordered_bits(double v)
{
    unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b & 0x8000000000000000ULL) ? ~b : (b | 0x8000000000000000ULL);
}

__global__ void coo_check_kernel(const int *rows, const int *cols, long long n, int n_rows, int n_cols, int symmetric,
                                 int *bad, int *mirror_flag)
{
    const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= n)
        return;
    const int r = rows[e], c = cols[e];
    bool ok = r >= 0 && r < n_rows && c >= 0 && c < n_cols;
    if (symmetric) // the mirrored record (c, r) must fit too
        ok = ok && c < n_rows && r < n_cols;
    if (!ok)
        atomicExch(bad, 1);
    if (mirror_flag)
        mirror_flag[e] = (symmetric && r != c) ? 1 : 0;
}

// record e -> slot e; its mirror -> slot n + mirror_pos[e]
__global__ void coo_expand_kernel(const int *rows, const int *cols, const double *vals, long long n,
                                  const int *mirror_flag, const int *mirror_pos, unsigned long long *key,
                                  unsigned long long *vkey, double *xval, unsigned *idx)
{
    const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= n)
        return;
    const unsigned r = (unsigned)rows[e], c = (unsigned)cols[e];
    const double v = vals[e];
    key[e] = ((unsigned long long)r << 32) | c;
    vkey[e] = ordered_bits(v);
    xval[e] = v;
    idx[e] = (unsigned)e;
    if (mirror_flag && mirror_flag[e])
    {
        const long long m = n + mirror_pos[e];
        key[m] = ((unsigned long long)c << 32) | r;
        vkey[m] = ordered_bits(v);
        xval[m] = v;
        idx[m] = (unsigned)m;
    }
}

__global__ void gather_keys_kernel(const unsigned long long *key, const unsigned *idx, long long m, unsigned long long *out)
{
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < m)
        out[i] = key[idx[i]];
}

__global__ void emit_csr_kernel(const unsigned long long *sorted_key, const unsigned *sorted_idx, const double *xval,
                                long long m, int *colidx, double *vals)
{
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= m)
        return;
    colidx[i] = (int)(sorted_key[i] & 0xffffffffULL);
    vals[i] = xval[sorted_idx[i]];
}

// rowptr[r] = number of records whose row is < r
__global__ void rowptr_kernel(const unsigned long long *sorted_key, long long m, int n_rows, int *rowptr)
{
    const long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (r > n_rows)
        return;
    long long lo = 0, hi = m;
    while (lo < hi)
    {
        const long long mid = (lo + hi) >> 1;
        if ((long long)(sorted_key[mid] >> 32) < r)
            lo = mid + 1;
        else
            hi = mid;
    }
    rowptr[r] = (int)lo;
}

int bits_for(unsigned long long max_value)
{
    int b = 1;
    while (b < 64 && (max_value >> b))
        ++b;
    return b;
}

} // namespace

static int csr_from_coo_device_impl(int device, int n_rows, int n_cols, long long n, const int *d_rows,
                                    const int *d_cols, const double *d_vals, int symmetric, spmm_csr_t *out)
{
    SPMM_REQUIRE(out != nullptr, "out handle is NULL");
    SPMM_REQUIRE(n >= 0 && n <= INT_MAX, "record count outside int32");
    SPMM_REQUIRE(n == 0 || (d_rows && d_cols && d_vals), "coordinate arrays are NULL");
    SPMM_CUDA(cudaSetDevice(device));
    cudaStream_t st = nullptr;

    DevBuf bad, flag, pos;
    SPMM_CUDA(bad.alloc(2 * sizeof(int)));
    SPMM_CUDA(cudaMemsetAsync(bad.p, 0, 2 * sizeof(int), st));
    long long m = n;
    if (symmetric)
    {
        SPMM_CUDA(flag.alloc(sizeof(int) * (size_t)n));
        SPMM_CUDA(pos.alloc(sizeof(int) * ((size_t)n + 1)));
    }
    if (n)
    {
        coo_check_kernel<<<blocks_for(n), TPB, 0, st>>>(d_rows, d_cols, n, n_rows, n_cols, symmetric, bad.as<int>(),
                                                       symmetric ? flag.as<int>() : nullptr);
        SPMM_CUDA(cudaGetLastError());
    }
    if (symmetric && n)
    {
        size_t tmp_bytes = 0;
        SPMM_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, flag.as<int>(), pos.as<int>(), (int)n, st));
        DevBuf tmp;
        SPMM_CUDA(tmp.alloc(tmp_bytes));
        SPMM_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, flag.as<int>(), pos.as<int>(), (int)n, st));
        int last_pos = 0, last_flag = 0;
        SPMM_CUDA(cudaMemcpyAsync(&last_pos, pos.as<int>() + (n - 1), sizeof(int), cudaMemcpyDeviceToHost, st));
        SPMM_CUDA(cudaMemcpyAsync(&last_flag, flag.as<int>() + (n - 1), sizeof(int), cudaMemcpyDeviceToHost, st));
        SPMM_CUDA(cudaStreamSynchronize(st));
        m = n + last_pos + last_flag;
    }
    int h_bad = 0;
    SPMM_CUDA(cudaMemcpy(&h_bad, bad.p, sizeof(int), cudaMemcpyDeviceToHost));
    SPMM_REQUIRE(h_bad == 0, "coordinate outside the matrix");
    SPMM_REQUIRE(m <= INT_MAX, "expanded non-zero count exceeds the int32 rowPtr of the reference data model");

    spmm_csr_s *A = nullptr;
    int rc = make_handle(device, n_rows, n_cols, m, &A);
    if (rc)
        return rc;
    rc = alloc_arrays(A);
    if (rc)
    {
        spmm_csr_destroy(A);
        return rc;
    }
    auto fail = [&](cudaError_t e, const char *what) {
        spmm_csr_destroy(A);
        return cuda_fail(e, what, __FILE__, __LINE__);
    };
#define BUILD_CUDA(call)              \
    do                                \
    {                                 \
        cudaError_t e__ = (call);     \
        if (e__ != cudaSuccess)       \
            return fail(e__, #call);  \
    } while (0)

    if (m > 0)
    {
        DevBuf key, key_alt, vkey, vkey_alt, xval, idx, idx_alt, gkey;
        BUILD_CUDA(key.alloc(sizeof(unsigned long long) * (size_t)m));
        BUILD_CUDA(key_alt.alloc(sizeof(unsigned long long) * (size_t)m));
        BUILD_CUDA(vkey.alloc(sizeof(unsigned long long) * (size_t)m));
        BUILD_CUDA(vkey_alt.alloc(sizeof(unsigned long long) * (size_t)m));
        BUILD_CUDA(xval.alloc(sizeof(double) * (size_t)m));
        BUILD_CUDA(idx.alloc(sizeof(unsigned) * (size_t)m));
        BUILD_CUDA(idx_alt.alloc(sizeof(unsigned) * (size_t)m));
        BUILD_CUDA(gkey.alloc(sizeof(unsigned long long) * (size_t)m));
        coo_expand_kernel<<<blocks_for(n), TPB, 0, st>>>(d_rows, d_cols, d_vals, n, symmetric ? flag.as<int>() : nullptr,
                                                        symmetric ? pos.as<int>() : nullptr,
                                                        key.as<unsigned long long>(), vkey.as<unsigned long long>(),
                                                        xval.as<double>(), idx.as<unsigned>());
        BUILD_CUDA(cudaGetLastError());

        // pass 1: order record ids by value
        cub::DoubleBuffer<unsigned long long> vk(vkey.as<unsigned long long>(), vkey_alt.as<unsigned long long>());
        cub::DoubleBuffer<unsigned> ids(idx.as<unsigned>(), idx_alt.as<unsigned>());
        size_t tmp_bytes = 0;
        BUILD_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, vk, ids, (int)m, 0, 64, st));
        {
            DevBuf tmp;
            BUILD_CUDA(tmp.alloc(tmp_bytes));
            BUILD_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, vk, ids, (int)m, 0, 64, st));
            BUILD_CUDA(cudaStreamSynchronize(st));
        }
        // pass 2: stable sort by row:col of the value-ordered ids
        gather_keys_kernel<<<blocks_for(m), TPB, 0, st>>>(key.as<unsigned long long>(), ids.Current(), m,
                                                         gkey.as<unsigned long long>());
        BUILD_CUDA(cudaGetLastError());
        cub::DoubleBuffer<unsigned long long> rk(gkey.as<unsigned long long>(), key_alt.as<unsigned long long>());
        const int end_bit = 32 + bits_for((unsigned long long)std::max(n_rows, 1));
        tmp_bytes = 0;
        BUILD_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, rk, ids, (int)m, 0, end_bit, st));
        {
            DevBuf tmp;
            BUILD_CUDA(tmp.alloc(tmp_bytes));
            BUILD_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, rk, ids, (int)m, 0, end_bit, st));
            BUILD_CUDA(cudaStreamSynchronize(st));
        }
        emit_csr_kernel<<<blocks_for(m), TPB, 0, st>>>(rk.Current(), ids.Current(), xval.as<double>(), m, A->d_colidx,
                                                      A->d_vals);
        BUILD_CUDA(cudaGetLastError());
        rowptr_kernel<<<blocks_for((long long)n_rows + 1), TPB, 0, st>>>(rk.Current(), m, n_rows, A->d_rowptr);
        BUILD_CUDA(cudaGetLastError());
        BUILD_CUDA(cudaStreamSynchronize(st));
    }
    else
    {
        BUILD_CUDA(cudaMemset(A->d_rowptr, 0, sizeof(int) * ((size_t)n_rows + 1)));
    }
#undef BUILD_CUDA
    rc = build_schedule(A, nullptr);
    if (rc)
    {
        spmm_csr_destroy(A);
        return rc;
    }
    *out = A;
    return SPMM_OK;
}

// ---- column block ----------------------------------------------------------------------
namespace
{
__global__ void colblock_count_kernel(const int *rowptr, const int *colidx, int n_rows, int c0, int c1, int *count)
{
    const long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (r >= n_rows)
        return;
    int n = 0;
    for (int j = rowptr[r]; j < rowptr[r + 1]; ++j)
    {
        const int c = colidx[j];
        n += (c >= c0 && c < c1) ? 1 : 0;
    }
    count[r] = n;
}
__global__ void colblock_fill_kernel(const int *rowptr, const int *colidx, const double *vals, int n_rows, int c0, int c1,
                                     const int *out_rowptr, int *out_colidx, double *out_vals)
{
    const long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (r >= n_rows)
        return;
    int o = out_rowptr[r];
    for (int j = rowptr[r]; j < rowptr[r + 1]; ++j)
    {
        const int c = colidx[j];
        if (c >= c0 && c < c1)
        {
            out_colidx[o] = c - c0;
            out_vals[o] = vals[j];
            ++o;
        }
    }
}

// ---- generators ------------------------------------------------------------------------
// Row i: nnz_per_row distinct ascending columns, one per stratum of the window
// [ws, ws+wd) with ws = clamp(i - hb, 0, n - wd), wd = min(2*hb+1, n).
__global__ void banded_kernel(int n, int row_begin, int n_local, int npr, int hb, unsigned long long seed, int *rowptr,
                              int *colidx, double *vals)
{
    const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long total = (long long)n_local * npr;
    if (t <= n_local)
        rowptr[t] = (int)(t * npr);
    if (t >= total)
        return;
    const int lr = (int)(t / npr), s = (int)(t % npr);
    const long long i = (long long)row_begin + lr;
    const long long wd = min((long long)2 * hb + 1, (long long)n);
    long long ws = i - hb;
    ws = max(0LL, min(ws, (long long)n - wd));
    const long long a = (long long)s * wd / npr, b = (long long)(s + 1) * wd / npr;
    const unsigned long long h = splitmix64(seed ^ splitmix64((unsigned long long)i * 0x100000001B3ULL + (unsigned long long)s));
    colidx[t] = (int)(ws + a + (long long)(h % (unsigned long long)(b - a)));
    vals[t] = 0.5 + u01(splitmix64(h));
}

__global__ void rmat_kernel(int scale, long long n_edges, double a, double b, double c, unsigned long long seed, int *rows,
                            int *cols, double *vals)
{
    const long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (e >= n_edges)
        return;
    unsigned long long h = splitmix64(seed ^ splitmix64((unsigned long long)e));
    int r = 0, col = 0;
    for (int lvl = 0; lvl < scale; ++lvl)
    {
        h = splitmix64(h);
        const double p = u01(h);
        const int rb = p >= a + b ? 1 : 0;                    // lower half of the quadrant grid
        const int cb = (p >= a && p < a + b) || p >= a + b + c; // right half
        r = (r << 1) | rb;
        col = (col << 1) | cb;
    }
    rows[e] = r;
    cols[e] = col;
    vals[e] = 0.5 + u01(splitmix64(h ^ 0xD1B54A32D192ED03ULL));
}

__global__ void fatvec_kernel(double *out, long long n, long long first, unsigned long long seed)
{
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n)
        out[i] = (double)(splitmix64(seed ^ splitmix64((unsigned long long)(first + i))) % 100ULL + 1ULL);
}
} // namespace

} // namespace spmm

using namespace spmm;

extern "C"
{

int spmm_csr_from_coo_device(int device, int n_rows, int n_cols, long long n_entries, const int *d_rows,
                             const int *d_cols, const double *d_vals, int symmetric, spmm_csr_t *out)
{
    SPMM_REQUIRE(n_rows >= 0 && n_cols >= 0, "negative size");
    int count = 0;
    SPMM_CUDA(cudaGetDeviceCount(&count));
    SPMM_REQUIRE(device >= 0 && device < count, "no such CUDA device");
    return csr_from_coo_device_impl(device, n_rows, n_cols, n_entries, d_rows, d_cols, d_vals, symmetric, out);
}

int spmm_csr_from_coo_host(int device, int n_rows, int n_cols, long long n_entries, const int *rows, const int *cols,
                           const double *vals, int symmetric, spmm_csr_t *out)
{
    SPMM_REQUIRE(n_rows >= 0 && n_cols >= 0 && n_entries >= 0, "negative size");
    SPMM_REQUIRE(n_entries == 0 || (rows && cols && vals), "coordinate arrays are NULL");
    int count = 0;
    SPMM_CUDA(cudaGetDeviceCount(&count));
    SPMM_REQUIRE(device >= 0 && device < count, "no such CUDA device");
    SPMM_CUDA(cudaSetDevice(device));
    DevBuf r, c, v;
    SPMM_CUDA(r.alloc(sizeof(int) * (size_t)n_entries));
    SPMM_CUDA(c.alloc(sizeof(int) * (size_t)n_entries));
    SPMM_CUDA(v.alloc(sizeof(double) * (size_t)n_entries));
    if (n_entries)
    {
        SPMM_CUDA(cudaMemcpy(r.p, rows, sizeof(int) * (size_t)n_entries, cudaMemcpyHostToDevice));
        SPMM_CUDA(cudaMemcpy(c.p, cols, sizeof(int) * (size_t)n_entries, cudaMemcpyHostToDevice));
        SPMM_CUDA(cudaMemcpy(v.p, vals, sizeof(double) * (size_t)n_entries, cudaMemcpyHostToDevice));
    }
    return csr_from_coo_device_impl(device, n_rows, n_cols, n_entries, r.as<int>(), c.as<int>(), v.as<double>(),
                                    symmetric, out);
}

int spmm_csr_column_block(spmm_csr_t A, int col_begin, int col_end, spmm_csr_t *out)
{
    SPMM_REQUIRE(A != nullptr && out != nullptr, "handle is NULL");
    if (A->d_rowptr64)
        return refuse_offsets64("spmm_csr_column_block", "spmm_csr_download64 and a handle built from the block's arrays");
    SPMM_REQUIRE(0 <= col_begin && col_begin <= col_end && col_end <= A->n_cols, "column range outside the matrix");
    SPMM_CUDA(cudaSetDevice(A->device));
    const int n_rows = A->n_rows;
    DevBuf count, scan;
    SPMM_CUDA(count.alloc(sizeof(int) * ((size_t)n_rows + 1)));
    SPMM_CUDA(scan.alloc(sizeof(int) * ((size_t)n_rows + 1)));
    SPMM_CUDA(cudaMemset(count.p, 0, sizeof(int) * ((size_t)n_rows + 1)));
    if (n_rows)
    {
        colblock_count_kernel<<<blocks_for(n_rows), TPB>>>(A->d_rowptr, A->d_colidx, n_rows, col_begin, col_end,
                                                           count.as<int>());
        SPMM_CUDA(cudaGetLastError());
    }
    size_t tmp_bytes = 0;
    SPMM_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, count.as<int>(), scan.as<int>(), n_rows + 1));
    DevBuf tmp;
    SPMM_CUDA(tmp.alloc(tmp_bytes));
    SPMM_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, count.as<int>(), scan.as<int>(), n_rows + 1));
    int nnz = 0;
    SPMM_CUDA(cudaMemcpy(&nnz, scan.as<int>() + n_rows, sizeof(int), cudaMemcpyDeviceToHost));
    spmm_csr_s *S = nullptr;
    int rc = make_handle(A->device, n_rows, col_end - col_begin, nnz, &S);
    if (rc)
        return rc;
    rc = alloc_arrays(S);
    if (!rc)
    {
        cudaError_t e = cudaMemcpy(S->d_rowptr, scan.p, sizeof(int) * ((size_t)n_rows + 1), cudaMemcpyDeviceToDevice);
        if (e == cudaSuccess && n_rows)
        {
            colblock_fill_kernel<<<blocks_for(n_rows), TPB>>>(A->d_rowptr, A->d_colidx, A->d_vals, n_rows, col_begin,
                                                              col_end, S->d_rowptr, S->d_colidx, S->d_vals);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess)
            e = cudaDeviceSynchronize();
        if (e != cudaSuccess)
            rc = cuda_fail(e, "column block build", __FILE__, __LINE__);
    }
    if (!rc)
        rc = build_schedule(S, nullptr);
    if (rc)
    {
        spmm_csr_destroy(S);
        return rc;
    }
    *out = S;
    return SPMM_OK;
}

int spmm_gen_banded_rows(int device, int n, int row_begin, int row_end, int nnz_per_row, int half_bandwidth,
                         unsigned long long seed, spmm_csr_t *out)
{
    SPMM_REQUIRE(out != nullptr, "out handle is NULL");
    SPMM_REQUIRE(n > 0 && nnz_per_row > 0 && half_bandwidth >= 0, "sizes must be positive");
    SPMM_REQUIRE(0 <= row_begin && row_begin <= row_end && row_end <= n, "row range outside the matrix");
    const long long wd = std::min<long long>(2LL * half_bandwidth + 1, n);
    SPMM_REQUIRE(nnz_per_row <= wd, "nnz_per_row exceeds the band width");
    const int n_local = row_end - row_begin;
    const long long nnz = (long long)n_local * nnz_per_row;
    spmm_csr_s *A = nullptr;
    int rc = make_handle(device, n_local, n, nnz, &A);
    if (rc)
        return rc;
    rc = alloc_arrays(A);
    if (!rc)
    {
        banded_kernel<<<blocks_for(std::max<long long>(nnz, n_local + 1)), TPB>>>(
            n, row_begin, n_local, nnz_per_row, half_bandwidth, seed, A->d_rowptr, A->d_colidx, A->d_vals);
        cudaError_t e = cudaGetLastError();
        if (e == cudaSuccess)
            e = cudaDeviceSynchronize();
        if (e != cudaSuccess)
            rc = cuda_fail(e, "banded generator", __FILE__, __LINE__);
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

int spmm_gen_banded(int device, int n, int nnz_per_row, int half_bandwidth, unsigned long long seed, spmm_csr_t *out)
{
    return spmm_gen_banded_rows(device, n, 0, n, nnz_per_row, half_bandwidth, seed, out);
}

int spmm_gen_rmat(int device, int scale, long long n_edges, double a, double b, double c, unsigned long long seed,
                  spmm_csr_t *out)
{
    SPMM_REQUIRE(out != nullptr, "out handle is NULL");
    SPMM_REQUIRE(scale >= 1 && scale <= 30, "scale outside [1,30]");
    SPMM_REQUIRE(n_edges >= 0 && n_edges <= INT_MAX, "edge count outside int32");
    SPMM_REQUIRE(a > 0 && b >= 0 && c >= 0 && a + b + c < 1.0, "bad R-MAT probabilities");
    int count = 0;
    SPMM_CUDA(cudaGetDeviceCount(&count));
    SPMM_REQUIRE(device >= 0 && device < count, "no such CUDA device");
    SPMM_CUDA(cudaSetDevice(device));
    DevBuf r, cidx, v;
    SPMM_CUDA(r.alloc(sizeof(int) * (size_t)n_edges));
    SPMM_CUDA(cidx.alloc(sizeof(int) * (size_t)n_edges));
    SPMM_CUDA(v.alloc(sizeof(double) * (size_t)n_edges));
    if (n_edges)
    {
        rmat_kernel<<<blocks_for(n_edges), TPB>>>(scale, n_edges, a, b, c, seed, r.as<int>(), cidx.as<int>(), v.as<double>());
        SPMM_CUDA(cudaGetLastError());
    }
    const int n = 1 << scale;
    return csr_from_coo_device_impl(device, n, n, n_edges, r.as<int>(), cidx.as<int>(), v.as<double>(), 0, out);
}

int spmm_gen_fat_vector_device(int device, double *d_out, long long n_elems, long long first_elem,
                               unsigned long long seed, void *stream)
{
    SPMM_REQUIRE(n_elems >= 0, "negative size");
    if (n_elems == 0)
        return SPMM_OK;
    SPMM_REQUIRE(d_out != nullptr, "d_out is NULL");
    SPMM_CUDA(cudaSetDevice(device));
    fatvec_kernel<<<blocks_for(n_elems), TPB, 0, (cudaStream_t)stream>>>(d_out, n_elems, first_elem, seed);
    SPMM_CUDA(cudaGetLastError());
    return SPMM_OK;
}

} // extern "C"
