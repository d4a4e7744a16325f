// spmm_bsr.cu — matrices made of dense b x b blocks (b = 2..6), read as BSR straight from the CSR arrays.
//
// Replaces, for an exactly blocked A, the loop nest of
//   /root/reference "Source Code/SparseMatrixFatVectorMultiply.cpp":17-28
// An exactly b-blocked CSR already is a BSR matrix: row R*b+i stores its entries as whole groups of b consecutive
// columns, entry rowptr[R*b+i] + q*b + t is A[R*b+i, c_q + t], and c_q = colidx[rowptr[R*b] + q*b] is the same for the b
// rows of block row R. So the view is a block size validated once (bsr_check_kernel) and kept on the handle: no copy of
// the ids or values, nothing to refresh after spmm_csr_update_values_*.
// Why: the CSR kernels gather every B row piece once per non-zero, b times per block. Here a team owns a whole block row,
// loads each of the b B row pieces of a block once and feeds it to b FMAs, one per row: the B gather through L1 falls by
// b, the column-id stream by b^2. The arithmetic is the CSR kernels' own: per (row, column) one FMA chain over the row's
// entries in storage order from +0.0, so the result does not depend on the team shape, the k-slab or the launch form.
#include <algorithm>

#include "spmm_launch.cuh"

namespace spmm
{

namespace
{
// ---- the pattern rule, checked on the device -------------------------------------------
// flags[b - 2] = min over the block rows that break b-blocking of (block row << 8 | reason); ~0 when b fits
enum BsrReason : unsigned
{
    BSR_UNEQUAL = 1, // rows of one block row have different lengths
    BSR_LENGTH = 2,  // a row length is not a multiple of b
    BSR_GROUP = 3,   // a group is not the b consecutive columns c_q .. c_q+b-1 of the block row's first row
    BSR_ALIGN = 4    // a group does not start at a multiple of b
};

const char *reason_text(unsigned r)
{
    switch (r)
    {
    case BSR_UNEQUAL: return "its rows have different lengths";
    case BSR_LENGTH: return "a row length is not a multiple of the block size";
    case BSR_GROUP: return "a group of entries is not the block size's consecutive columns of the block row's first row";
    case BSR_ALIGN: return "a block column does not start at a multiple of the block size";
    }
    return "?";
}

// one warp per row; `mask` bit b = candidate block size b (2..6)
__global__ void __launch_bounds__(256) bsr_check_kernel(const int *__restrict__ rowptr, const int *__restrict__ colidx,
                                                        int n_rows, unsigned mask, unsigned long long *flags)
{
    const int lane = threadIdx.x & 31;
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n_rows; r += n_warps)
    {
        const int s = rowptr[r], len = rowptr[r + 1] - s;
        for (int b = 2; b <= 6; ++b)
        {
            if (!(mask & (1u << b)))
                continue;
            const long long R = r / b, r0 = R * b;
            const int s0 = rowptr[r0], len0 = rowptr[r0 + 1] - s0;
            unsigned reason = 0;
            if (len != len0)
                reason = BSR_UNEQUAL;
            else if (len % b)
                reason = BSR_LENGTH;
            else
            {
                bool group = false, align = false;
                for (int p = lane; p < len; p += 32)
                {
                    const int q = p / b, t = p - q * b;
                    const int cq = colidx[s0 + q * b];
                    group |= colidx[s + p] != cq + t;
                    align |= t == 0 && cq % b != 0;
                }
                group = __any_sync(0xffffffffu, group);
                align = __any_sync(0xffffffffu, align);
                reason = group ? BSR_GROUP : (align ? BSR_ALIGN : 0);
            }
            if (reason && lane == 0)
                atomicMin(flags + (b - 2), ((unsigned long long)R << 8) | reason);
        }
    }
}

// ---- CTA cuts: contiguous chunks of block rows of equal cost (non-zeros + ROW_COST per row) ----------------------
__global__ void bsr_bounds_kernel(const int *__restrict__ rowptr, int n_brows, int bd, int grid, int *__restrict__ bounds)
{
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g > grid)
        return;
    auto cost = [&](int R) { return (long long)rowptr[(long long)R * bd] + (long long)ROW_COST * bd * R; };
    int r;
    if (g == 0)
        r = 0;
    else if (g == grid)
        r = n_brows;
    else
    {
        const long long target = (cost(n_brows) * g + grid - 1) / grid;
        int lo = 0, hi = n_brows;
        while (lo < hi)
        {
            const int mid = lo + ((hi - lo) >> 1);
            if (cost(mid) < target)
                lo = mid + 1;
            else
                hi = mid;
        }
        r = lo;
    }
    bounds[g] = r;
}

struct BsrArgs
{
    const int *rowptr;
    const int *colidx;
    const double *vals;
    const double *B; // already offset to the first computed column
    double *C;       // already offset to the first computed column
    long long ldb, ldc;
    int kc;
    const int *bounds; // gridDim.x + 1 block-row cuts
};

// A team of KL lanes spans one k-tile of KL*NV*W columns and owns one block row at a time, with BD rows of accumulators.
// Per block: the block column once, the BD B row pieces once each, BD x BD values; every piece feeds BD FMAs.
template <int BD, int KL, int NV, int W>
__global__ void __launch_bounds__(THREADS) spmm_bsr_kernel(const BsrArgs a)
{
    using S = Slice<KL, NV, W>;
    constexpr int RW = 32 / KL;
    constexpr int SLOTS = (THREADS / 32) * RW;
    const int lane = threadIdx.x & 31;
    const int kl = lane % KL;
    const int slot = (threadIdx.x >> 5) * RW + lane / KL;
    const int lo = a.bounds[blockIdx.x], hi = a.bounds[blockIdx.x + 1];
    const int tile0 = (int)blockIdx.y * S::TILE;
    const unsigned mask = slice_mask<KL, NV, W>(tile0, kl, a.kc);
    const double *__restrict__ Bk = a.B + tile0 + kl * W;

    for (int R = lo + slot; R < hi; R += SLOTS)
    {
        const long long r0 = (long long)R * BD;
        int s[BD];
#pragma unroll
        for (int i = 0; i < BD; ++i)
            s[i] = a.rowptr[r0 + i];
        const int nb = (a.rowptr[r0 + 1] - s[0]) / BD; // blocks of the block row (its rows have equal lengths)
        S acc[BD];
#pragma unroll
        for (int i = 0; i < BD; ++i)
            acc[i].zero();
        int c = nb > 0 ? ld_stream_i32(a.colidx + s[0]) : 0;
        for (int q = 0; q < nb; ++q)
        {
            S b[BD];
#pragma unroll
            for (int t = 0; t < BD; ++t)
                b[t].template load<false>(Bk + (long long)(c + t) * a.ldb, mask);
            // the next block column is fetched while the B pieces are in flight
            const int cn = q + 1 < nb ? ld_stream_i32(a.colidx + s[0] + (q + 1) * BD) : 0;
            double x[BD][BD];
#pragma unroll
            for (int i = 0; i < BD; ++i)
#pragma unroll
                for (int t = 0; t < BD; ++t)
                    x[i][t] = ld_stream_f64(a.vals + s[i] + q * BD + t);
            // storage order: for row i the entries (q, 0), (q, 1), ... follow (q-1, BD-1)
#pragma unroll
            for (int t = 0; t < BD; ++t)
#pragma unroll
                for (int i = 0; i < BD; ++i)
                    acc[i].fma(x[i][t], b[t]);
            c = cn;
        }
#pragma unroll
        for (int i = 0; i < BD; ++i)
            acc[i].store(a.C + (r0 + i) * a.ldc + tile0 + kl * W, mask);
    }
}

template <int BD, int KL, int NV, int W>
int launch_bsr_t(const spmm_csr_s *A, BsrArgs args, int tiles, cudaStream_t stream)
{
    auto kern = spmm_bsr_kernel<BD, KL, NV, W>;
    int per_sm = 1;
    int rc = kernel_info(kern, &per_sm);
    if (rc)
        return rc;
    constexpr int SLOTS = (THREADS / 32) * (32 / KL);
    const int n_brows = A->n_rows / BD;
    const int grid = (int)std::max(1LL, std::min((long long)device_props(A->device).sm_count * per_sm,
                                                  ((long long)n_brows + SLOTS - 1) / SLOTS));
    // kind 9 + (grid size in the key): the cuts depend on BD too; spmm_csr_build_bsr drops them when BD changes
    rc = cached_bounds(A, 9, grid, stream, &args.bounds, [&](int *out) {
        bsr_bounds_kernel<<<(grid + 256) / 256, 256, 0, stream>>>(A->d_rowptr, n_brows, BD, grid, out);
    });
    if (rc)
        return rc;
    kern<<<dim3((unsigned)grid, (unsigned)tiles), THREADS, 0, stream>>>(args);
    SPMM_CUDA(cudaGetLastError());
    return SPMM_OK;
}

// Team shape: the k-tile KL*NV*W covers the columns with KL up to 32 lanes. BD x NV*W accumulators and the BD B pieces
// in flight stay in registers: NV = 2 only for BD <= 3 (24 accumulators at BD = 3); larger blocks take more k-tiles.
template <int BD, int W>
int launch_bsr_bd(const spmm_csr_s *A, const BsrArgs &args, cudaStream_t stream)
{
    const int kq = (args.kc + W - 1) / W;
    int kl = 32, nv = 1;
    if (kq <= 32)
        for (kl = 1; kl < kq; kl <<= 1)
            ;
    if (BD <= 3 && kq > 8)
    {
        nv = 2;
        kl = kq <= 16 ? 8 : (kq <= 32 ? 16 : 32);
    }
    const int tiles = (kq + kl * nv - 1) / (kl * nv);
    if (nv == 2)
    {
        if constexpr (BD <= 3)
        {
            switch (kl)
            {
            case 8: return launch_bsr_t<BD, 8, 2, W>(A, args, tiles, stream);
            case 16: return launch_bsr_t<BD, 16, 2, W>(A, args, tiles, stream);
            case 32: return launch_bsr_t<BD, 32, 2, W>(A, args, tiles, stream);
            }
        }
    }
    else
    {
        switch (kl)
        {
        case 1: return launch_bsr_t<BD, 1, 1, W>(A, args, tiles, stream);
        case 2: return launch_bsr_t<BD, 2, 1, W>(A, args, tiles, stream);
        case 4: return launch_bsr_t<BD, 4, 1, W>(A, args, tiles, stream);
        case 8: return launch_bsr_t<BD, 8, 1, W>(A, args, tiles, stream);
        case 16: return launch_bsr_t<BD, 16, 1, W>(A, args, tiles, stream);
        case 32: return launch_bsr_t<BD, 32, 1, W>(A, args, tiles, stream);
        }
    }
    set_error("bsr kernel: unsupported team shape");
    return SPMM_ERR_UNSUPPORTED;
}

template <int W>
int launch_bsr_w(const spmm_csr_s *A, const BsrArgs &args, cudaStream_t stream)
{
    switch (A->bsr_b)
    {
    case 2: return launch_bsr_bd<2, W>(A, args, stream);
    case 3: return launch_bsr_bd<3, W>(A, args, stream);
    case 4: return launch_bsr_bd<4, W>(A, args, stream);
    case 5: return launch_bsr_bd<5, W>(A, args, stream);
    case 6: return launch_bsr_bd<6, W>(A, args, stream);
    }
    set_error("bsr kernel: spmm_csr_build_bsr was not called");
    return SPMM_ERR_INVALID;
}
} // namespace

int launch_bsr(const spmm_csr_s *A, const double *d_B, long long ldb, double *d_C, long long ldc, int kc, cudaStream_t stream)
{
    if (A->n_rows == 0 || kc <= 0)
        return SPMM_OK;
    BsrArgs args = {};
    args.rowptr = A->d_rowptr;
    args.colidx = A->d_colidx;
    args.vals = A->d_vals;
    args.B = d_B;
    args.C = d_C;
    args.ldb = ldb;
    args.ldc = ldc;
    args.kc = kc;
    // 16-byte accesses under the conditions of the CSR kernels (spmm_dispatch.cu, pick_shape)
    const bool even = kc % 2 == 0 && ldb % 2 == 0 && ldc % 2 == 0 && (uintptr_t)d_B % 16 == 0 && (uintptr_t)d_C % 16 == 0;
    note_kernel("spmm_bsr_kernel");
    return even ? launch_bsr_w<2>(A, args, stream) : launch_bsr_w<1>(A, args, stream);
}

} // namespace spmm

using namespace spmm;

extern "C" int spmm_csr_build_bsr(spmm_csr_t A, int block_dim, int *out_dim)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    if (A->d_rowptr64)
        return refuse_offsets64("spmm_csr_build_bsr", "SPMM_KERNEL_AUTO, ROWS, MERGE or STREAM");
    SPMM_REQUIRE(block_dim == -1 || block_dim == 0 || (block_dim >= 2 && block_dim <= 6),
                 "block_dim must be 0 (drop the view), 2..6, or -1 (largest that fits)");
    auto set = [&](int b) {
        if (b != A->bsr_b)
            drop_bounds(A, 9);
        A->bsr_b = b;
        if (out_dim)
            *out_dim = b;
        return SPMM_OK;
    };
    if (block_dim == 0)
        return set(0);
    unsigned mask = 0;
    for (int b = 2; b <= 6; ++b)
        if ((block_dim == -1 || block_dim == b) && A->n_rows % b == 0)
            mask |= 1u << b;
    if (block_dim > 0 && !mask)
    {
        set_error("spmm_csr_build_bsr: " + std::to_string(A->n_rows) + " rows are not a multiple of the block size " +
                  std::to_string(block_dim));
        return SPMM_ERR_UNSUPPORTED;
    }
    unsigned long long h[5];
    std::fill(h, h + 5, ~0ull);
    if (mask && A->n_rows > 0)
    {
        SPMM_CUDA(cudaSetDevice(A->device));
        unsigned long long *d = nullptr;
        SPMM_CUDA(cudaMalloc(&d, sizeof h));
        cudaError_t e = cudaMemcpy(d, h, sizeof h, cudaMemcpyHostToDevice);
        if (e == cudaSuccess)
        {
            const int blocks = (int)std::min<long long>(((long long)A->n_rows * 32 + 255) / 256,
                                                        (long long)device_props(A->device).sm_count * 16);
            bsr_check_kernel<<<blocks, 256>>>(A->d_rowptr, A->d_colidx, A->n_rows, mask, d);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess)
            e = cudaMemcpy(h, d, sizeof h, cudaMemcpyDeviceToHost);
        cudaFree(d);
        SPMM_CUDA(e);
    }
    if (block_dim > 0)
    {
        const unsigned long long f = h[block_dim - 2];
        if (f != ~0ull)
        {
            set_error("spmm_csr_build_bsr: the pattern is not " + std::to_string(block_dim) + "x" +
                      std::to_string(block_dim) + "-blocked: block row " + std::to_string(f >> 8) + " (rows " +
                      std::to_string((f >> 8) * block_dim) + ".." + std::to_string((f >> 8) * block_dim + block_dim - 1) +
                      "): " + reason_text((unsigned)(f & 0xff)));
            return SPMM_ERR_UNSUPPORTED;
        }
        return set(block_dim);
    }
    for (int b = 6; b >= 2; --b)
        if ((mask & (1u << b)) && h[b - 2] == ~0ull)
            return set(b);
    return set(0);
}
