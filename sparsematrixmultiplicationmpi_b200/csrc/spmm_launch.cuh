// spmm_launch.cuh — team-shape selection and template dispatch for the row kernel and
// the merge-path kernel (spmm_kernels.cuh). Included by one translation unit per
// vector width W (spmm_w1.cu: 8-byte accesses, spmm_w2.cu: 16-byte accesses) so the
// instantiations compile in parallel.
//
// Team shape:
//   W   doubles per access  = 2 when k, ldb, ldc are even and B/C are 16-byte aligned, else 1
//   KL  lanes across a row  / NV accesses per lane: the smallest team whose KL*NV*W covers k
//                             with KL >= 8 once a piece of a B row fills a 128-byte line
//   NP  non-zeros of one row side by side (only when NV == 1): from the mean row length
//   U   steps in flight
// All of these can be overridden through spmm_tune_set() for measurement.
#pragma once
#include <algorithm>
#include <map>
#include <mutex>
#include <unordered_map>

#include "spmm_internal.h"
#include "spmm_kernels.cuh"

namespace spmm
{

constexpr int THREADS = 256;

struct KernelInfo
{
    int ctas_per_sm = 0;
};

// One-time per-kernel set-up: give the whole unified array to L1D (B-row reuse lives
// there; the kernels use a few bytes of static smem only) and query occupancy.
template <typename K>
int kernel_info(K kern, int *ctas_per_sm)
{
    static std::mutex mu;
    static std::map<std::pair<const void *, int>, KernelInfo> cache; // function attributes and occupancy are per device
    int dev = 0;
    SPMM_CUDA(cudaGetDevice(&dev));
    const void *fn = (const void *)kern;
    const std::pair<const void *, int> key(fn, dev);
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(key);
    if (it == cache.end())
    {
        SPMM_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, 0));
        KernelInfo ki;
        SPMM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ki.ctas_per_sm, kern, THREADS, 0));
        if (ki.ctas_per_sm < 1)
            ki.ctas_per_sm = 1;
        it = cache.emplace(key, ki).first;
    }
    *ctas_per_sm = it->second.ctas_per_sm;
    return SPMM_OK;
}

template <int KL, int NV, int W, int NP, int U, bool FULL>
int launch_rows_full(const spmm_csr_s *A, const SpmmArgs &args, int tiles, int device, cudaStream_t stream)
{
    auto kern = spmm_rows_kernel<KL, NV, W, NP, U, FULL, THREADS>;
    int per_sm = 1;
    int rc = kernel_info(kern, &per_sm);
    if (rc)
        return rc;
    const Tuning &t = tuning();
    if (t.rows_ctas_per_sm > 0)
        per_sm = std::min(per_sm, t.rows_ctas_per_sm);
    constexpr int SLOTS = (THREADS / 32) * (32 / (KL * NP));
    const long long rows = (long long)args.row_end - args.row_begin;
    long long grid = (long long)device_props(device).sm_count * per_sm;
    grid = std::max(1LL, std::min(grid, (rows + SLOTS - 1) / SLOTS));
    SpmmArgs a2 = args;
    a2.bounds = nullptr;
    const Tuning &tn = tuning();
    // enough rows for >= 16 tiles per CTA: deal tiles round-robin (L2-resident B window), else one chunk per CTA
    // (tile height measured on cfg4, 2^25 banded rows x 32, k=16: 16.3 ms at 8 rows per team slot, 12.5 ms at 3 — short tiles keep
    // the CTAs of a wave on neighbouring rows, whose B window they then share in L2; gpurun_out/r2l_tune_cfg4.jsonl)
    const int tile = tn.rows_tile > 0 ? tn.rows_tile : SLOTS * 3;
    a2.tile_rows = (tn.rows_tile > 0 || (tn.rows_tile == 0 && rows >= grid * 16LL * tile)) ? tile : 0;
    if (a2.tile_rows)
        ;
    else if (args.row_begin == 0 && args.row_end == A->n_rows && args.nnz_lo == 0 && args.nnz_hi == A->nnz)
    {
        // whole matrix: the equal-cost CTA cuts are part of the handle's schedule
        rc = cached_bounds(A, 0, (int)grid, stream, &a2.bounds, [&](int *out) {
            chunk_bounds_kernel<<<((unsigned)grid + 256) / 256, 256, 0, stream>>>(args.rowptr, A->n_rows, (int)A->nnz,
                                                                             (int)grid, out);
        });
        if (rc)
            return rc;
    }
    // programmatic dependent launch: the kernel's prologue (CTA cuts, row extents, L2 prefetches) may run under the tail of the
    // kernel before it in the stream; it executes griddepcontrol.wait before it reads B or writes C (spmm_kernels.cuh)
    if (tn.tiled_pdl != 0)
    {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)grid, (unsigned)tiles);
        cfg.blockDim = dim3(THREADS);
        cfg.dynamicSmemBytes = 0;
        cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        SPMM_CUDA(cudaLaunchKernelEx(&cfg, kern, a2));
    }
    else
        kern<<<dim3((unsigned)grid, (unsigned)tiles), THREADS, 0, stream>>>(a2);
    SPMM_CUDA(cudaGetLastError());
    return SPMM_OK;
}

template <int KL, int NV, int W, int NP, int U>
int launch_rows_one(const spmm_csr_s *A, const SpmmArgs &args, int tiles, int device, cudaStream_t stream)
{
    // FULL: the k columns fill every chunk of every column tile
    if (args.kc == tiles * KL * NV * W)
        return launch_rows_full<KL, NV, W, NP, U, true>(A, args, tiles, device, stream);
    return launch_rows_full<KL, NV, W, NP, U, false>(A, args, tiles, device, stream);
}

template <int KL, int NV, int W, int NP>
int launch_rows_u(const spmm_csr_s *A, int u, const SpmmArgs &a, int tiles, int dev, cudaStream_t s)
{
    if constexpr (NP >= 8)
    {
        if (u >= 2)
            return launch_rows_one<KL, NV, W, NP, 2>(A, a, tiles, dev, s);
        return launch_rows_one<KL, NV, W, NP, 1>(A, a, tiles, dev, s);
    }
    else if constexpr (NP >= 2)
    {
        if (u >= 4)
            return launch_rows_one<KL, NV, W, NP, 4>(A, a, tiles, dev, s);
        if (u >= 2)
            return launch_rows_one<KL, NV, W, NP, 2>(A, a, tiles, dev, s);
        return launch_rows_one<KL, NV, W, NP, 1>(A, a, tiles, dev, s);
    }
    else
    {
        if constexpr (NV <= 2)
            if (u >= 8)
                return launch_rows_one<KL, NV, W, NP, 8>(A, a, tiles, dev, s);
        if (u >= 4)
            return launch_rows_one<KL, NV, W, NP, 4>(A, a, tiles, dev, s);
        if (u >= 2)
            return launch_rows_one<KL, NV, W, NP, 2>(A, a, tiles, dev, s);
        return launch_rows_one<KL, NV, W, NP, 1>(A, a, tiles, dev, s);
    }
}

template <int KL, int W>
int launch_rows_np(const spmm_csr_s *A, int np, int u, const SpmmArgs &a, int tiles, int dev, cudaStream_t s)
{
    constexpr int MAXNP = 32 / KL;
    np = std::max(1, std::min(np, MAXNP));
#define SPMM_NP_CASE(N)           \
    if constexpr (N <= MAXNP)     \
        if (np >= N)              \
            return launch_rows_u<KL, 1, W, N>(A, u, a, tiles, dev, s);
    SPMM_NP_CASE(32)
    SPMM_NP_CASE(16)
    SPMM_NP_CASE(8)
    SPMM_NP_CASE(4)
    SPMM_NP_CASE(2)
#undef SPMM_NP_CASE
    return launch_rows_u<KL, 1, W, 1>(A, u, a, tiles, dev, s);
}

template <int W>
int launch_rows_shape(const spmm_csr_s *A, int kl, int nv, int np, int u, const SpmmArgs &a, int tiles, int dev, cudaStream_t s)
{
    if (nv == 1)
    {
        switch (kl)
        {
        case 1: return launch_rows_np<1, W>(A, np, u, a, tiles, dev, s);
        case 2: return launch_rows_np<2, W>(A, np, u, a, tiles, dev, s);
        case 4: return launch_rows_np<4, W>(A, np, u, a, tiles, dev, s);
        case 8: return launch_rows_np<8, W>(A, np, u, a, tiles, dev, s);
        case 16: return launch_rows_np<16, W>(A, np, u, a, tiles, dev, s);
        case 32: return launch_rows_np<32, W>(A, np, u, a, tiles, dev, s);
        }
    }
    else if (nv == 2)
    {
        switch (kl)
        {
        case 8: return launch_rows_u<8, 2, W, 1>(A, u, a, tiles, dev, s);
        case 16: return launch_rows_u<16, 2, W, 1>(A, u, a, tiles, dev, s);
        case 32: return launch_rows_u<32, 2, W, 1>(A, u, a, tiles, dev, s);
        }
    }
    else if (nv == 4)
    {
        switch (kl)
        {
        case 8: return launch_rows_u<8, 4, W, 1>(A, u, a, tiles, dev, s);
        case 16: return launch_rows_u<16, 4, W, 1>(A, u, a, tiles, dev, s);
        case 32: return launch_rows_u<32, 4, W, 1>(A, u, a, tiles, dev, s);
        }
    }
    set_error("rows kernel: unsupported team shape kl=" + std::to_string(kl) + " nv=" + std::to_string(nv));
    return SPMM_ERR_UNSUPPORTED;
}

// ---- merge-path ---------------------------------------------------------------------
template <int KL, int NV, int W, int U, bool FULL>
int launch_merge_full(const SpmmArgs &args, int tiles, cudaStream_t stream)
{
    constexpr int TEAMS_PER_CTA = (THREADS / 32) * (32 / KL);
    auto kern = spmm_merge_kernel<KL, NV, W, U, FULL, THREADS>;
    auto fix = spmm_merge_fixup_kernel<KL, NV, W, THREADS>;
    int per_sm = 1;
    int rc = kernel_info(kern, &per_sm);
    if (rc)
        return rc;
    const long long grid = ((long long)args.n_teams + TEAMS_PER_CTA - 1) / TEAMS_PER_CTA;
    kern<<<dim3((unsigned)grid, (unsigned)tiles), THREADS, 0, stream>>>(args);
    SPMM_CUDA(cudaGetLastError());
    const long long fgrid = (2LL * args.n_teams + TEAMS_PER_CTA - 1) / TEAMS_PER_CTA;
    fix<<<dim3((unsigned)fgrid, (unsigned)tiles), THREADS, 0, stream>>>(args);
    SPMM_CUDA(cudaGetLastError());
    return SPMM_OK;
}

template <int KL, int NV, int W, int U>
int launch_merge_one(const SpmmArgs &args, int tiles, cudaStream_t stream)
{
    if (args.kc == tiles * KL * NV * W)
        return launch_merge_full<KL, NV, W, U, true>(args, tiles, stream);
    return launch_merge_full<KL, NV, W, U, false>(args, tiles, stream);
}

template <int KL, int NV, int W>
int launch_merge_u(int u, const SpmmArgs &a, int tiles, cudaStream_t s)
{
    // (unroll 1 and 8 were measured on cfg3 and lost to 2 and 4: gpurun_out/s5_tune_mb1.jsonl)
    if (u >= 4)
        return launch_merge_one<KL, NV, W, 4>(a, tiles, s);
    return launch_merge_one<KL, NV, W, 2>(a, tiles, s);
}

template <int W>
int launch_merge_shape(int kl, int nv, int u, const SpmmArgs &a, int tiles, cudaStream_t s)
{
#define SPMM_M_CASE(K, N)        \
    if (kl == K && nv == N)      \
        return launch_merge_u<K, N, W>(u, a, tiles, s);
    SPMM_M_CASE(1, 1)
    SPMM_M_CASE(2, 1)
    SPMM_M_CASE(4, 1)
    SPMM_M_CASE(8, 1)
    SPMM_M_CASE(8, 2)
    SPMM_M_CASE(8, 4)
    SPMM_M_CASE(16, 1)
    SPMM_M_CASE(16, 2)
    SPMM_M_CASE(16, 4)
    SPMM_M_CASE(32, 1)
    SPMM_M_CASE(32, 2)
    SPMM_M_CASE(32, 4)
#undef SPMM_M_CASE
    set_error("merge kernel: unsupported team shape kl=" + std::to_string(kl) + " nv=" + std::to_string(nv));
    return SPMM_ERR_UNSUPPORTED;
}

// entry points of the two per-W translation units
int launch_rows_w1(const spmm_csr_s *A, int kl, int nv, int np, int u, const SpmmArgs &a, int tiles, int dev, cudaStream_t s);
int launch_rows_w2(const spmm_csr_s *A, int kl, int nv, int np, int u, const SpmmArgs &a, int tiles, int dev, cudaStream_t s);
int launch_merge_w1(int kl, int nv, int u, const SpmmArgs &a, int tiles, cudaStream_t s);
int launch_merge_w2(int kl, int nv, int u, const SpmmArgs &a, int tiles, cudaStream_t s);

} // namespace spmm
