// spmm_kernels.cuh — sm_100a SpMM kernels: C = A * B, A CSR (FP64 values, int32 ids),
// B/C dense row-major FP64 ("fat vectors").
//
// Replaces the reference's host triple loop
//   /root/reference "Source Code/SparseMatrixFatVectorMultiply.cpp":17-28
// and the per-rank loops of the three strategies (RowWise.cpp:36-50,
// ColumnWise.cpp:34-48, NonZeroElement.cpp:56-67).
//
// The path is not a dense contraction: no tensor cores. It is bound by HBM
// (A streamed once, B and C touched once) and, at large k, by the L1 -> register
// gather of B rows (128 B/clk/SM). Design rules used below (DESIGN.md has the
// arithmetic):
//   * a "team" of KL lanes maps across the k columns of a B row. Lane kl owns NV
//     chunks of W doubles (W=2: one 16-byte load) interleaved at stride KL*W, so
//     every load instruction of a team covers one contiguous KL*W*8-byte piece of
//     the B row (a full 128-byte line for KL=8, W=2) — no half-used L1 wavefronts;
//   * 32/(KL*NP) teams share a warp, each on its own row, so one index/value load
//     instruction serves several non-zeros; NP>1 puts NP non-zeros of the SAME row
//     side by side (small k) and folds them with warp shuffles;
//   * every CTA owns ONE CONTIGUOUS chunk of rows, cut so that chunks cost the
//     same (nnz + row overhead), and the grid is one resident wave
//     (SMs x CTAs/SM): neighbouring rows of FEM-like matrices share B rows, and
//     a contiguous sweep turns that into L1 hits instead of L2 traffic;
//   * A (col ids, values) is streamed with L1::no_allocate so it does not evict
//     B rows from L1; C is written with streaming stores;
//   * U steps of independent B-row loads are in flight per team before the FMAs.
//
// Row extents are always read through RowClip: the per-rank non-zero range of
// the NonZeroElement strategy (NonZeroElement.cpp:24-39) is the same CSR with
// every row clipped to [nnz_lo, nnz_hi).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace spmm
{

// ---- cache-hinted accessors ------------------------------------------------------
#if defined(SPMM_ABLATE) && (SPMM_ABLATE & 1) // diagnostic build: A stream allocates in L1
#define SPMM_A_HINT ""
#else
#define SPMM_A_HINT ".L1::no_allocate"
#endif
__device__ __forceinline__ int ld_stream_i32(const int *p)
{
    int v;
    asm("ld.global.nc" SPMM_A_HINT ".s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ double ld_stream_f64(const double *p)
{
    double v;
    asm("ld.global.nc" SPMM_A_HINT ".f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ int ld_b_i32(const int *p)
{
    int v;
    asm("ld.global.nc.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ double ld_b1(const double *p)
{
    double v;
    asm("ld.global.nc.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ double2 ld_b2(const double *p)
{
    double2 v;
    asm("ld.global.nc.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_c1(double *p, double v)
{
    asm volatile("st.global.cs.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ void st_c2(double *p, double x, double y)
{
    asm volatile("st.global.cs.v2.f64 [%0], {%1, %2};" ::"l"(p), "d"(x), "d"(y) : "memory");
}

// Fire-and-forget TMA prefetch of a byte range into L2 (UBLKPF.L2). Called by every thread of a
// CTA; thread t takes the pieces t, t+THREADS, ... of `piece` bytes. base must be 16-byte aligned.
__device__ __forceinline__ void bulk_prefetch_l2(const char *base, size_t bytes, int tid, int nthreads)
{
    constexpr size_t piece = 4096;
    bytes &= ~(size_t)15;
    for (size_t off = (size_t)tid * piece; off < bytes; off += (size_t)nthreads * piece)
    {
        const unsigned n = (unsigned)(bytes - off < piece ? bytes - off : piece);
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(base + off), "r"(n) : "memory");
    }
}

// Row extents clipped to a non-zero range (no-op for the whole matrix).
struct RowClip
{
    const int *rowptr;
    int lo, hi;
    __device__ __forceinline__ int operator()(int r) const { return min(max(rowptr[r], lo), hi); }
};

// The slice of one B/C row a lane owns: NV chunks of W doubles, chunk i at
// column (i*KL + kl)*W of the launch's column tile.
template <int KL, int NV, int W>
struct Slice
{
    double v[NV * W];
    static constexpr int TILE = KL * NV * W; // columns covered by one team
    __device__ __forceinline__ void zero()
    {
#pragma unroll
        for (int i = 0; i < NV * W; ++i)
            v[i] = 0.0;
    }
    // p = row base + tile base + kl*W; `mask` bit i = chunk i lies inside the k columns.
    // FULL (every chunk inside): unconditional loads, which ptxas batches ahead of the FMAs.
    template <bool FULL>
    __device__ __forceinline__ void load(const double *p, unsigned mask)
    {
#pragma unroll
        for (int i = 0; i < NV; ++i)
        {
            if constexpr (!FULL)
            {
#pragma unroll
                for (int w = 0; w < W; ++w)
                    v[i * W + w] = 0.0;
                if (!(mask & (1u << i)))
                    continue;
            }
            if constexpr (W == 2)
            {
                double2 t = ld_b2(p + i * KL * W);
                v[2 * i] = t.x;
                v[2 * i + 1] = t.y;
            }
            else
                v[i] = ld_b1(p + i * KL * W);
        }
    }
    __device__ __forceinline__ void store(double *p, unsigned mask) const
    {
#pragma unroll
        for (int i = 0; i < NV; ++i)
            if (mask & (1u << i))
            {
                if constexpr (W == 2)
                    st_c2(p + i * KL * W, v[2 * i], v[2 * i + 1]);
                else
                    st_c1(p + i * KL * W, v[i]);
            }
    }
    // plain (cached) store/load for the merge kernel's carry rows
    __device__ __forceinline__ void store_plain(double *p) const
    {
#pragma unroll
        for (int i = 0; i < NV; ++i)
#pragma unroll
            for (int w = 0; w < W; ++w)
                p[i * KL * W + w] = v[i * W + w];
    }
    __device__ __forceinline__ void add_plain(const double *p)
    {
#pragma unroll
        for (int i = 0; i < NV; ++i)
#pragma unroll
            for (int w = 0; w < W; ++w)
                v[i * W + w] += p[i * KL * W + w];
    }
    __device__ __forceinline__ void load_plain(const double *p) // volatile: a group of these is issued back to back
    {
#pragma unroll
        for (int i = 0; i < NV; ++i)
        {
            if constexpr (W == 2)
                asm volatile("ld.global.v2.f64 {%0, %1}, [%2];" : "=d"(v[2 * i]), "=d"(v[2 * i + 1]) : "l"(p + i * KL * W));
            else
                asm volatile("ld.global.f64 %0, [%1];" : "=d"(v[i]) : "l"(p + i * KL * W));
        }
    }
    __device__ __forceinline__ void add(const Slice &b)
    {
#pragma unroll
        for (int i = 0; i < NV * W; ++i)
            v[i] += b.v[i];
    }
    __device__ __forceinline__ void add_if(const Slice &b, bool c) // (adds +0.0 otherwise: no branch around the loads)
    {
#pragma unroll
        for (int i = 0; i < NV * W; ++i)
            v[i] += c ? b.v[i] : 0.0;
    }
    __device__ __forceinline__ void fma(double a, const Slice &b)
    {
#if defined(SPMM_ABLATE) && (SPMM_ABLATE & 64) // diagnostic: one integer op per loaded double instead of a DFMA
#pragma unroll
        for (int i = 0; i < NV * W; ++i)
            v[i] = __longlong_as_double(__double_as_longlong(v[i]) ^ __double_as_longlong(b.v[i]) ^ __double_as_longlong(a));
#else
#pragma unroll
        for (int i = 0; i < NV * W; ++i)
            v[i] = ::fma(a, b.v[i], v[i]);
#endif
    }
};

template <int KL, int NV, int W>
__device__ __forceinline__ unsigned slice_mask(int tile0, int kl, int kc)
{
    unsigned m = 0;
#pragma unroll
    for (int i = 0; i < NV; ++i)
        if (tile0 + (i * KL + kl) * W < kc) // W==2 launches have even kc: a chunk is all in or all out
            m |= 1u << i;
    return m;
}

// Cost model used to cut rows into equal-cost contiguous chunks: one unit per
// non-zero plus ROW_COST units per row (row-pointer loads, C store, loop set-up).
constexpr int ROW_COST = 4;

__device__ __forceinline__ long long chunk_cost(const RowClip &rp, int row_begin, int r)
{
    return (long long)(rp(r) - rp(row_begin)) + (long long)ROW_COST * (r - row_begin);
}

// First row r in [row_begin,row_end] whose prefix cost reaches `target`: a 32-ary search by one
// warp (all 32 lanes must call it) — 4 rounds of independent probes for 10^5..10^6 rows instead of
// 17-20 dependent cache misses.
__device__ __forceinline__ int chunk_lower_bound_warp(const RowClip &rp, int row_begin, int row_end, long long target)
{
    const int lane = threadIdx.x & 31;
    int l = row_begin, h = row_end; // answer in [l, h]
    while (h > l)
    {
        const int step = (h - l + 31) >> 5;
        const int m = min(l + lane * step, h);
        const bool ge = chunk_cost(rp, row_begin, m) >= target;
        const unsigned bal = __ballot_sync(0xffffffffu, ge);
        if (bal == 0)
            l = min(l + 31 * step, h - 1) + 1;
        else
        {
            const int f = __ffs(bal) - 1;
            const int nh = min(l + f * step, h);
            if (f > 0)
                l = min(l + (f - 1) * step, h) + 1;
            h = nh;
        }
    }
    return l;
}

// Equal-cost contiguous chunk [lo,hi) of CTA b out of g. `bounds` (g+1 entries, precomputed once per
// handle and grid size for whole-matrix launches) short-cuts the search.
__device__ __forceinline__ void cta_chunk(const RowClip &rp, int row_begin, int row_end, const int *bounds, int *s_chunk)
{
    const long long g = gridDim.x, b = blockIdx.x;
    if (bounds)
    {
        if (threadIdx.x < 2)
            s_chunk[threadIdx.x] = bounds[b + threadIdx.x];
    }
    else if (threadIdx.x < 64)
    {
        const int w = threadIdx.x >> 5;
        const long long total = chunk_cost(rp, row_begin, row_end);
        const long long bb = b + w;
        int r;
        if (bb == 0)
            r = row_begin;
        else if (bb == g)
            r = row_end;
        else
            r = chunk_lower_bound_warp(rp, row_begin, row_end, (total * bb + g - 1) / g);
        if ((threadIdx.x & 31) == 0)
            s_chunk[w] = r;
    }
    __syncthreads();
}

// One thread per CTA boundary: the same cuts, computed once (spmm_dispatch.cu caches them per handle).
static __global__ void chunk_bounds_kernel(const int *rowptr, int n_rows, int nnz, int grid, int *bounds)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b > grid)
        return;
    const RowClip rp{rowptr, 0, nnz};
    const long long total = chunk_cost(rp, 0, n_rows);
    int r;
    if (b == 0)
        r = 0;
    else if (b == grid)
        r = n_rows;
    else
    {
        const long long target = (total * b + grid - 1) / grid;
        int lo = 0, hi = n_rows;
        while (lo < hi)
        {
            const int mid = lo + ((hi - lo) >> 1);
            if (chunk_cost(rp, 0, mid) < target)
                lo = mid + 1;
            else
                hi = mid;
        }
        r = lo;
    }
    bounds[b] = r;
}

// Extra destinations of the C rows a launch produces (peer GPUs' buffers mapped over NVLink): element offsets
// relative to the primary C pointer, same leading dimension. The kernel stores every finished row piece to all
// of them from registers — the row-wise strategy's gather / all-gather fused into the multiply.
constexpr int SPMM_MAX_EXTRA = 7;
struct ExtraDst
{
    int n = 0;
    long long off[SPMM_MAX_EXTRA] = {0, 0, 0, 0, 0, 0, 0};
};

struct SpmmArgs
{
    ExtraDst extra;
    const int *rowptr;
    const int *colidx;
    const double *vals;
    const double *B; // already offset to the first computed column
    double *C;       // already offset to the first computed column; row `c_row0` is at C[0]
    long long ldb, ldc;
    int row_begin, row_end; // rows computed by this launch
    int nnz_lo, nnz_hi;     // rows are clipped to this non-zero range
    int c_row0;             // row id stored at C[0]
    int kc;                 // columns computed
    const int *bounds;      // optional precomputed CTA row cuts (gridDim.x+1 entries)
    int tile_rows;          // > 0: CTAs take row tiles of this size round-robin (b, b+grid, ...) instead of one chunk
    int prefetch;           // bit0: CTA prefetches its own A chunk into L2; bit1: its share of B
    long long b_bytes;      // bytes of the B operand (0: not contiguous, no prefetch)
    // merge-path kernel only
    int items_per_team;
    int n_teams;
    double *carry;  // [2*n_teams][ldcarry]
    int *carry_row; // [2*n_teams], -1 = unused
    int ldcarry;
};

// Resident CTAs per SM the register allocator is asked to honour: room for the U in-flight B
// slices plus double-buffered indices. Without it ptxas schedules for minimum registers and
// serialises every B load behind the FMA of the previous one (ncu: 100 % long-scoreboard stalls).
constexpr int min_blocks(int nv, int w, int u, int rows, int threads)
{
    const int est = 24 + nv * w * 2 * (rows + u) + 6 * u;
    const int mb = 65536 / (threads * est);
    return mb < 1 ? 1 : (mb > 8 ? 8 : mb);
}

// Row kernel. A team of KL*NP lanes owns one row at a time: KL lanes across the
// columns, NP non-zeros of the row in flight side by side, U steps per group.
// 32/(KL*NP) teams share a warp. Software pipeline: while the U B-row slices of a
// group are in flight, the column ids / values of the next group and the extent of
// the team's next row are already being fetched, so a group costs one memory latency.
template <int KL, int NV, int W, int NP, int U, bool FULL, int THREADS>
__global__ void __launch_bounds__(THREADS, min_blocks(NV, W, U, 1, THREADS)) spmm_rows_kernel(const SpmmArgs a)
{
    constexpr int T = KL * NP;
    constexpr int RW = 32 / T;
    constexpr int SLOTS = (THREADS / 32) * RW;
    static_assert(T <= 32 && 32 % T == 0, "team must divide a warp");
    using S = Slice<KL, NV, W>;

    const RowClip rp{a.rowptr, a.nnz_lo, a.nnz_hi};
    __shared__ int s_chunk[2];
    // programmatic dependent launch (no-ops without the launch attribute): the next kernel of the stream may start its
    // prologue as this grid drains; B is read and C written only after the grids before this one have completed
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // Large matrices: row tiles dealt round-robin, so that at any moment all CTAs of the grid work
    // inside one window of grid*tile_rows consecutive rows and the B rows they share stay in L2
    // (one far-apart chunk per CTA would keep hundreds of disjoint B windows alive at once).
    const bool tiled = a.tile_rows > 0;
    if (!tiled)
        cta_chunk(rp, a.row_begin, a.row_end, a.bounds, s_chunk);
  // chunk mode: exactly one pass; tile mode: tiles blockIdx.x, blockIdx.x + gridDim.x, ...
  const int n_tiles = tiled ? (a.row_end - a.row_begin + a.tile_rows - 1) / a.tile_rows : (int)blockIdx.x + 1;
  for (int tile_id = blockIdx.x; tile_id < n_tiles; tile_id += gridDim.x)
  {
    const int lo = tiled ? a.row_begin + tile_id * a.tile_rows : s_chunk[0];
    const int hi = tiled ? min(a.row_end, lo + a.tile_rows) : s_chunk[1];

    // L2 prefetch by the TMA unit, issued before any work: the CTA's own slice of the A stream and
    // its share of B. Every later load then finds L2-hit latency instead of a first-touch DRAM miss.
    if ((a.prefetch & 1) && !tiled)
    {
        const size_t n0 = (size_t)rp(lo), n1 = (size_t)rp(hi);
        if (n1 > n0)
        {
            const size_t c0 = (n0 * 4) & ~(size_t)15, v0 = (n0 * 8) & ~(size_t)15;
            bulk_prefetch_l2((const char *)a.colidx + c0, n1 * 4 - c0, threadIdx.x, THREADS);
            bulk_prefetch_l2((const char *)a.vals + v0, n1 * 8 - v0, threadIdx.x, THREADS);
        }
    }
    if ((a.prefetch & 2) && a.b_bytes > 0 && blockIdx.y == 0 && !tiled)
    {
        const size_t share = (((size_t)a.b_bytes + gridDim.x - 1) / gridDim.x + 15) & ~(size_t)15;
        const size_t b0 = share * blockIdx.x;
        if (b0 < (size_t)a.b_bytes)
            bulk_prefetch_l2((const char *)a.B + b0, min(share, (size_t)a.b_bytes - b0), threadIdx.x, THREADS);
    }

    asm volatile("griddepcontrol.wait;" ::: "memory");
    const int lane = threadIdx.x & 31;
    const int lt = lane % T; // lane inside the team
    const int g = lt / KL;   // which of the NP concurrent non-zeros
    const int kl = lt % KL;  // which column group
    const int slot = (threadIdx.x >> 5) * RW + lane / T;
    const int tile0 = (int)blockIdx.y * S::TILE;
    const unsigned mask = slice_mask<KL, NV, W>(tile0, kl, a.kc);
    const double *__restrict__ Bk = a.B + tile0 + kl * W;

    int row = lo + slot;
    int js = 0, je = 0;
    if (row < hi)
    {
        js = rp(row);
        je = rp(row + 1);
    }
    for (int base = lo; base < hi; base += SLOTS)
    {
        const bool valid = row < hi;
        const int nrow = row + SLOTS; // the team's next row: fetch its extent now
        int njs = 0, nje = 0;
        if (nrow < hi)
        {
            njs = rp(nrow);
            nje = rp(nrow + 1);
        }
        S acc;
        acc.zero();
        int j = js + g;
        if (j < je)
        {
            int c[U];
            double x[U];
#pragma unroll
            for (int u = 0; u < U; ++u)
            {
                const int jj = min(j + u * NP, je - 1); // clamped: a valid element, never accumulated past the end
                c[u] = ld_stream_i32(a.colidx + jj);
                x[u] = ld_stream_f64(a.vals + jj);
            }
            while (true)
            {
                S b[U];
#if defined(SPMM_ABLATE) && (SPMM_ABLATE & 2) // diagnostic: no B gather
#pragma unroll
                for (int u = 0; u < U; ++u)
#pragma unroll
                    for (int i = 0; i < NV * W; ++i)
                        b[u].v[i] = (double)c[u];
#elif defined(SPMM_ABLATE) && (SPMM_ABLATE & 8) // diagnostic: real index dependency, but every B row folded into 64 rows (all L1 hits)
#pragma unroll
                for (int u = 0; u < U; ++u)
                    b[u].template load<FULL>(Bk + (long long)(c[u] & 63) * a.ldb, mask);
#elif defined(SPMM_ABLATE) && (SPMM_ABLATE & 16) // diagnostic: B rows folded into a 16 MB window (L2 hits, L1 misses)
#pragma unroll
                for (int u = 0; u < U; ++u)
                    b[u].template load<FULL>(Bk + (long long)((c[u] * 7919) & 32767) * a.ldb, mask);
#else
#pragma unroll
                for (int u = 0; u < U; ++u)
                    b[u].template load<FULL>(Bk + (long long)c[u] * a.ldb, mask);
#endif
                const int jn = j + NP * U;
                const bool more = jn < je;
                int cn[U];
                double xn[U];
                // unconditional (clamped) so the fetch is issued while the B slices are in flight
#pragma unroll
                for (int u = 0; u < U; ++u)
                {
                    const int jj = min(jn + u * NP, je - 1);
                    cn[u] = ld_stream_i32(a.colidx + jj);
                    xn[u] = ld_stream_f64(a.vals + jj);
                }
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (j + u * NP < je)
                        acc.fma(x[u], b[u]);
                if (!more)
                    break;
#pragma unroll
                for (int u = 0; u < U; ++u)
                {
                    c[u] = cn[u];
                    x[u] = xn[u];
                }
                j = jn;
            }
        }
        if constexpr (NP > 1)
        {
#pragma unroll
            for (int off = KL; off < T; off <<= 1)
#pragma unroll
                for (int i = 0; i < NV * W; ++i)
                    acc.v[i] += __shfl_xor_sync(0xffffffffu, acc.v[i], off);
        }
#if defined(SPMM_ABLATE) && (SPMM_ABLATE & 32) // diagnostic: no C stores (kept alive by an impossible condition)
        if (valid && g == 0 && acc.v[0] == -1.2345e300)
#else
        if (valid && g == 0)
#endif
        {
            double *const cp = a.C + (long long)(row - a.c_row0) * a.ldc + tile0 + kl * W;
            acc.store(cp, mask);
            for (int d = 0; d < a.extra.n; ++d)
                acc.store(cp + a.extra.off[d], mask);
        }
        row = nrow;
        js = njs;
        je = nje;
    }
  }
}

// ---- nnz-balanced merge-path kernel ---------------------------------------------------
// The work list is the merge of the row-end offsets (one "flush" item per row) with
// the non-zero indices; every team takes items_per_team consecutive items, found by a
// diagonal binary search. A row that starts inside a team's range and ends there is
// stored straight to C. A row cut by a team boundary is never stored by the sweep:
// every team that touched it leaves its partial sum in a carry slot (head = the team
// that reaches the row's end, tail = teams that ran out of items inside the row), and
// spmm_merge_fixup_kernel adds the slots of a row in team order — deterministic, no
// atomics.
__device__ __forceinline__ void merge_path_search(const RowClip &rp, int row_begin, int n_rows, int nnz_lo,
                                                  int n_nnz, long long diag, int &x_out, int &y_out)
{
    long long x_min = diag > n_nnz ? diag - n_nnz : 0;
    long long x_max = diag < n_rows ? diag : n_rows;
    while (x_min < x_max)
    {
        const long long pivot = (x_min + x_max) >> 1;
        // row-end item `pivot` precedes non-zero item (diag - pivot - 1) when its offset is <= that index
        if ((long long)rp(row_begin + (int)pivot + 1) <= (long long)nnz_lo + (diag - pivot - 1))
            x_min = pivot + 1;
        else
            x_max = pivot;
    }
    x_out = (int)x_min;
    y_out = (int)(diag - x_min);
}

// The merge kernel hides its gather latency with resident warps (measured on R-MAT: fewer registers and more warps beat deeper
// unrolling, gpurun_out/s4_tune_cfg3.jsonl), so it asks for more CTAs per SM than the row kernel's estimate.
#ifndef SPMM_MERGE_EXTRA_BLOCKS
#define SPMM_MERGE_EXTRA_BLOCKS 1
#endif
constexpr int merge_min_blocks(int nv, int w, int u, int threads)
{
    const int mb = min_blocks(nv, w, u, 1, threads) + SPMM_MERGE_EXTRA_BLOCKS;
    return mb > 8 ? 8 : mb;
}

template <int KL, int NV, int W, int U, bool FULL, int THREADS>
__global__ void __launch_bounds__(THREADS, merge_min_blocks(NV, W, U, THREADS)) spmm_merge_kernel(const SpmmArgs a)
{
    constexpr int RW = 32 / KL;
    using S = Slice<KL, NV, W>;
    // the non-zero items of the work list are those of rows [row_begin,row_end) inside [nnz_lo,nnz_hi)
    const int nnz_lo = max(a.nnz_lo, a.rowptr[a.row_begin]);
    const int nnz_hi = max(nnz_lo, min(a.nnz_hi, a.rowptr[a.row_end]));
    const RowClip rp{a.rowptr, nnz_lo, nnz_hi};

    const int lane = threadIdx.x & 31;
    const int kl = lane % KL;
    const long long team = ((long long)blockIdx.x * (THREADS / 32) + (threadIdx.x >> 5)) * RW + lane / KL;
    if (team >= a.n_teams)
        return;
    const int tile0 = blockIdx.y * S::TILE;
    const unsigned mask = slice_mask<KL, NV, W>(tile0, kl, a.kc);
    const double *__restrict__ Bk = a.B + tile0 + kl * W;
    const int n_rows = a.row_end - a.row_begin;
    const int n_nnz = nnz_hi - nnz_lo;
    const long long total = (long long)n_rows + n_nnz;
    const long long d0 = min(team * (long long)a.items_per_team, total);
    const long long d1 = min(d0 + a.items_per_team, total);

    int x, y;
    merge_path_search(rp, a.row_begin, n_rows, nnz_lo, n_nnz, d0, x, y);
    int row = a.row_begin + x;
    int j = nnz_lo + y;
    int items = (int)(d1 - d0);

    double *carry_head = a.carry + (2 * team) * (long long)a.ldcarry + tile0 + kl * W;
    double *carry_tail = carry_head + a.ldcarry;
    int head_row = -1, tail_row = -1;

    S acc;
    acc.zero();
    // fresh = no earlier team consumed a non-zero of `row`
    bool fresh = row < a.row_end ? (j == rp(row)) : true;
    // The team's items are walked in batches of up to U NON-ZEROS, whatever rows they belong to: their column ids,
    // values and B rows are loaded before the row structure is looked at, so U gathers are in flight per team even
    // where rows hold one or two entries (R-MAT: half the rows are empty, a fifth hold one or two). Row ends are
    // consumed in path order between the FMAs; `re` / `re2` = end offsets of the open row and of the row after it
    // (fetched one row ahead, so closing a row does not wait for memory).
    int re = row < a.row_end ? rp(row + 1) : 0x7FFFFFFF;
    int re2 = row + 1 < a.row_end ? rp(row + 2) : 0x7FFFFFFF;
    auto close_row = [&]() {
        if (fresh)
        {
            double *const cp = a.C + (long long)(row - a.c_row0) * a.ldc + tile0 + kl * W;
            acc.store(cp, mask);
            for (int d = 0; d < a.extra.n; ++d)
                acc.store(cp + a.extra.off[d], mask);
        }
        else
        {
            acc.store_plain(carry_head);
            head_row = row;
        }
        acc.zero();
        fresh = true;
        ++row;
        --items;
        re = re2;
        re2 = row + 1 < a.row_end ? rp(row + 2) : 0x7FFFFFFF;
    };
    // A batch = KL consecutive non-zeros: lane kl of the team loads column id and value of non-zero j + kl (one coalesced
    // request per team instead of one per non-zero), the next batch is requested before this one is worked on, and the
    // B rows are gathered UU at a time with the ids passed around by shuffles inside the team.
    constexpr int UU = U < KL ? U : KL;
    const unsigned team_mask = KL == 32 ? 0xFFFFFFFFu : (((1u << KL) - 1u) << (lane - kl));
    const int team_lane0 = lane - kl;
    auto fetch = [&](int base, int &c_out, double &v_out) {
        const int jj = max(min(base + kl, nnz_hi - 1), 0);
        c_out = nnz_hi > 0 ? ld_stream_i32(a.colidx + jj) : 0;
        v_out = nnz_hi > 0 ? ld_stream_f64(a.vals + jj) : 0.0;
    };
    int cc, cn;
    double vv, vn;
    fetch(j, cc, vv);
    while (items > 0 && row < a.row_end)
    {
        const int nb = min(min(KL, items), nnz_hi - j); // non-zeros of this batch (0: only row ends are left)
        if (nb <= 0)
        {
            close_row(); // j == nnz_hi: every remaining row ends here
            continue;
        }
        fetch(j + nb, cn, vn);
#pragma unroll
        for (int g = 0; g < KL; g += UU)
        {
            if (g < nb)
            {
                int c[UU];
                double xv[UU];
                S b[UU];
#pragma unroll
                for (int u = 0; u < UU; ++u)
                {
                    c[u] = __shfl_sync(team_mask, cc, team_lane0 + g + u);
                    xv[u] = __shfl_sync(team_mask, vv, team_lane0 + g + u);
                }
#pragma unroll
                for (int u = 0; u < UU; ++u)
                    b[u].template load<FULL>(Bk + (long long)c[u] * a.ldb, mask);
#pragma unroll
                for (int u = 0; u < UU; ++u)
                {
                    if (g + u < nb)
                    {
                        while (j >= re && items > 0) // the rows that end before this non-zero (row < row_end: the non-zero lies in one)
                            close_row();
                        if (items > 0)
                        {
                            acc.fma(xv[u], b[u]);
                            ++j;
                            --items;
                        }
                    }
                }
            }
        }
        cc = cn;
        vv = vn;
    }
    // ran out of items inside a row some of whose non-zeros are already consumed
    if (row < a.row_end && j > rp(row))
    {
        acc.store_plain(carry_tail);
        tail_row = row;
    }
    if (kl == 0 && blockIdx.y == 0)
    {
        a.carry_row[2 * team] = head_row;
        a.carry_row[2 * team + 1] = tail_row;
    }
}

// One team per carry slot. The first slot of a row's run sums the run in slot order
// and stores the row. Used slots of one row are at most one unused slot apart.
template <int KL, int NV, int W, int THREADS>
__global__ void __launch_bounds__(THREADS, 2) spmm_merge_fixup_kernel(const SpmmArgs a)
{
    constexpr int RW = 32 / KL;
    using S = Slice<KL, NV, W>;
    const int lane = threadIdx.x & 31;
    const int kl = lane % KL;
    const long long n_slots = 2LL * a.n_teams;
    const long long s = ((long long)blockIdx.x * (THREADS / 32) + (threadIdx.x >> 5)) * RW + lane / KL;
    if (s >= n_slots)
        return;
    const int row = a.carry_row[s];
    if (row < 0)
        return;
    if (s >= 1)
    {
        const int p1 = a.carry_row[s - 1];
        if (p1 == row)
            return;
        if (p1 < 0 && s >= 2 && a.carry_row[s - 2] == row)
            return;
    }
    const int tile0 = blockIdx.y * S::TILE;
    const unsigned mask = slice_mask<KL, NV, W>(tile0, kl, a.kc);
    const double *cp = a.carry + tile0 + kl * W;
    // The run is walked eight slots at a time: eight row ids are loaded together, then the eight slots (unconditional loads
    // from clamped, always valid slots) and those that belong to the run are added into four partial sums, folded in a fixed
    // order at the end — deterministic, and a hub row cut by a thousand teams no longer costs a thousand dependent memory
    // round trips (the fix-up of cfg3's first non-zero range took 752 us against 212 us for the multiply itself).
    S acc, part[4];
    acc.zero();
#pragma unroll
    for (int t = 0; t < 4; ++t)
        part[t].zero();
    acc.add_plain(cp + s * (long long)a.ldcarry);
    int gap = 0;
    bool open = true;
    for (long long q = s + 1; open && q < n_slots; q += 8)
    {
        long long qi[8];
        int r[8];
#pragma unroll
        for (int t = 0; t < 8; ++t)
            qi[t] = min(q + t, n_slots - 1);
#pragma unroll
        for (int t = 0; t < 8; ++t) // (volatile: issued back to back, in this order, before anything waits for one of them)
            asm volatile("ld.global.s32 %0, [%1];" : "=r"(r[t]) : "l"(a.carry_row + qi[t]));
        bool take[8];
#pragma unroll
        for (int t = 0; t < 8; ++t)
        {
            const bool inside = q + t < n_slots;
            const bool mine = open && inside && r[t] == row;
            const bool unused = open && inside && r[t] == -1;
            take[t] = mine;
            gap = mine ? 0 : (unused ? gap + 1 : gap);
            open = open && inside && (mine || (unused && gap < 2));
        }
#pragma unroll
        for (int h = 0; h < 2; ++h)
        {
            S x[4];
#pragma unroll
            for (int t = 0; t < 4; ++t)
                x[t].load_plain(cp + qi[4 * h + t] * (long long)a.ldcarry);
#pragma unroll
            for (int t = 0; t < 4; ++t)
                part[t].add_if(x[t], take[4 * h + t]);
        }
    }
#pragma unroll
    for (int t = 0; t < 4; ++t)
        acc.add(part[t]);
    double *const dst = a.C + (long long)(row - a.c_row0) * a.ldc + tile0 + kl * W;
    acc.store(dst, mask);
    for (int d = 0; d < a.extra.n; ++d)
        acc.store(dst + a.extra.off[d], mask);
}

} // namespace spmm
