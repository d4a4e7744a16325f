// spmm_tiled.cu — row tiles whose B rows live in a software-managed shared-memory window fed by TMA.
//
// Replaces, for whole-matrix multiplies with k >= 16, the gather of B rows through L1
// (one LDG per non-zero and 128-byte line) of
//   /root/reference "Source Code/SparseMatrixFatVectorMultiply.cpp":17-28
// Why (profiles/r1_ncu_rows_k64.md): the CSR row kernels sit on a 105-118 us plateau on the
// cop20k_A-shaped k=64 case although HBM traffic is compulsory — 1.34 GB of B rows pass the
// LSU/L1 path, 36-60 % of them L1 misses (0.9 GB of L2 -> SM traffic) that hold registers while in flight.
//
// Layout ("tiles", built once on the device next to the untouched CSR):
//   * a tile = T consecutive rows; a chunk = a run of consecutive tiles that one CTA walks in order.
//   * B is cut into aligned "boxes" of BR consecutive rows (box id = column / BR). The CTA keeps a
//     window of NS box slots in shared memory. The builder replays the chunk: a box a tile needs and
//     the window already holds is a hit; a missing box with at least `thr` non-zeros in the tile is
//     loaded into the least recently used slot that no tile in flight reads; non-zeros of sparser
//     boxes (hub couplings, stragglers) get one "single" B row each in a small ring pool. For FEM-like
//     rows the window slides with the tiles: a B row is fetched from L2 about once per band and chunk
//     instead of once per non-zero.
//   * every non-zero becomes a value (8 bytes) and a 16-bit slab row id (rows padded to 4 ids); slab row =
//     slot*BR + column%BR, or a pool row. The rows of a tile are grouped into "units" of 8 rows of similar length (one row per
//     team of 4 lanes); a row of 48+ non-zeros becomes a unit of its own, cut in 8 segments. Header,
//     unit table and records of a tile form one contiguous 16-byte aligned blob; per tile there is a
//     load list (box, slot) and a singles list (column).
// Kernel (one persistent CTA per SM, warp-specialised, no CTA-wide barrier in the main loop):
//   * 4 producer warps (each owns every 4th work item = tile x k-tile) run up to `depth` items ahead of the consumers: one
//     cp.async.bulk for the blob, one cp.async.bulk.tensor.2d per missing box (KT columns x BR rows of
//     B, zero filled outside the matrix), one gather4 TMA per four single rows; everything
//     completes on the item's mbarrier. B rows reach shared memory without registers or L1 tags.
//   * consumer warps take the units of an item round-robin. A team walks its row with one broadcast
//     LDS.128 per record and conflict-free LDS.128 reads of the slab row, FP64 FMAs in ascending
//     record order (the reference's order), and stores the row piece from registers. Split rows are
//     folded across the 8 teams with warp shuffles. Warps only meet at the mbarriers, so a warp that
//     finishes its share of an item moves on to the next one.
// Shared-memory port arithmetic (DESIGN.md §4.5): KT=16 -> 9 wavefronts per 8 records and k-tile.
#include <cuda.h>

#include <cub/block/block_radix_sort.cuh>
#include <cub/block/block_scan.cuh>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "spmm_launch.cuh"

namespace spmm
{

namespace
{
constexpr int TB_THREADS = 512;
constexpr int TB_ITEMS = 12;
constexpr int TB_CAP = TB_THREADS * TB_ITEMS; // records per tile the builder can sort
constexpr int TB_UMAX = 1024;                 // distinct boxes per tile the builder tracks
constexpr int TB_NSMAX = 192;                 // window slots
constexpr int TB_MAXT = 248;                  // rows per tile (row field of a unit entry: 0xFF = padding)
constexpr int TB_SPLIT = 48;                  // rows this long become a unit of their own
constexpr int TB_SPLITCAP = 8;                // split units per tile (further long rows stay whole)
constexpr int TB_DMAX = 8;                    // work items in flight
constexpr int UW = 8;                         // rows per unit = teams per warp
constexpr int TL = 4;                         // lanes per team
constexpr int SMEM_CAP = 232448;              // 227 KB opt-in limit per CTA on sm_100

// unit entry: begin (13 bits) | len (10 bits) << 13 | row (8 bits) << 23 | split << 31
constexpr unsigned UE_PAD_ROW = 0xFFu;

struct TileDesc // 16 bytes
{
    unsigned off16;  // blob offset in 16-byte units
    unsigned bytes;  // blob bytes (multiple of 16)
    unsigned counts; // n_loads | n_singles (13 bits) << 16 | fence << 29: tiles back to the last tile that drains the pipeline (7 = none near)
    int pool_start;  // first pool row of this tile's singles (ring)
};

struct BuildParams
{
    int n_rows, T, lgBR, NS, POOL, thr, tiles_per_chunk, n_tiles, hdr_bytes, depth;
};

// status words written by the builder
enum
{
    ST_FAIL = 0,
    ST_MAXREC = 1,
    ST_MAXPOOL = 2, // most singles in `depth` consecutive tiles
    ST_MAXLOAD = 3,
    ST_DRAINS = 4, // tiles that only fit once everything before them has finished
    ST_MAXBLOB = 5, // largest blob in bytes
    ST_WORDS = 6
};
// 64-bit totals behind the status words
enum
{
    TOT_LOADS = 0,
    TOT_SINGLES = 1,
    TOT_WORDS = 2
};

__host__ __device__ inline int units_cap(int T) { return (T + UW - 1) / UW + TB_SPLITCAP; }
// Byte offset of tile t's blob (first non-zero e0): a closed form that leaves room for the header, the padded
// value stream (8 e) and the padded id stream (2 (e + 3T) at most) of every earlier tile.
__host__ __device__ inline unsigned long long blob_offset(int t, long long e0, int hdr_bytes, int T)
{
    // (+ 112 T: the rows of a unit start on distinct banks, at most 7 values and 7 id groups of padding per row)
    return (unsigned long long)t * (unsigned long long)(hdr_bytes + 120 * T + 48) + ((10ull * (unsigned long long)e0 + 15ull) & ~15ull);
}

// Builder: one CTA per chunk, tiles replayed in order. DRY: only count.
template <bool DRY>
__global__ void __launch_bounds__(TB_THREADS) tile_build_kernel(const int *__restrict__ rowptr,
                                                                 const int *__restrict__ colidx,
                                                                 const double *__restrict__ vals, const BuildParams p,
                                                                 unsigned char *__restrict__ blob,
                                                                 TileDesc *__restrict__ tdesc, int2 *__restrict__ loads,
                                                                 int *__restrict__ singles, int *__restrict__ status,
                                                                 unsigned long long *__restrict__ totals,
                                                                 const int *__restrict__ order)
{
    using Sort = cub::BlockRadixSort<int, TB_THREADS, TB_ITEMS>;
    using Scan = cub::BlockScan<int, TB_THREADS>;
    __shared__ union
    {
        typename Sort::TempStorage sort;
        int sorted[TB_CAP];
    } sm;
    __shared__ typename Scan::TempStorage scan_tmp;
    __shared__ int s_ubox[TB_UMAX], s_ucnt[TB_UMAX], s_uslot[TB_UMAX];
    __shared__ int s_slot_box[TB_NSMAX], s_slot_stamp[TB_NSMAX];
    __shared__ int s_rp[TB_MAXT + 1];
    __shared__ unsigned s_units[(TB_MAXT / UW + 1 + TB_SPLITCAP) * UW]; // word 0 of the unit entries
    __shared__ int s_uidx[(TB_MAXT / UW + 1 + TB_SPLITCAP) * UW];      // word 1: first slot of the row (segment) in the id stream
    __shared__ int s_ioff[TB_MAXT + 1];                                 // id-stream offset of each row (rows padded to 4 ids)
    __shared__ int s_voff[TB_MAXT + 1];                                 // value-stream offset of each row
    __shared__ int s_nload, s_nsplit, s_pool_ptr, s_drain, s_nval, s_nid;
    __shared__ int s_usz_v[TB_MAXT / UW + 1 + TB_SPLITCAP], s_usz_i[TB_MAXT / UW + 1 + TB_SPLITCAP]; // unit sizes, then unit starts
    __shared__ int s_recent[TB_DMAX]; // singles of the last `depth` tiles

    const int BR = 1 << p.lgBR;
    const int t_begin = blockIdx.x * p.tiles_per_chunk;
    const int t_end = min(p.n_tiles, t_begin + p.tiles_per_chunk);
    for (int s = threadIdx.x; s < TB_NSMAX; s += TB_THREADS)
    {
        s_slot_box[s] = -1;
        s_slot_stamp[s] = -1000;
    }
    if (threadIdx.x < TB_DMAX)
        s_recent[threadIdx.x] = 0;
    if (threadIdx.x == 0)
        s_pool_ptr = 0;
    unsigned long long my_loads = 0, my_singles = 0; // thread 0 only
    int last_fence = 0; // last tile (of the chunk) that waits for everything before it; tile 0 does by construction

    // `pos` is a tile's place in the walking order (what the kernel iterates and what tdesc / loads / singles are indexed
    // by); `t` is the tile itself (its rows, its blob). order == nullptr: tiles are walked as they lie.
    for (int pos = t_begin; pos < t_end; ++pos)
    {
        const int t = order ? order[pos] : pos;
        const int lt = pos - t_begin;
        const int r0 = t * p.T, r1 = min(p.n_rows, r0 + p.T);
        const int nr = r1 - r0;
        const int e0 = rowptr[r0], e1 = rowptr[r1];
        const int n = e1 - e0;
        if (n > TB_CAP)
        {
            if (threadIdx.x == 0)
                atomicOr(status + ST_FAIL, 1);
            return;
        }
        __syncthreads(); // previous tile done with sm.sorted / s_rp / s_u*
        for (int i = threadIdx.x; i <= p.T; i += TB_THREADS)
            s_rp[i] = rowptr[min(r0 + i, r1)] - e0;
        if (threadIdx.x == 0)
            s_nsplit = 0;

        // ---- distinct boxes of the tile, ascending, with their non-zero counts
        int keys[TB_ITEMS];
#pragma unroll
        for (int i = 0; i < TB_ITEMS; ++i)
        {
            const int j = threadIdx.x * TB_ITEMS + i;
            keys[i] = j < n ? (colidx[e0 + j] >> p.lgBR) : 0x7FFFFFFF;
        }
        Sort(sm.sort).Sort(keys);
        __syncthreads();
#pragma unroll
        for (int i = 0; i < TB_ITEMS; ++i)
            sm.sorted[threadIdx.x * TB_ITEMS + i] = keys[i];
        __syncthreads();
        int heads = 0;
#pragma unroll
        for (int i = 0; i < TB_ITEMS; ++i)
        {
            const int j = threadIdx.x * TB_ITEMS + i;
            heads += (j < n && (j == 0 || sm.sorted[j] != sm.sorted[j - 1])) ? 1 : 0;
        }
        int upos, nu;
        Scan(scan_tmp).ExclusiveSum(heads, upos, nu);
        if (nu > TB_UMAX)
        {
            if (threadIdx.x == 0)
                atomicOr(status + ST_FAIL, 2);
            return;
        }
#pragma unroll
        for (int i = 0; i < TB_ITEMS; ++i)
        {
            const int j = threadIdx.x * TB_ITEMS + i;
            if (j < n && (j == 0 || sm.sorted[j] != sm.sorted[j - 1]))
            {
                const int b = sm.sorted[j];
                int lo = j, hi = n; // first position with a larger box id
                while (lo < hi)
                {
                    const int mid = (lo + hi) >> 1;
                    if (sm.sorted[mid] <= b)
                        lo = mid + 1;
                    else
                        hi = mid;
                }
                s_ubox[upos] = b;
                s_ucnt[upos] = lo - j;
                ++upos;
            }
        }
        __syncthreads();

        // ---- window lookup: hit -> slot, miss -> -2 (dense enough to load) or -1 (singles)
        for (int u = threadIdx.x; u < nu; u += TB_THREADS)
        {
            const int b = s_ubox[u];
            int slot = -1;
            for (int s = 0; s < p.NS; ++s)
                if (s_slot_box[s] == b)
                    slot = s;
            if (slot >= 0)
                s_slot_stamp[slot] = lt;
            s_uslot[u] = slot >= 0 ? slot : (s_ucnt[u] >= p.thr ? -2 : -1);
        }
        __syncthreads();
        // ---- misses, ascending box id: least recently used slot that no tile in flight reads
        if (threadIdx.x == 0)
        {
            // enough slots that no tile in flight reads? otherwise this tile waits for everything before it (drain)
            int wanted = 0, eligible = 0;
            for (int u = 0; u < nu; ++u)
                wanted += s_uslot[u] == -2 ? 1 : 0;
            for (int s = 0; s < p.NS; ++s)
                eligible += s_slot_stamp[s] <= lt - p.depth ? 1 : 0;
            const bool drain = wanted > eligible;
            s_drain = drain ? 1 : 0;
            const int limit = drain ? lt - 1 : lt - p.depth; // a slot may be overwritten if its stamp <= limit
            int nl = 0;
            for (int u = 0; u < nu; ++u)
            {
                if (s_uslot[u] != -2)
                    continue;
                int best = -1, best_stamp = limit + 1;
                for (int s = 0; s < p.NS; ++s)
                    if (s_slot_stamp[s] < best_stamp)
                    {
                        best = s;
                        best_stamp = s_slot_stamp[s];
                    }
                if (best < 0)
                {
                    s_uslot[u] = -1; // window full of live boxes: this box goes row by row
                    continue;
                }
                s_slot_box[best] = s_ubox[u];
                s_slot_stamp[best] = lt;
                s_uslot[u] = best;
                if (!DRY)
                    loads[(size_t)pos * p.NS + nl] = make_int2(s_ubox[u] << p.lgBR, best);
                ++nl;
            }
            s_nload = nl;
            my_loads += (unsigned long long)nl;
        }

        // ---- units: rows of 48+ non-zeros are split (at most TB_SPLITCAP per tile), the rest ranked by length
        for (int r = threadIdx.x; r < nr; r += TB_THREADS)
            if (s_rp[r + 1] - s_rp[r] >= TB_SPLIT)
                atomicAdd(&s_nsplit, 1);
        __syncthreads();
        // (stream offsets of the rows are laid out unit by unit further down: s_voff / s_ioff)
        const int n_split = min(s_nsplit, TB_SPLITCAP);
        const int n_normal_units = (nr - n_split + UW - 1) / UW;
        const int n_units = n_normal_units + n_split;
        for (int i = threadIdx.x; i < n_units * UW; i += TB_THREADS)
        {
            s_units[i] = UE_PAD_ROW << 23; // padding entry: no row, no records
            s_uidx[i] = 0;
        }
        __syncthreads();
        for (int r = threadIdx.x; r < nr; r += TB_THREADS)
        {
            const int len = s_rp[r + 1] - s_rp[r];
            // split rank: position among the long rows (by row id); the first TB_SPLITCAP are split
            int srank = -1;
            if (len >= TB_SPLIT)
            {
                srank = 0;
                for (int q = 0; q < r; ++q)
                    srank += (s_rp[q + 1] - s_rp[q] >= TB_SPLIT) ? 1 : 0;
            }
            if (srank >= 0 && srank < TB_SPLITCAP)
            {
                const int seg = (((len + UW - 1) / UW) + 3) & ~3; // segments start at multiples of 4 ids
                for (int j = 0; j < UW; ++j)
                {
                    const int b = min(j * seg, len), e = min(b + seg, len);
                    s_units[(n_normal_units + srank) * UW + j] =
                        (unsigned)b | ((unsigned)(e - b) << 13) | ((unsigned)r << 23) | 0x80000000u; // begin: relative, placed below
                    s_uidx[(n_normal_units + srank) * UW + j] = b;
                }
            }
            else
            {
                // rank among the whole rows: longer first, ties by row id
                int rank = 0, skipped = 0;
                for (int q = 0; q < nr; ++q)
                {
                    const int lq = s_rp[q + 1] - s_rp[q];
                    if (lq >= TB_SPLIT && skipped < TB_SPLITCAP)
                    {
                        ++skipped; // the first TB_SPLITCAP long rows are split, not ranked
                        continue;
                    }
                    rank += (lq > len || (lq == len && q < r)) ? 1 : 0;
                }
                if (len > 0x3FF)
                    atomicOr(status + ST_FAIL, 8); // more than TB_SPLITCAP very long rows in one tile
                s_units[rank] = ((unsigned)(len & 0x3FF) << 13) | ((unsigned)r << 23); // begin: placed below
                s_uidx[rank] = 0;
            }
        }
        __syncthreads();
        // ---- stream layout, unit by unit: the eight rows of a unit are walked in lockstep by the eight teams of a warp, one
        // 8-byte value load (and one 8-byte load of four ids) per team and step. Eight unrelated addresses collide on the
        // shared-memory banks (13 % of this kernel's load wavefronts, profiles/r1_tiled.md); rows whose streams start on
        // eight different 8-byte bank pairs never do (tools/microbench/lds_patterns.cu), so each row is pushed to the next
        // offset whose residue mod 16 no earlier row of its unit holds: at most 7 slots of padding per row and stream.
        // (The pushes of a unit depend on the lengths of its rows only, not on where the unit starts — a different start
        // rotates all residues alike — so every unit is laid out by its own thread from offset 0 and the unit sizes are
        // scanned afterwards.)
        if (threadIdx.x < n_units)
        {
            const int u = threadIdx.x;
            int pos = 0, ipos = 0; // doubles / groups of four ids, relative to the start of the unit
            if (u >= n_normal_units)
            {
                // split row: its eight segments lie one after the other
                const int r = (int)((s_units[u * UW] >> 23) & 0xFF), len = s_rp[r + 1] - s_rp[r];
                pos = len;
                ipos = (len + 3) >> 2;
                s_voff[r] = 0;
                s_ioff[r] = 0;
            }
            else
            {
                unsigned used_v = 0, used_i = 0;
                for (int j = 0; j < UW; ++j)
                {
                    const unsigned w = s_units[u * UW + j];
                    const int r = (int)((w >> 23) & 0xFF);
                    if (r == (int)UE_PAD_ROW)
                        continue;
                    const int len = s_rp[r + 1] - s_rp[r];
                    if (len > 0)
                    {
                        while ((used_v >> (pos & 15)) & 1u)
                            ++pos;
                        used_v |= 1u << (pos & 15);
                        while ((used_i >> (ipos & 15)) & 1u)
                            ++ipos;
                        used_i |= 1u << (ipos & 15);
                    }
                    s_units[u * UW + j] = (w & ~0x1FFFu) | (unsigned)pos;
                    s_uidx[u * UW + j] = ipos * 4;
                    s_voff[r] = pos;
                    s_ioff[r] = ipos * 4;
                    pos += len;
                    ipos += (len + 3) >> 2;
                }
            }
            s_usz_v[u] = pos;
            s_usz_i[u] = ipos;
        }
        __syncthreads();
        if (threadIdx.x == 0)
        {
            int pos = 0, ipos = 0;
            for (int u = 0; u < n_units; ++u)
            {
                const int sv = s_usz_v[u], si = s_usz_i[u];
                s_usz_v[u] = pos;
                s_usz_i[u] = ipos;
                pos += sv;
                ipos += si;
            }
            s_nval = pos;
            s_nid = ipos * 4;
            if (pos > 0x1FFF)
                atomicOr(status + ST_FAIL, 16); // the begin field of a unit entry holds 13 bits
        }
        __syncthreads();
        if (threadIdx.x < n_units)
        {
            const int u = threadIdx.x, bv = s_usz_v[u], bi = s_usz_i[u] * 4;
            for (int j = 0; j < UW; ++j)
            {
                const unsigned w = s_units[u * UW + j];
                const int r = (int)((w >> 23) & 0xFF);
                if (r == (int)UE_PAD_ROW)
                    continue;
                s_units[u * UW + j] = (w & ~0x1FFFu) | (unsigned)((int)(w & 0x1FFF) + bv);
                s_uidx[u * UW + j] += bi;
                if (u < n_normal_units || j == 0)
                {
                    s_voff[r] += bv;
                    s_ioff[r] += bi;
                }
            }
        }
        __syncthreads();

        // ---- records (blocked: thread i owns records 12i .. 12i+11)
        int srow[TB_ITEMS], col[TB_ITEMS], nsingle = 0;
#pragma unroll
        for (int i = 0; i < TB_ITEMS; ++i)
        {
            const int j = threadIdx.x * TB_ITEMS + i;
            srow[i] = 0;
            col[i] = 0;
            if (j < n)
            {
                col[i] = colidx[e0 + j];
                const int b = col[i] >> p.lgBR;
                int lo = 0, hi = nu - 1;
                while (lo < hi)
                {
                    const int mid = (lo + hi) >> 1;
                    if (s_ubox[mid] < b)
                        lo = mid + 1;
                    else
                        hi = mid;
                }
                const int slot = s_uslot[lo];
                srow[i] = slot >= 0 ? slot * BR + (col[i] & (BR - 1)) : -1;
                nsingle += slot < 0 ? 1 : 0;
            }
        }
        int spos, ns_real;
        Scan(scan_tmp).ExclusiveSum(nsingle, spos, ns_real);
        __syncthreads();
        const int ns_total = (ns_real + 3) & ~3; // single rows travel four at a time (TMA gather4): pad the list
        // pool ring: the singles of the tiles in flight must all fit (a drained tile has the pool to itself)
        int recent = ns_total;
        for (int i = 1; i < p.depth; ++i)
            recent += s_recent[(lt + i) % p.depth]; // entries of tiles lt-depth+1 .. lt-1
        const bool drain = s_drain != 0 || recent > p.POOL;
        if (drain)
        {
            recent = ns_total;
            last_fence = lt;
        }
        // tiles right behind a fence may only assume the tiles before the fence are done if they wait for them too
        const int fence = min(lt - last_fence, 7); // 7 = far enough: the depth rule alone is enough (depth <= 8)
        if (recent > p.POOL || ns_total > 0x1FFF)
        {
            if (threadIdx.x == 0)
                atomicOr(status + ST_FAIL, 4);
            return;
        }
        const int pool_start = s_pool_ptr;
        __syncthreads();
        if (threadIdx.x == 0)
        {
            if (drain)
            {
                for (int i = 0; i < TB_DMAX; ++i)
                    s_recent[i] = 0;
                atomicAdd(status + ST_DRAINS, 1);
            }
            s_recent[lt % p.depth] = ns_total;
            s_pool_ptr = (pool_start + ns_total) % p.POOL;
            my_singles += (unsigned long long)ns_real;
            atomicMax(status + ST_MAXREC, n);
            atomicMax(status + ST_MAXBLOB,
                      p.hdr_bytes + (int)(((unsigned)s_nval * 8u + 15u) & ~15u) + (int)(((unsigned)s_nid * 2u + 15u) & ~15u));
            atomicMax(status + ST_MAXPOOL, recent);
            atomicMax(status + ST_MAXLOAD, s_nload);
        }
        if (DRY)
            continue;

        // blob = header | unit table | values (8 bytes per non-zero) | slab-row ids (2 bytes, rows padded to 4 ids)
        const int n_ids = s_nid;
        const unsigned val_bytes = ((unsigned)s_nval * 8u + 15u) & ~15u, id_bytes = ((unsigned)n_ids * 2u + 15u) & ~15u;
        const unsigned off16 = (unsigned)(blob_offset(t, e0, p.hdr_bytes, p.T) >> 4);
        unsigned char *mine = blob + ((unsigned long long)off16 << 4);
        if (threadIdx.x == 0)
        {
            TileDesc d;
            d.off16 = off16;
            d.bytes = (unsigned)p.hdr_bytes + val_bytes + id_bytes;
            d.counts = (unsigned)s_nload | ((unsigned)ns_total << 16) | ((unsigned)fence << 29);
            d.pool_start = pool_start;
            tdesc[pos] = d;
            *reinterpret_cast<int4 *>(mine) = make_int4(n, n_units, t, (int)((unsigned)p.hdr_bytes + val_bytes)); // .z: the tile (its C rows)
        }
        uint2 *units_out = reinterpret_cast<uint2 *>(mine + 16);
        for (int i = threadIdx.x; i < (p.hdr_bytes - 16) / 8; i += TB_THREADS)
            units_out[i] = i < n_units * UW ? make_uint2(s_units[i], (unsigned)s_uidx[i]) : make_uint2(UE_PAD_ROW << 23, 0u);
        double *val_out = reinterpret_cast<double *>(mine + p.hdr_bytes);
        unsigned short *id_out = reinterpret_cast<unsigned short *>(mine + p.hdr_bytes + val_bytes);
        for (int i = threadIdx.x; i < (int)(id_bytes / 2); i += TB_THREADS)
            id_out[i] = 0; // padding ids are never used for arithmetic; keep them inside the slab
        if (threadIdx.x < ns_total - ns_real)
            singles[(size_t)pos * p.POOL + ns_real + threadIdx.x] = 0; // padding rows: any valid B row
        __syncthreads(); // id padding written before the real ids
#pragma unroll
        for (int i = 0; i < TB_ITEMS; ++i)
        {
            const int j = threadIdx.x * TB_ITEMS + i;
            if (j >= n)
                continue;
            int sr = srow[i];
            if (sr < 0)
            {
                singles[(size_t)pos * p.POOL + spos] = col[i];
                sr = p.NS * BR + (pool_start + spos) % p.POOL;
                ++spos;
            }
            // row holding record j: last local row with s_rp[r] <= j (skips empty rows)
            int lo = 0, hi = nr;
            while (hi - lo > 1)
            {
                const int mid = (lo + hi) >> 1;
                if (s_rp[mid] <= j)
                    lo = mid;
                else
                    hi = mid;
            }
            val_out[s_voff[lo] + (j - s_rp[lo])] = vals[e0 + j];
            id_out[s_ioff[lo] + (j - s_rp[lo])] = (unsigned short)sr;
        }
    }
    if (threadIdx.x == 0)
    {
        atomicAdd(totals + TOT_LOADS, my_loads);
        atomicAdd(totals + TOT_SINGLES, my_singles);
    }
}

// Value refresh (spmm_csr_update_values_*): new values into the value streams of the blobs, nothing else of the layout
// changes. One CTA per tile: its unit table says where each row's run starts in the value stream (a split row: its eight
// segments lie one after the other from the first one's begin), so the table becomes a row -> offset map in shared memory
// and the tile's non-zeros are then copied in CSR order, coalesced on the source side. Padding slots are left as they are.
// csr_out != nullptr: the same values also go to the CSR value array (one read of the source, two writes).
constexpr int TR_THREADS = 256;
constexpr int TR_U = 4; // loads in flight per thread
__global__ void __launch_bounds__(TR_THREADS) tile_refresh_kernel(const int *__restrict__ rowptr, const double *__restrict__ src,
                                                                   double *__restrict__ csr_out, unsigned char *__restrict__ blob,
                                                                   int n_rows, int T, int hdr_bytes)
{
    __shared__ int s_rp[TB_MAXT + 1];
    __shared__ int s_voff[TB_MAXT];
    const int t = blockIdx.x;
    const int r0 = t * T, r1 = min(n_rows, r0 + T), nr = r1 - r0;
    const int e0 = rowptr[r0];
    for (int i = threadIdx.x; i <= nr; i += TR_THREADS)
        s_rp[i] = rowptr[r0 + i] - e0;
    unsigned char *mine = blob + blob_offset(t, e0, hdr_bytes, T);
    const int n_units = reinterpret_cast<const int4 *>(mine)->y;
    const uint2 *units = reinterpret_cast<const uint2 *>(mine + 16);
    for (int i = threadIdx.x; i < n_units * UW; i += TR_THREADS)
    {
        const unsigned w = units[i].x;
        const int r = (int)((w >> 23) & 0xFF);
        if (r != (int)UE_PAD_ROW && ((w >> 31) == 0 || i % UW == 0))
            s_voff[r] = (int)(w & 0x1FFF);
    }
    __syncthreads();
    const int n = s_rp[nr];
    double *val_out = reinterpret_cast<double *>(mine + hdr_bytes);
    for (int base = 0; base < n; base += TR_THREADS * TR_U)
    {
        double v[TR_U];
#pragma unroll
        for (int u = 0; u < TR_U; ++u)
        {
            const int j = base + u * TR_THREADS + threadIdx.x;
            v[u] = j < n ? src[e0 + j] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < TR_U; ++u)
        {
            const int j = base + u * TR_THREADS + threadIdx.x;
            if (j >= n)
                continue;
            if (csr_out)
                csr_out[e0 + j] = v[u];
            // row holding non-zero j: last local row with s_rp[r] <= j (skips empty rows), as in the builder
            int lo = 0, hi = nr;
            while (hi - lo > 1)
            {
                const int mid = (lo + hi) >> 1;
                if (s_rp[mid] <= j)
                    lo = mid;
                else
                    hi = mid;
            }
            val_out[s_voff[lo] + (j - s_rp[lo])] = v[u];
        }
    }
}

// ---- PTX helpers: mbarrier, bulk copies -------------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity)
{
    asm volatile("{\n\t.reg .pred p;\n\tWAIT_%=:\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
                 "@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}" ::"r"(bar),
                 "r"(parity)
                 : "memory");
}
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void *src, unsigned bytes, unsigned bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void tma_box(unsigned dst, const CUtensorMap *map, int c0, int c1, unsigned bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
                 "l"(map), "r"(c0), "r"(c1), "r"(bar)
                 : "memory");
}
// four rows of B (any row ids) x the box width into four consecutive smem rows
__device__ __forceinline__ void tma_gather4(unsigned dst, const CUtensorMap *map, int c0, int4 rows, unsigned bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cta.global.tile::gather4.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];" ::"r"(dst),
                 "l"(map), "r"(c0), "r"(rows.x), "r"(rows.y), "r"(rows.z), "r"(rows.w), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ int4 lds128i(unsigned addr)
{
    int4 v;
    asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ double2 lds128d(unsigned addr)
{
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint2 lds64u(unsigned addr)
{
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ double lds64d(unsigned addr)
{
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}

#if defined(SPMM_ABLATE) && (SPMM_ABLATE & 512) // diagnostic build: consumers only wait and release (producer/TMA-side time)
#define T_NO_COMPUTE 1
#else
#define T_NO_COMPUTE 0
#endif
#if defined(SPMM_ABLATE) && (SPMM_ABLATE & 1024) // diagnostic build: no B rows are staged, only the blobs (consumer-side time)
#define T_NO_STAGE 1
#else
#define T_NO_STAGE 0
#endif
#if defined(SPMM_ABLATE) && (SPMM_ABLATE & 256) // diagnostic build: cycle counters per CTA
#define TPROF 1
#define TCLK() clock64()
#else
#define TPROF 0
#define TCLK() 0ll
#endif

struct TiledArgs
{
    long long *prof; // TPROF builds: 12 counters per CTA
    ExtraDst extra;  // peer copies of C (element offsets from C)
    const unsigned char *blob;
    const TileDesc *tdesc;
    const int2 *loads;
    const int *singles;
    const double *B;
    double *C;
    long long ldb, ldc;
    int n_tiles, n_chunks /* shares: chunks x ksplit */, ksplit, tiles_per_chunk, T, BR, NS, POOL, kc, nkt, depth;
    unsigned hdr_bytes;   // header + unit table bytes of a blob
    unsigned blob_stride; // bytes reserved per blob buffer in smem
    unsigned slab_off;    // offset of the slab (window slots, then the singles pool) from the aligned smem base
};

// smem map: [0,64) full barriers | [64,128) empty barriers | pad to 1024 | blob[depth] | slab (1024-aligned)
constexpr unsigned BLOB_OFF = 1024;

template <int KT, int NCW, int U, int NPW>
__global__ void __launch_bounds__((NCW + NPW) * 32, 1) spmm_tiled_kernel(const TiledArgs a,
                                                                         const __grid_constant__ CUtensorMap box_map,
                                                                         const __grid_constant__ CUtensorMap row_map)
{
    constexpr int NL = KT / (2 * TL); // LDS.128 per lane and record
    static_assert(NL >= 1 && NL * 2 * TL == KT, "a team of TL lanes covers the k-tile with NL 16-byte accesses per lane");
    // (NL = 1, the 8-column k-tile for k <= 8: the two teams of a quarter-warp read 64-byte slab rows that share their banks
    // when the rows have the same parity — 1.5 wavefronts per quarter-warp on average instead of the 2 a half-empty 16-column
    // k-tile costs, and half the bytes staged)
    extern __shared__ __align__(1024) unsigned char smem[];
    const unsigned s0 = (smem_u32(smem) + 1023u) & ~1023u;
    const unsigned full = s0, empty = s0 + 64; // 8 bytes each, indexed by work item mod depth
    const unsigned s_blob = s0 + BLOB_OFF;
    const unsigned s_slab = s0 + a.slab_off;
    const int D = a.depth;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // Programmatic dependent launch: the next multiply of the stream may place its CTAs as ours retire and run its prologue
    // (barriers, tile descriptors, the first value/id blob — all derived from A) under our tail; everything that touches
    // B or C waits for the grids before it (griddepcontrol.wait below). Launched without the attribute both are no-ops.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (threadIdx.x == 0)
    {
        for (int i = 0; i < D; ++i)
        {
            mbar_init(full + 8 * i, 1); // the expect_tx arrive of the item's producer warp
            mbar_init(empty + 8 * i, NCW);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    // work items in loop order: for share (blockIdx.x, += gridDim.x) / for k-tile of the share / for tile of the chunk.
    // A share = a chunk x one of `ksplit` groups of consecutive k-tiles: with many k-tiles the chunks are made ksplit
    // times longer and ksplit CTAs walk each of them, so the window is warmed up once per CTA instead of once per k-tile.
    struct Work
    {
        int c, kt, kt_end, t, t_begin, t_end;
    };
    auto work_chunk = [&](Work &x) {
        const int chunk = x.c / a.ksplit, part = x.c % a.ksplit;
        x.t_begin = chunk * a.tiles_per_chunk;
        x.t_end = min(a.n_tiles, x.t_begin + a.tiles_per_chunk);
        x.t = x.t_begin;
        const int per = (a.nkt + a.ksplit - 1) / a.ksplit;
        x.kt = min(a.nkt, part * per);
        x.kt_end = min(a.nkt, x.kt + per);
        if (x.kt >= x.kt_end) // fewer k-tiles than sharers: this share is empty
            x.t = x.t_end = x.t_begin;
    };
    auto work_next = [&](Work &x) {
        if (++x.t < x.t_end)
            return;
        x.t = x.t_begin;
        if (++x.kt < x.kt_end)
            return;
        for (x.c += gridDim.x; x.c < a.n_chunks; x.c += gridDim.x)
        {
            work_chunk(x);
            if (x.t < x.t_end)
                return;
        }
    };
    Work cur;
    for (cur.c = blockIdx.x; cur.c < a.n_chunks; cur.c += gridDim.x)
    {
        work_chunk(cur);
        if (cur.t < cur.t_end)
            break;
    }
    if (cur.c >= a.n_chunks)
        return;

    if (warp >= NCW)
    {
        // ---------------- producers: every item's copies are dealt round-robin over the NPW warps ----------------
        const int pw = warp - NCW;
        const unsigned box_bytes = (unsigned)(a.BR * KT * 8);
        struct Meta
        {
            TileDesc d;
            int2 ld; // box entry pw + NPW*lane of the item
            int4 sg; // single-row group pw + NPW*lane of the item (4 rows)
        };
        auto fetch = [&](const Work &x) {
            Meta m;
            m.d = a.tdesc[x.t];
            m.ld = a.loads[(size_t)x.t * a.NS + min(pw + NPW * lane, a.NS - 1)];
            m.sg = reinterpret_cast<const int4 *>(a.singles + (size_t)x.t * a.POOL)[min(pw + NPW * lane, a.POOL / 4 - 1)];
            return m;
        };
        long long p_wait = 0, p_issue = 0, p_sgl = 0, p_items = 0, p_t0 = TCLK();
        // one item: its copies are issued from `m`; `fill` receives the metadata of the item two turns ahead
        // (three Meta registers rotate through the roles, so no load result is touched before it is needed)
        Work ahead = cur; // the item whose metadata is fetched next
        int w = 0;
        // items <= known are finished. A parity wait on an mbarrier is only meaningful one phase ahead of what
        // this warp has seen, so waiting for item y walks the phases of y's ring entry that lie behind `known`.
        int known = -1;
        auto ensure = [&](int y) {
            if (y <= known)
                return;
            for (int z = y - ((y - known - 1) / D) * D; z <= y; z += D)
                mbar_wait(empty + 8 * (z % D), (z / D) & 1);
            known = y;
        };
        auto step = [&](const Meta &m, Meta &fill) {
            const long long c0 = TCLK();
            if (ahead.c < a.n_chunks)
            {
                fill = fetch(ahead);
                work_next(ahead);
            }
            const int st = w % D;
            // Item w overwrites its ring entry, pool rows and window slots. The builder guarantees that whatever it
            // overwrites was last read by item w-D at the latest — or, for a tile `fence` tiles behind one that needs more
            // than that rule leaves (and behind the start of a pass: unknown window), by the items before that fence.
            // Consumers finish items in order, so one wait on the newest such item is enough.
            const int fence = (int)(m.d.counts >> 29);
            ensure(max(w - D, fence < 7 ? w - fence - 1 : -1));
            const long long c1 = TCLK();
            const unsigned bar = full + 8 * st;
            const int n_loads = (int)(m.d.counts & 0xFFFFu), n_singles = (int)((m.d.counts >> 16) & 0x1FFFu);
            const int k0 = cur.kt * KT;
            // (copies of the other warps may complete before warp 0 announces the byte count: the transaction count
            // of an mbarrier may run negative, and the phase cannot end before warp 0's arrive)
            if (pw == 0 && lane == 0)
            {
                mbar_expect_tx(bar, T_NO_STAGE ? m.d.bytes
                                               : m.d.bytes + (unsigned)n_loads * box_bytes + (unsigned)n_singles * (KT * 8));
                bulk_g2s(s_blob + st * a.blob_stride, a.blob + ((unsigned long long)m.d.off16 << 4), m.d.bytes, bar);
            }
            if (w == 0)
                asm volatile("griddepcontrol.wait;" ::: "memory"); // B may be the result of the kernel before this one
            if (!T_NO_STAGE && pw + NPW * lane < n_loads)
                tma_box(s_slab + (unsigned)m.ld.y * box_bytes, &box_map, k0, m.ld.x, bar);
            for (int i = pw + NPW * (lane + 32); !T_NO_STAGE && i < n_loads; i += NPW * 32) // more than NPW*32 boxes: rare
            {
                const int2 e = a.loads[(size_t)cur.t * a.NS + i];
                tma_box(s_slab + (unsigned)e.y * box_bytes, &box_map, k0, e.x, bar);
            }
            const long long c1a = TCLK();
            // single rows, four per gather (the builder pads the list and keeps a group inside the pool ring)
            const unsigned pool = s_slab + (unsigned)(a.NS * a.BR) * (KT * 8);
            for (int g = pw + NPW * lane; !T_NO_STAGE && g * 4 < n_singles; g += NPW * 32)
            {
                const int4 rows = g == pw + NPW * lane
                                      ? m.sg
                                      : reinterpret_cast<const int4 *>(a.singles + (size_t)cur.t * a.POOL)[g]; // > 512 singles
                const int pr = (m.d.pool_start + g * 4) % a.POOL;
                tma_gather4(pool + (unsigned)pr * (KT * 8), &row_map, k0, rows, bar);
            }
            work_next(cur);
            ++w;
            if (TPROF)
            {
                const long long c2 = TCLK();
                p_wait += c1 - c0;
                p_issue += c1a - c1;
                p_sgl += c2 - c1a;
                ++p_items;
            }
        };
        Meta m0 = {}, m1 = {}, m2 = {};
        // prologue: metadata of this warp's first two items
        if (ahead.c < a.n_chunks)
        {
            m0 = fetch(ahead);
            work_next(ahead);
        }
        if (ahead.c < a.n_chunks)
        {
            m1 = fetch(ahead);
            work_next(ahead);
        }
        while (cur.c < a.n_chunks)
        {
            step(m0, m2);
            if (cur.c >= a.n_chunks)
                break;
            step(m1, m0);
            if (cur.c >= a.n_chunks)
                break;
            step(m2, m1);
        }
        if (TPROF && lane == 0 && pw == 0)
        {
            a.prof[blockIdx.x * 12 + 0] = p_wait;
            a.prof[blockIdx.x * 12 + 1] = p_issue;
            a.prof[blockIdx.x * 12 + 2] = p_items;
            a.prof[blockIdx.x * 12 + 3] = TCLK() - p_t0;
            a.prof[blockIdx.x * 12 + 4] = p_sgl;
        }
        return;
    }

    // ---------------- consumers ----------------
    const int tw = lane / TL, l = lane % TL;
    const int tq = tw & 1; // team inside its quarter-warp: the two teams read opposite halves of each 128 bytes
    int colo[NL];          // column (in doubles) of accumulator i inside the k-tile
#pragma unroll
    for (int i = 0; i < NL; ++i)
        colo[i] = ((NL > 1 ? (i ^ tq) : i) * TL + l) * 2;

    long long q_wait = 0, q_main = 0, q_t0 = TCLK();
    int st = 0, use = 0;
    asm volatile("griddepcontrol.wait;" ::: "memory"); // C may still be read (as its B) by the kernel before this one
    for (int w = 0; cur.c < a.n_chunks; ++w, work_next(cur))
    {
        const long long c0 = TCLK();
        const int k0 = cur.kt * KT;
        const unsigned blob = s_blob + st * a.blob_stride;
        mbar_wait(full + 8 * st, use & 1);
        const long long c1 = TCLK();
        const int4 hdr = lds128i(blob);
        const int n_units = hdr.y;
        const unsigned units = blob + 16;
        const unsigned vals_s = blob + a.hdr_bytes, ids_s = blob + (unsigned)hdr.w;
        double *__restrict__ Ck = a.C + (long long)hdr.z * a.T * a.ldc + k0; // hdr.z: the tile at this place of the walking order

        // units round-robin over the warps, rotated by the item so the remainder moves around
        for (int u = (warp + w) % NCW; !T_NO_COMPUTE && u < n_units; u += NCW)
        {
            const uint2 e = lds64u(units + (u * UW + tw) * 8);
            const int begin = e.x & 0x1FFF, len = (e.x >> 13) & 0x3FF, row = (e.x >> 23) & 0xFF;
            const bool split = (e.x >> 31) != 0;
            const int maxlen = __reduce_max_sync(0xFFFFFFFFu, len);
            double2 acc[NL];
#pragma unroll
            for (int i = 0; i < NL; ++i)
                acc[i] = make_double2(0.0, 0.0);
            const unsigned vbase = vals_s + begin * 8, ibase = ids_s + e.y * 2;
            int i = 0;
            {
                // Fast path: the steps every team of the unit still has (rows of a unit are of similar length) run without
                // predicates, zero fills and per-load address arithmetic — the predicated loop below issues ~95 instructions
                // per 4 steps for 29 loads and FMAs, and the kernel's issue slots were 59 % busy (profiles/r1_tiled.md).
                // The slab address of accumulator 0 has bit 6 = tq (the slab is 1024-byte aligned, a slab row is a multiple of
                // 128 bytes, l*16 < 64): accumulator x^1 is the same address with bit 6 flipped, x+2 lies 128 bytes further.
                const int fast_end = __reduce_min_sync(0xFFFFFFFFu, len) & ~(U - 1);
                const unsigned b0 = s_slab + colo[0] * 8;
                for (; i < fast_end; i += U)
                {
                    double v[U];
                    unsigned id[U];
#pragma unroll
                    for (int g = 0; g < U; g += 4)
                    {
                        const uint2 four = lds64u(ibase + (i + g) * 2);
                        id[g] = four.x & 0xFFFFu;
                        id[g + 1] = four.x >> 16;
                        id[g + 2] = four.y & 0xFFFFu;
                        id[g + 3] = four.y >> 16;
                    }
#pragma unroll
                    for (int q = 0; q < U; ++q)
                        v[q] = lds64d(vbase + (i + q) * 8);
                    double2 b[U][NL];
#pragma unroll
                    for (int q = 0; q < U; ++q)
                    {
                        const unsigned a0 = b0 + id[q] * (KT * 8), a1 = a0 ^ 64u;
#pragma unroll
                        for (int x = 0; x < NL; ++x)
                            b[q][x] = lds128d(((x & 1) ? a1 : a0) + (x >> 1) * 128);
                    }
#pragma unroll
                    for (int q = 0; q < U; ++q)
#pragma unroll
                        for (int x = 0; x < NL; ++x)
                        {
                            acc[x].x = fma(v[q], b[q][x].x, acc[x].x);
                            acc[x].y = fma(v[q], b[q][x].y, acc[x].y);
                        }
                }
            }
            for (; i < maxlen; i += U)
            {
                static_assert(U % 4 == 0, "ids are read four at a time");
                double v[U];
                unsigned id[U];
#pragma unroll
                for (int g = 0; g < U; g += 4)
                {
                    uint2 four = make_uint2(0u, 0u);
                    if (i + g < len)
                        four = lds64u(ibase + (i + g) * 2);
                    id[g] = four.x & 0xFFFFu;
                    id[g + 1] = four.x >> 16;
                    id[g + 2] = four.y & 0xFFFFu;
                    id[g + 3] = four.y >> 16;
                }
#pragma unroll
                for (int q = 0; q < U; ++q)
                {
                    v[q] = 0.0;
                    if (i + q < len)
                        v[q] = lds64d(vbase + (i + q) * 8);
                }
                double2 b[U][NL];
#pragma unroll
                for (int q = 0; q < U; ++q)
#pragma unroll
                    for (int x = 0; x < NL; ++x)
                    {
                        b[q][x] = make_double2(0.0, 0.0);
                        if (i + q < len)
                            b[q][x] = lds128d(s_slab + id[q] * (KT * 8) + colo[x] * 8);
                    }
#pragma unroll
                for (int q = 0; q < U; ++q)
                {
#pragma unroll
                    for (int x = 0; x < NL; ++x)
                    {
                        acc[x].x = fma(v[q], b[q][x].x, acc[x].x);
                        acc[x].y = fma(v[q], b[q][x].y, acc[x].y);
                    }
                }
            }
            if (split)
            {
                // the 8 teams hold the 8 segments of one row: fold them (fixed order, deterministic).
                // Accumulator x of an odd team sits at the column of accumulator x^1 of an even team: align first.
                double2 al[NL];
#pragma unroll
                for (int x = 0; x < NL; ++x)
                    al[x] = (NL > 1 && tq) ? acc[NL > 1 ? (x ^ 1) : x] : acc[x];
#pragma unroll
                for (int x = 0; x < NL; ++x)
#pragma unroll
                    for (int off = TL; off < 32; off <<= 1)
                    {
                        al[x].x += __shfl_xor_sync(0xFFFFFFFFu, al[x].x, off);
                        al[x].y += __shfl_xor_sync(0xFFFFFFFFu, al[x].y, off);
                    }
                if (tw == 0 && row != (int)UE_PAD_ROW)
                {
                    double *cr = Ck + (long long)row * a.ldc;
#pragma unroll
                    for (int x = 0; x < NL; ++x)
                        if (k0 + (x * TL + l) * 2 < a.kc)
                        {
                            st_c2(cr + (x * TL + l) * 2, al[x].x, al[x].y);
                            for (int d = 0; d < a.extra.n; ++d)
                                st_c2(cr + a.extra.off[d] + (x * TL + l) * 2, al[x].x, al[x].y);
                        }
                }
            }
            else if (row != (int)UE_PAD_ROW)
            {
                double *cr = Ck + (long long)row * a.ldc;
#pragma unroll
                for (int x = 0; x < NL; ++x)
                    if (k0 + colo[x] < a.kc)
                    {
                        st_c2(cr + colo[x], acc[x].x, acc[x].y);
                        for (int d = 0; d < a.extra.n; ++d)
                            st_c2(cr + a.extra.off[d] + colo[x], acc[x].x, acc[x].y);
                    }
            }
        }
        __syncwarp();
        if (lane == 0)
            mbar_arrive(empty + 8 * st); // this warp no longer reads the item's blob, pool rows and slots
        if (++st == D)
        {
            st = 0;
            ++use;
        }
        if (TPROF)
        {
            const long long c2 = TCLK();
            q_wait += c1 - c0;
            q_main += c2 - c1;
        }
    }
    if (TPROF && threadIdx.x == 0)
    {
        a.prof[blockIdx.x * 12 + 8] = q_wait;
        a.prof[blockIdx.x * 12 + 9] = q_main;
        a.prof[blockIdx.x * 12 + 10] = TCLK() - q_t0;
    }
}

// ---- host side ------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn()
{
    static EncodeTiledFn fn = [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return (EncodeTiledFn)p;
    }();
    return fn;
}

int encode_b_map(CUtensorMap *map, const double *d_B, long long ldb, int kc, int n_cols, int kt, int rows)
{
    EncodeTiledFn enc = encode_fn();
    if (!enc)
    {
        set_error("cuTensorMapEncodeTiled is not available from this driver");
        return SPMM_ERR_CUDA;
    }
    const cuuint64_t gdim[2] = {(cuuint64_t)kc, (cuuint64_t)n_cols};
    const cuuint64_t gstride[1] = {(cuuint64_t)ldb * 8};
    const cuuint32_t box[2] = {(cuuint32_t)kt, (cuuint32_t)rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult cr = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double *>(d_B), gdim, gstride, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS)
    {
        set_error("cuTensorMapEncodeTiled failed with CUresult " + std::to_string((int)cr));
        return SPMM_ERR_CUDA;
    }
    return SPMM_OK;
}

int lg2(int x)
{
    int l = 0;
    while ((1 << l) < x)
        ++l;
    return l;
}

unsigned hdr_bytes_of(int T) { return 16u + 64u * (unsigned)units_cap(T); }

struct TiledSmem
{
    size_t blob_stride, slab_off, slab_bytes, total;
};

TiledSmem tiled_smem(int kt, int depth, int T, int BR, int NS, int POOL, int max_blob)
{
    TiledSmem m;
    (void)T;
    m.blob_stride = ((size_t)max_blob + 32 + 127) & ~127ull; // header + unit table + values + ids of the largest tile
    m.slab_off = (BLOB_OFF + (size_t)depth * m.blob_stride + 1023) & ~1023ull;
    m.slab_bytes = ((size_t)NS * BR + (size_t)POOL) * kt * 8;
    m.total = m.slab_off + m.slab_bytes + 1024; // + slack: the kernel aligns its base to 1024
    return m;
}

template <int KT, int NCW, int U, int NPW>
int launch_tiled_t(const spmm_csr_s *A, const double *d_B, long long ldb, double *d_C, long long ldc, int kc,
                   cudaStream_t stream, const ExtraDst &extra)
{
    auto kern = spmm_tiled_kernel<KT, NCW, U, NPW>;
    const TiledSmem m = tiled_smem(KT, A->tl_depth, A->tl_T, A->tl_BR, A->tl_NS, A->tl_POOL, A->tl_max_blob);
    if (m.total > (size_t)SMEM_CAP)
    {
        set_error("tiled kernel: the tile layout does not fit in shared memory");
        return SPMM_ERR_UNSUPPORTED;
    }
    static std::mutex mu;
    static std::map<std::pair<const void *, int>, int> configured; // function attributes are per device
    {
        std::lock_guard<std::mutex> lk(mu);
        int &have = configured[{(const void *)kern, A->device}];
        if (!have)
        {
            SPMM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_CAP));
            have = 1;
        }
    }
    CUtensorMap box_map, row_map;
    int rc = encode_b_map(&box_map, d_B, ldb, kc, A->n_cols, KT, A->tl_BR);
    if (!rc)
        rc = encode_b_map(&row_map, d_B, ldb, kc, A->n_cols, KT, 1);
    if (rc)
        return rc;
    TiledArgs a = {};
    a.blob = A->d_tblob;
    a.tdesc = reinterpret_cast<const TileDesc *>(A->d_tdesc);
    a.loads = reinterpret_cast<const int2 *>(A->d_tloads);
    a.singles = A->d_tsingles;
    a.B = d_B;
    a.C = d_C;
    a.extra = extra;
    a.ldb = ldb;
    a.ldc = ldc;
    a.n_tiles = A->tl_tiles;
    a.tiles_per_chunk = A->tl_chunk;
    a.ksplit = std::max(1, A->tl_ksplit);
    a.n_chunks = ((A->tl_tiles + A->tl_chunk - 1) / A->tl_chunk) * a.ksplit;
    a.T = A->tl_T;
    a.BR = A->tl_BR;
    a.NS = A->tl_NS;
    a.POOL = A->tl_POOL;
    a.kc = kc;
    a.nkt = (kc + KT - 1) / KT;
    a.depth = A->tl_depth;
    a.hdr_bytes = hdr_bytes_of(A->tl_T);
    a.blob_stride = (unsigned)m.blob_stride;
    a.slab_off = (unsigned)m.slab_off;
    const int grid = std::max(1, std::min(a.n_chunks, device_props(A->device).sm_count));
#if TPROF
    static long long *d_prof = nullptr;
    static int prof_calls = 0;
    if (!d_prof)
        SPMM_CUDA(cudaMalloc(&d_prof, sizeof(long long) * 12 * 1024));
    a.prof = d_prof;
#endif
    // The prologue copies the first blob of each CTA before griddepcontrol.wait: after a value refresh this launch must not
    // start under the tail of the kernels before it.
    const bool pdl = tuning().tiled_pdl != 0 && !A->tl_refreshed;
    A->tl_refreshed = false;
    if (pdl)
    {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)grid);
        cfg.blockDim = dim3((unsigned)((NCW + NPW) * 32));
        cfg.dynamicSmemBytes = m.total;
        cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        SPMM_CUDA(cudaLaunchKernelEx(&cfg, kern, a, box_map, row_map));
    }
    else
        kern<<<grid, (NCW + NPW) * 32, m.total, stream>>>(a, box_map, row_map);
    SPMM_CUDA(cudaGetLastError());
#if TPROF
    if (++prof_calls == 20)
    {
        std::vector<long long> h(12 * grid);
        SPMM_CUDA(cudaStreamSynchronize(stream));
        SPMM_CUDA(cudaMemcpy(h.data(), d_prof, sizeof(long long) * 12 * grid, cudaMemcpyDeviceToHost));
        double s[12] = {0};
        for (int i = 0; i < grid; ++i)
            for (int j = 0; j < 12; ++j)
                s[j] += (double)h[i * 12 + j] / grid;
        fprintf(stderr,
                "[tiled prof] per CTA (clk): producer 0 wait %.0f blob+boxes %.0f items %.0f total %.0f singles+rest %.0f "
                "(%.0f) | consumer warp 0 wait-full %.0f work %.0f total %.0f\n",
                s[0], s[1], s[2], s[3], s[4], s[5], s[8], s[9], s[10]);
    }
#endif
    return SPMM_OK;
}

struct BuildResult
{
    int status[ST_WORDS];
    unsigned long long totals[TOT_WORDS];
};

int build_tiles_once(spmm_csr_s *A, const BuildParams &p, bool dry, BuildResult *res)
{
    const int n_chunks = (p.n_tiles + p.tiles_per_chunk - 1) / p.tiles_per_chunk;
    const size_t bytes = sizeof(int) * ST_WORDS + sizeof(unsigned long long) * TOT_WORDS;
    int *d_status = nullptr;
    SPMM_CUDA(cudaMalloc(&d_status, bytes));
    unsigned long long *d_total = reinterpret_cast<unsigned long long *>(d_status + ST_WORDS);
    cudaError_t e = cudaMemset(d_status, 0, bytes);
    if (e == cudaSuccess)
    {
        if (dry)
            tile_build_kernel<true><<<n_chunks, TB_THREADS>>>(A->d_rowptr, A->d_colidx, A->d_vals, p, nullptr, nullptr,
                                                              nullptr, nullptr, d_status, d_total, A->d_torder);
        else
            tile_build_kernel<false><<<n_chunks, TB_THREADS>>>(A->d_rowptr, A->d_colidx, A->d_vals, p, A->d_tblob,
                                                               reinterpret_cast<TileDesc *>(A->d_tdesc),
                                                               reinterpret_cast<int2 *>(A->d_tloads), A->d_tsingles,
                                                               d_status, d_total, A->d_torder);
        e = cudaGetLastError();
    }
    unsigned char h[sizeof(int) * ST_WORDS + sizeof(unsigned long long) * TOT_WORDS];
    if (e == cudaSuccess)
        e = cudaMemcpy(h, d_status, bytes, cudaMemcpyDeviceToHost);
    cudaFree(d_status);
    SPMM_CUDA(e);
    memcpy(res->status, h, sizeof(int) * ST_WORDS);
    memcpy(res->totals, h + sizeof(int) * ST_WORDS, sizeof(unsigned long long) * TOT_WORDS);
    if (getenv("SPMM_TILED_DEBUG"))
        fprintf(stderr,
                "[tiled build] %s T=%d BR=%d NS=%d POOL=%d depth=%d thr=%d chunk=%d band=%d group=%d: fail=%d max_recs=%d max_pool=%d max_loads=%d "
                "drains=%d loads=%llu singles=%llu\n",
                dry ? "dry" : "final", p.T, 1 << p.lgBR, p.NS, p.POOL, p.depth, p.thr, p.tiles_per_chunk, A->tl_stride, A->tl_group, res->status[ST_FAIL],
                res->status[ST_MAXREC], res->status[ST_MAXPOOL], res->status[ST_MAXLOAD], res->status[ST_DRAINS], res->totals[TOT_LOADS],
                res->totals[TOT_SINGLES]);
    return SPMM_OK;
}
} // namespace

namespace
{
// Histogram of the distances col - row >= NEAR over every `step`-th row, in bins of `bin` rows (counts and sums).
__global__ void far_band_hist_kernel(const int *__restrict__ rowptr, const int *__restrict__ colidx, int n_rows, int step,
                                     int near, int bin, unsigned long long *__restrict__ cnt, unsigned long long *__restrict__ sum)
{
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long r = i * step;
    if (r >= n_rows)
        return;
    for (int j = rowptr[r]; j < rowptr[r + 1]; ++j)
    {
        const int d = colidx[j] - (int)r;
        if (d >= near)
        {
            atomicAdd(cnt + d / bin, 1ull);
            atomicAdd(sum + d / bin, (unsigned long long)d);
        }
    }
}

// Distance (in rows) of the matrix's dominant far band: FEM-like matrices on a 3-D grid couple row r with rows r +- P
// (the next grid plane). 0 when no band far from the diagonal holds a sizeable share of the non-zeros. Found on the device
// from a sample of the rows (every 8th: a band that matters shows in any sample); only the histogram comes back.
int detect_far_band(const spmm_csr_s *A, int *stride_rows)
{
    *stride_rows = 0;
    if (A->n_rows < 4096 || A->nnz == 0)
        return SPMM_OK;
    constexpr int NEAR = 256, STEP = 8;
    const int bin = std::max(64, A->n_cols / 32768);
    const size_t n_bins = (size_t)A->n_cols / bin + 2;
    unsigned long long *d_hist = nullptr;
    SPMM_CUDA(cudaMalloc(&d_hist, sizeof(unsigned long long) * 2 * n_bins));
    std::vector<unsigned long long> h(2 * n_bins);
    cudaError_t e = cudaMemset(d_hist, 0, sizeof(unsigned long long) * 2 * n_bins);
    if (e == cudaSuccess)
    {
        const long long sampled = ((long long)A->n_rows + STEP - 1) / STEP;
        far_band_hist_kernel<<<(unsigned)((sampled + 255) / 256), 256>>>(A->d_rowptr, A->d_colidx, A->n_rows, STEP, NEAR, bin,
                                                                          d_hist, d_hist + n_bins);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess)
        e = cudaMemcpy(h.data(), d_hist, sizeof(unsigned long long) * 2 * n_bins, cudaMemcpyDeviceToHost);
    cudaFree(d_hist);
    SPMM_CUDA(e);
    const unsigned long long *cnt = h.data(), *sum = h.data() + n_bins;
    size_t m = 0;
    for (size_t i = 1; i < n_bins; ++i)
        if (cnt[i] > cnt[m])
            m = i;
    unsigned long long c = 0, sm = 0;
    for (size_t i = m >= 2 ? m - 2 : 0; i <= m + 2 && i < n_bins; ++i)
    {
        c += cnt[i];
        sm += sum[i];
    }
    // the band holds at least 1/12 of all non-zeros (a third of the upper triangle of a 27-point stencil); c counts a sample
    if (c > 0 && (long long)c * STEP * 12 >= A->nnz)
        *stride_rows = (int)(sm / c);
    return SPMM_OK;
}

// Walking order for tiles of T rows: tiles one far band (S tiles) apart are visited in turn, G bands per group, so the B rows
// a tile stages for the next plane are still in the window when that plane's tile comes (1 + 2/G stagings per B row
// instead of 3). nullptr order = as they lie.
int set_tile_order(spmm_csr_s *A, int n_tiles, int T, int stride_rows, int G)
{
    cudaFree(A->d_torder);
    A->d_torder = nullptr;
    A->tl_stride = A->tl_group = 0;
    const int S = T > 0 ? (stride_rows + T / 2) / T : 0;
    if (stride_rows <= 0 || G <= 1 || S < 2 || n_tiles < 2 * S)
        return SPMM_OK;
    std::vector<int> order;
    order.reserve((size_t)n_tiles);
    for (int g0 = 0; g0 < n_tiles; g0 += G * S)
        for (int i = 0; i < S; ++i)
            for (int q = 0; q < G; ++q)
            {
                const int t = g0 + q * S + i;
                if (t < n_tiles)
                    order.push_back(t);
            }
    SPMM_CUDA(cudaMalloc(&A->d_torder, sizeof(int) * (size_t)n_tiles));
    SPMM_CUDA(cudaMemcpy(A->d_torder, order.data(), sizeof(int) * (size_t)n_tiles, cudaMemcpyHostToDevice));
    A->tl_stride = stride_rows;
    A->tl_group = G;
    return SPMM_OK;
}
} // namespace

void free_tiles(spmm_csr_s *A)
{
    cudaFree(A->d_tblob);
    cudaFree(A->d_tdesc);
    cudaFree(A->d_tloads);
    cudaFree(A->d_tsingles);
    cudaFree(A->d_torder);
    A->d_torder = nullptr;
    A->tl_stride = A->tl_group = 0;
    A->d_tblob = nullptr;
    A->d_tdesc = nullptr;
    A->d_tloads = nullptr;
    A->d_tsingles = nullptr;
    A->tl_T = A->tl_BR = A->tl_tiles = A->tl_NS = A->tl_POOL = A->tl_max_recs = A->tl_max_blob = A->tl_chunk = A->tl_kt = A->tl_depth = A->tl_ksplit = 0;
    A->tl_box_rows_loaded = A->tl_single_rows = 0;
}

static bool tiled_shape_ok(const spmm_csr_s *A, const Request &r)
{
    return A->tl_T > 0 && r.kc >= 2 && r.kc % 2 == 0 && r.ldb % 2 == 0 && r.ldc % 2 == 0 && ((uintptr_t)r.B % 16 == 0) &&
           ((uintptr_t)r.C % 16 == 0) && (unsigned long long)r.ldb * 8ull < (1ull << 40);
}

int tiled_check(const spmm_csr_s *A, const Request &r)
{
    SPMM_REQUIRE(A->tl_T != 0, "tiled kernel requested but spmm_csr_build_tiles was not called (or found no fitting tile shape)");
    if (tiled_shape_ok(A, r))
        return SPMM_OK;
    set_error("tiled kernel: needs even k, even leading dimensions and 16-byte aligned B and C");
    return SPMM_ERR_UNSUPPORTED;
}

// AUTO builds the tile layout the first time a multiply can use it (even k >= 4, mid-sized matrix with regular rows):
// one-off, ~10 ms, about 10 bytes per non-zero next to the CSR; it is rebuilt when k moves to the other k-tile width (8 columns
// for k <= 8) or to fewer k-tiles than CTAs share a chunk. spmm_tune_set("tiled", 0) or an explicit
// spmm_csr_build_tiles(A, 0, 0) keeps the CSR kernels. Failure to build is not an error: the CSR kernels stay in charge.
void auto_tile_layout(spmm_csr_s *A, int k)
{
    if (A->tl_auto && A->tl_T != 0 && (A->tl_ksplit > std::max(1, (k + 15) / 16) || (A->tl_kt == 8) != (k <= 8)))
    {
        free_tiles(A);
        A->tl_tried = false;
    }
    if (A->tl_tried || A->tl_T != 0 || tuning().tiled == 0 || k < 4 || k % 2 != 0 || A->nnz < 200000 || A->nnz > (64ll << 20))
        return;
    // The layout costs about 150 multiplies to build: a handle that is multiplied once (the reference calls each function
    // once per run, main.cpp:78) keeps the CSR row kernels; the layout is built when the handle comes back.
    if (A->auto_calls++ < tuning().tiled_auto_after)
        return;
    A->tl_tried = true;
    const int brc = build_tiles(A, -1, 0, tiles_kt_for(k), tuning().tiled_ksplit > 0 ? tuning().tiled_ksplit : tiles_ksplit_for(k));
    A->tl_auto = true;
    if (brc != SPMM_OK)
        free_tiles(A);
}

// tile layout: measured faster than the CSR kernels from k = 8 up when rows of a tile share B rows (profiles/r1_tiled.md)
bool tiled_auto_ok(const spmm_csr_s *A, const Request &r)
{
    const Tuning &t = tuning();
    if (t.tiled == 0 || !tiled_shape_ok(A, r))
        return false;
    const double staged = (double)A->tl_box_rows_loaded + (double)A->tl_single_rows;
    const double reuse = staged > 0 ? (double)A->nnz / staged : 0.0;
    return t.tiled == 1 || (r.kc >= (A->tl_kt == 8 ? 4 : 8) && reuse >= 2.0 && A->tl_drains * 20 <= A->tl_tiles);
}

int launch_tiled(const spmm_csr_s *A, const Request &r, cudaStream_t stream)
{
    const ExtraDst x = r.extra ? *r.extra : ExtraDst();
    note_kernel("spmm_tiled_kernel");
    // the kernel's shape is the one the layout was cut for
    if (A->tl_kt == 8)
        return launch_tiled_t<8, 16, 4, 4>(A, r.B, r.ldb, r.C, r.ldc, r.kc, stream, x);
    return launch_tiled_t<16, 16, 4, 4>(A, r.B, r.ldb, r.C, r.ldc, r.kc, stream, x);
}

int update_values(spmm_csr_s *A, const double *d_src, cudaStream_t stream)
{
    double *csr_out = d_src == A->d_vals ? nullptr : A->d_vals; // the caller edited A's own array: only the layout is behind
    if (A->tl_T == 0)
    {
        if (csr_out)
            SPMM_CUDA(cudaMemcpyAsync(csr_out, d_src, sizeof(double) * (size_t)A->nnz, cudaMemcpyDeviceToDevice, stream));
        return SPMM_OK;
    }
    tile_refresh_kernel<<<A->tl_tiles, TR_THREADS, 0, stream>>>(A->d_rowptr, d_src, csr_out, A->d_tblob, A->n_rows, A->tl_T,
                                                                (int)hdr_bytes_of(A->tl_T));
    SPMM_CUDA(cudaGetLastError());
    A->tl_refreshed = true;
    return SPMM_OK;
}

} // namespace spmm

namespace spmm
{
// kt_want: k-tile width the layout is cut for, 8 or 16 (0 = 16), the two widths the tiled kernel is built for.
// ksplit_want: CTAs per chunk (0 = the tuning knob, else its default).
// Explicit parameters, not the process-wide tuning: concurrent multiplies of rank-threads build their layouts side by side.
int build_tiles(spmm_csr_t A, int rows_per_tile, int box_rows, int kt_want, int ksplit_want)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    SPMM_REQUIRE(rows_per_tile == 0 || rows_per_tile == -1 ||
                     (rows_per_tile >= 8 && rows_per_tile <= TB_MAXT && rows_per_tile % 8 == 0),
                 "rows_per_tile must be 0 (drop), -1 (auto) or a multiple of 8 in [8, 248]");
    SPMM_REQUIRE(box_rows == 0 || box_rows == 4 || box_rows == 8 || box_rows == 16 || box_rows == 32,
                 "box_rows must be 0 (auto), 4, 8, 16 or 32");
    SPMM_REQUIRE(kt_want == 0 || kt_want == 8 || kt_want == 16, "k-tile must be 0 (auto), 8 or 16");
    SPMM_CUDA(cudaSetDevice(A->device));
    free_tiles(A);
    A->tl_tried = true; // an explicit call (build or drop) settles it: AUTO does not try again
    A->tl_auto = false;
    if (rows_per_tile == 0 || A->n_rows == 0 || A->nnz == 0)
        return SPMM_OK;
    const Tuning &tn = tuning();
    const int BR = box_rows ? box_rows : 16;
    const int kt = kt_want ? kt_want : 16; // k-tile the window is sized for
    const int sms = device_props(A->device).sm_count;
    // measured on the cop20k_A shape (profiles/r1_tiled.md): tall tiles and a wide window beat a deeper pipeline
    const int kt_for_depth = kt;
    // (64-byte window rows leave room for a third work item in flight: measured 20.6 against 22.7 us at k=8, T=96)
    const int depth = (tn.tiled_depth >= 2 && tn.tiled_depth <= TB_DMAX) ? tn.tiled_depth : (kt_for_depth == 8 ? 3 : 2);
    const int ksplit = std::max(1, std::min(8, ksplit_want > 0 ? ksplit_want : tn.tiled_ksplit)); // CTAs per chunk

    BuildParams p = {};
    p.n_rows = A->n_rows;
    p.lgBR = lg2(BR);
    p.thr = tn.tiled_thr > 0 ? tn.tiled_thr : std::max(2, 3 * BR / 8);
    p.depth = depth;
    BuildResult res;
    int far_band = tn.tiled_stride;
    const int group = tn.tiled_group > 0 ? tn.tiled_group : 2; // measured on cfg2: 2 stages a third fewer B rows at no cost; 3+ overflow the window (drains)
    if (far_band == 0 && group > 1)
    {
        const int rc = detect_far_band(A, &far_band);
        if (rc)
            return rc;
    }
    const int auto_cand[] = {96, 80, 72, 64, 48, 32, 16};
    int chosen = 0;
    BuildParams best = {};
    double best_score = 0.0;
    // short chunks (one CTA per chunk walks every k-tile) favour 64-row tiles, long shared chunks taller ones (measured)
    const int first_cand = (ksplit > 1 || kt == 8) ? 0 : 3;
    for (int ci = first_cand; ci < (rows_per_tile > 0 ? first_cand + 1 : 7); ++ci)
    {
        const int T = rows_per_tile > 0 ? rows_per_tile : auto_cand[ci];
        p.T = T;
        p.n_tiles = (A->n_rows + T - 1) / T;
        p.hdr_bytes = (int)hdr_bytes_of(T);
        // chunks: a multiple of the SM count, about 48 tiles each (window warm-up amortised, work balanced)
        const int per_sm = std::max(1, (int)((p.n_tiles + (long long)sms * 48 - 1) / ((long long)sms * 48)));
        const int n_chunks_want = std::max(1, sms * per_sm / ksplit); // ksplit CTAs share a chunk (one k-tile group each)
        p.tiles_per_chunk =
            tn.tiled_chunk > 0 ? tn.tiled_chunk : std::max(1, (p.n_tiles + n_chunks_want - 1) / n_chunks_want);
        int rc = set_tile_order(A, p.n_tiles, T, far_band, group);
        if (rc)
            return rc;
        // dry run with the largest window: record maximum and singles of this tile height
        p.NS = TB_NSMAX;
        p.POOL = 1 << 20;
        rc = build_tiles_once(A, p, true, &res);
        if (rc)
            return rc;
        if (res.status[ST_FAIL])
            continue;
        // singles pool: one and a half times the average demand of `depth` tiles in flight (tiles that need more are
        // marked to wait for the pipeline to drain); window = what shared memory leaves after blob ring and pool
        const double avg = (double)res.totals[TOT_SINGLES] / std::max(1, p.n_tiles);
        int pool = tn.tiled_pool > 0 ? tn.tiled_pool : (int)(1.5 * depth * avg) + 32;
        pool = std::min(std::max(pool, 32), std::max(32, res.status[ST_MAXPOOL] + 8));
        pool = (pool + 7) & ~7;
        const TiledSmem fixed = tiled_smem(kt, depth, T, BR, 0, pool, res.status[ST_MAXBLOB]);
        if (fixed.total + 8ull * BR * kt * 8 > (size_t)SMEM_CAP)
            continue;
        p.NS = (int)std::min<size_t>(TB_NSMAX, ((size_t)SMEM_CAP - fixed.total) / ((size_t)BR * kt * 8));
        if (tn.tiled_ns > 0)
            p.NS = std::min(p.NS, tn.tiled_ns);
        p.POOL = pool;
        if ((long long)p.NS * BR + p.POOL > 65535)
            continue; // slab rows are 16-bit ids
        rc = build_tiles_once(A, p, true, &res);
        if (rc)
            return rc;
        if (res.status[ST_FAIL])
            continue;
        // B rows brought into shared memory per pass: the L2 -> SM traffic this layout costs
        // (a drain costs about as much as staging a few hundred rows)
        const double score =
            (double)res.totals[TOT_LOADS] * BR + (double)res.totals[TOT_SINGLES] + 256.0 * res.status[ST_DRAINS];
        if (!chosen || score < best_score)
        {
            chosen = T;
            best = p;
            best_score = score;
        }
        // tall tiles amortise the per-item latency: take the tallest one that rarely has to drain the pipeline
        if (res.status[ST_DRAINS] * 50 <= p.n_tiles)
        {
            chosen = T;
            best = p;
            break;
        }
    }
    p = best;
    if (!chosen)
    {
        if (rows_per_tile > 0)
        {
            set_error("tile layout: this tile height does not fit (more than 6144 non-zeros or 1024 boxes per tile, or "
                      "records + single rows exceed shared memory)");
            return SPMM_ERR_UNSUPPORTED;
        }
        return SPMM_OK; // no tile shape fits: the CSR kernels stay in charge
    }
    {
        const int orc = set_tile_order(A, p.n_tiles, p.T, far_band, group); // the order of the chosen tile height
        if (orc)
            return orc;
    }
    const unsigned long long blob_bytes = blob_offset(p.n_tiles, A->nnz, p.hdr_bytes, p.T) + 64;
    SPMM_REQUIRE((blob_bytes >> 4) < (1ull << 32), "matrix too large for the tile layout");
    SPMM_CUDA(cudaMalloc(&A->d_tblob, blob_bytes + 16));
    SPMM_CUDA(cudaMalloc(&A->d_tdesc, sizeof(TileDesc) * (size_t)p.n_tiles));
    SPMM_CUDA(cudaMalloc(&A->d_tloads, sizeof(int2) * (size_t)p.n_tiles * p.NS));
    SPMM_CUDA(cudaMalloc(&A->d_tsingles, sizeof(int) * (size_t)p.n_tiles * p.POOL));
    int rc = build_tiles_once(A, p, false, &res);
    if (rc || res.status[ST_FAIL])
    {
        free_tiles(A);
        if (rc)
            return rc;
        set_error("tile layout: build failed on the final pass (status " + std::to_string(res.status[ST_FAIL]) + ")");
        return SPMM_ERR_UNSUPPORTED;
    }
    A->tl_T = p.T;
    A->tl_BR = BR;
    A->tl_tiles = p.n_tiles;
    A->tl_NS = p.NS;
    A->tl_POOL = p.POOL;
    A->tl_max_recs = res.status[ST_MAXREC];
    A->tl_max_blob = res.status[ST_MAXBLOB];
    A->tl_chunk = p.tiles_per_chunk;
    A->tl_kt = kt;
    A->tl_depth = depth;
    A->tl_ksplit = ksplit;
    A->tl_drains = res.status[ST_DRAINS];
    A->tl_box_rows_loaded = (long long)res.totals[TOT_LOADS] * BR;
    A->tl_single_rows = (long long)res.totals[TOT_SINGLES];
    return SPMM_OK;
}

} // namespace spmm

using namespace spmm;

extern "C"
{

int spmm_csr_build_tiles(spmm_csr_t A, int rows_per_tile, int box_rows)
{
    if (A && A->d_rowptr64)
        return refuse_offsets64("spmm_csr_build_tiles", "SPMM_KERNEL_AUTO, ROWS, MERGE or STREAM");
    return build_tiles(A, rows_per_tile, box_rows, 0, 0);
}

int spmm_csr_build_tiles_for_k(spmm_csr_t A, int rows_per_tile, int box_rows, int k)
{
    SPMM_REQUIRE(k >= 0, "k is negative");
    if (A && A->d_rowptr64)
        return refuse_offsets64("spmm_csr_build_tiles_for_k", "SPMM_KERNEL_AUTO, ROWS, MERGE or STREAM");
    if (k == 0)
        return build_tiles(A, rows_per_tile, box_rows, 0, 0);
    return build_tiles(A, rows_per_tile, box_rows, tiles_kt_for(k), tiles_ksplit_for(k));
}

int spmm_csr_tile_info(spmm_csr_t A, int *rows_per_tile, int *box_rows, int *window_slots, int *max_records,
                       double *reuse, double *single_fraction)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    if (rows_per_tile) *rows_per_tile = A->tl_T;
    if (box_rows) *box_rows = A->tl_BR;
    if (window_slots) *window_slots = A->tl_NS;
    if (max_records) *max_records = A->tl_max_recs;
    const double staged = (double)A->tl_box_rows_loaded + (double)A->tl_single_rows;
    if (reuse)
        *reuse = (A->tl_T && staged > 0) ? (double)A->nnz / staged : 0.0;
    if (single_fraction)
        *single_fraction = (A->tl_T && A->nnz) ? (double)A->tl_single_rows / (double)A->nnz : 0.0;
    return SPMM_OK;
}

} // extern "C"
