// spmm_dispatch.cu — picks the team shape for a launch and forwards to the per-W
// translation units. See spmm_launch.cuh for the rules.
#include "spmm_launch.cuh"

namespace spmm
{

namespace
{
int next_pow2(int x)
{
    int p = 1;
    while (p < x)
        p <<= 1;
    return p;
}
int floor_pow2(int x)
{
    int p = 1;
    while (p * 2 <= x)
        p <<= 1;
    return p;
}

struct Shape
{
    int w, kl, nv, tiles;
};

Shape pick_shape(const double *d_B, long long ldb, const double *d_C, long long ldc, int kc)
{
    const Tuning &t = tuning();
    const bool even = (kc % 2 == 0) && (ldb % 2 == 0) && (ldc % 2 == 0) && ((uintptr_t)d_B % 16 == 0) &&
                      ((uintptr_t)d_C % 16 == 0);
    Shape s;
    s.w = even ? 2 : 1;
    if (t.rows_vec == 1)
        s.w = 1;
    const int kq = (kc + s.w - 1) / s.w; // accesses needed across the columns
    if (kq <= 8)
    {
        s.kl = next_pow2(kq);
        s.nv = 1;
    }
    else if (kq <= 16)
    {
        s.kl = 8;
        s.nv = 2;
    }
    else if (kq <= 32)
    {
        s.kl = 8;
        s.nv = 4;
    }
    else if (kq <= 64)
    {
        s.kl = 16;
        s.nv = 4;
    }
    else
    {
        s.kl = 32;
        s.nv = 4;
    }
    if (t.rows_kl > 0)
        s.kl = t.rows_kl;
    if (t.rows_nv > 0)
        s.nv = t.rows_nv;
    const int tile = s.kl * s.nv;
    s.tiles = (kq + tile - 1) / tile;
    return s;
}
} // namespace

// set around a launch whose B pointer is the virtual base of a window of rows (rows outside the window are not mapped):
// nothing may touch B beyond the rows the matrix's column ids name — no bulk prefetch of "all of B"
static thread_local bool t_b_is_window = false;
void set_b_window(bool on) { t_b_is_window = on; }

int launch_rows(const spmm_csr_s *A, int row_begin, int row_end, long long nnz_lo, long long nnz_hi, int c_row0,
                const double *d_B, long long ldb, double *d_C, long long ldc, int kc, int derived,
                cudaStream_t stream, const ExtraDst *extra)
{
    if (row_end <= row_begin || kc <= 0)
        return SPMM_OK;
    const Tuning &t = tuning();
    const Shape s = pick_shape(d_B, ldb, d_C, ldc, kc);
    // whole-matrix launch with a derived layout on the handle: use it when the shape fits
    const bool whole = row_begin == 0 && row_end == A->n_rows && nnz_lo == 0 && nnz_hi == A->nnz && c_row0 == 0;
    if (derived && whole)
    {
        if (derived == 6 || (derived == 1 && A->tl_T && t.tiled != 0))
        {
            // tile layout: measured faster than the CSR kernels from k = 8 up when rows of a tile share B rows (profiles/r1_tiled.md)
            const bool fits = tiled_shape_ok(A, d_B, ldb, d_C, ldc, kc);
            const double staged = (double)A->tl_box_rows_loaded + (double)A->tl_single_rows;
            const double reuse = staged > 0 ? (double)A->nnz / staged : 0.0;
            if (fits && (derived == 6 || t.tiled == 1 || (kc >= (A->tl_kt == 8 ? 4 : 8) && reuse >= 2.0 && A->tl_drains * 20 <= A->tl_tiles)))
                return launch_tiled(A, d_B, ldb, d_C, ldc, kc, stream, extra);
            if (derived == 6)
            {
                set_error("tiled kernel: needs even k, even leading dimensions and 16-byte aligned B and C");
                return SPMM_ERR_UNSUPPORTED;
            }
        }
    }
    int np = 1;
    if (s.nv == 1)
    {
        // lanes of a warp that a single row can keep busy: about half its mean length
        const int want = floor_pow2(std::max(1, (int)(A->sched.mean_len * 0.5)));
        np = std::max(1, std::min(want, 32 / s.kl));
        if (s.kl >= 4)
            np = std::min(np, 2); // measured (profiles/): 2 side-by-side non-zeros beat 4 once a row piece is >= 64 B
    }
    if (t.rows_np > 0)
        np = t.rows_np;
    if (s.nv != 1)
        np = 1;
    np = std::max(1, std::min(np, 32 / s.kl));
    // B larger than L2 (gathers go to HBM): more rows in flight per team pay (cfg5: 25.5 -> 23.6 ms at unroll 4); B resident
    // in L2 / L1 (cfg2): 2 is the measured optimum for wide pieces
    const bool b_beyond_l2 = (long long)A->n_cols * kc * 8 > device_props(A->device).l2_bytes;
    int u = t.rows_unroll > 0 ? t.rows_unroll : (np >= 8 ? 1 : np >= 2 ? 2 : (s.nv >= 4 ? (b_beyond_l2 ? 4 : 2) : 4));

    SpmmArgs args = {};
    if (extra)
        args.extra = *extra;
    args.rowptr = A->d_rowptr;
    args.colidx = A->d_colidx;
    args.vals = A->d_vals;
    args.B = d_B;
    args.C = d_C;
    args.ldb = ldb;
    args.ldc = ldc;
    args.row_begin = row_begin;
    args.row_end = row_end;
    args.nnz_lo = (int)nnz_lo;
    args.nnz_hi = (int)nnz_hi;
    args.c_row0 = c_row0;
    args.kc = kc;
    // L2 prefetch only when the operands are 16-byte aligned, B is one contiguous block that starts
    // at column 0 of its rows (no k-slab), and the A arrays are the handle's own (padded) allocations
    const bool aligned = ((uintptr_t)A->d_colidx % 16 == 0) && ((uintptr_t)A->d_vals % 16 == 0) && ((uintptr_t)d_B % 16 == 0);
    args.prefetch = aligned ? (t.rows_prefetch >= 0 ? t.rows_prefetch : 3) : 0;
    args.b_bytes = (ldb == kc && !t_b_is_window) ? (long long)A->n_cols * ldb * 8 : 0;
    note_kernel("spmm_rows_kernel");
    return s.w == 2 ? launch_rows_w2(A, s.kl, s.nv, np, u, args, s.tiles, A->device, stream)
                    : launch_rows_w1(A, s.kl, s.nv, np, u, args, s.tiles, A->device, stream);
}

int launch_merge(spmm_csr_s *A, int row_begin, int row_end, long long nnz_lo, long long nnz_hi, int c_row0,
                 const double *d_B, long long ldb, double *d_C, long long ldc, int kc, cudaStream_t stream,
                 const ExtraDst *extra)
{
    if (row_end <= row_begin || kc <= 0)
        return SPMM_OK;
    const Tuning &t = tuning();
    Shape s = pick_shape(d_B, ldb, d_C, ldc, kc);
    // Team shape: pick_shape's (8 lanes x 2 accesses at k = 32). Measured on cfg3 (R-MAT 2^22, k = 32) after the kernel was
    // rebuilt around batches of KL non-zeros (coalesced id/value loads one batch ahead, B rows gathered 4 at a time whatever
    // rows they belong to): 8 x 2 unroll 4 at 80 registers 2.17 ms, 16 x 1 2.34 ms, unroll 8 (127 registers) 4.5 ms
    // (gpurun_out/s5_tune_mb1.jsonl); the row-by-row kernel before it took 3.06-3.50 ms.
    const int u = t.rows_unroll > 0 ? t.rows_unroll : (s.nv >= 4 ? 2 : 4);
    const long long total = (long long)(row_end - row_begin) + (nnz_hi - nnz_lo);
    long long items = t.merge_items > 0 ? t.merge_items : 512;
    // enough teams to fill the machine, few enough that the carry rows stay a small fraction of C
    // (a shard of long rows — the first non-zero range of an R-MAT matrix averages 477 per row — is cut less finely: every
    // team inside a row leaves a carry slot and the fix-up walks them in order; measured per range in gpurun_out/s28_*)
    const double avg_row = (double)(nnz_hi - nnz_lo) / std::max(1, row_end - row_begin);
    const int wave = t.merge_wave > 0 ? t.merge_wave : (avg_row > 256.0 ? 32 : 64);
    const long long teams_per_wave = (long long)device_props(A->device).sm_count * wave * (32 / s.kl);
    while (items > 64 && (total + items - 1) / items < teams_per_wave)
        items >>= 1;
    const long long n_teams = std::max(1LL, (total + items - 1) / items);
    const int ldcarry = s.tiles * s.kl * s.nv * s.w;

    // the carry slots are the handle's: a merge multiply on another stream than the last one waits for that one's fix-up
    if (A->carry_done && A->carry_stream != stream)
        SPMM_CUDA(cudaStreamWaitEvent(stream, A->carry_done, 0));
    const size_t need_elems = (size_t)(2 * n_teams) * (size_t)ldcarry;
    if (A->carry_elems < need_elems)
    {
        cudaFree(A->d_carry);
        A->d_carry = nullptr;
        A->carry_elems = 0;
        SPMM_CUDA(cudaMalloc(&A->d_carry, sizeof(double) * need_elems));
        A->carry_elems = need_elems;
    }
    if (A->carry_rows < (size_t)(2 * n_teams))
    {
        cudaFree(A->d_carry_row);
        A->d_carry_row = nullptr;
        A->carry_rows = 0;
        SPMM_CUDA(cudaMalloc(&A->d_carry_row, sizeof(int) * (size_t)(2 * n_teams)));
        A->carry_rows = (size_t)(2 * n_teams);
    }

    SpmmArgs args = {};
    if (extra)
        args.extra = *extra;
    args.rowptr = A->d_rowptr;
    args.colidx = A->d_colidx;
    args.vals = A->d_vals;
    args.B = d_B;
    args.C = d_C;
    args.ldb = ldb;
    args.ldc = ldc;
    args.row_begin = row_begin;
    args.row_end = row_end;
    args.nnz_lo = (int)nnz_lo;
    args.nnz_hi = (int)nnz_hi;
    args.c_row0 = c_row0;
    args.kc = kc;
    args.items_per_team = (int)items;
    args.n_teams = (int)n_teams;
    args.carry = A->d_carry;
    args.carry_row = A->d_carry_row;
    args.ldcarry = ldcarry;
    note_kernel("spmm_merge_kernel");
    const int rc = s.w == 2 ? launch_merge_w2(s.kl, s.nv, u, args, s.tiles, stream)
                            : launch_merge_w1(s.kl, s.nv, u, args, s.tiles, stream);
    if (rc != SPMM_OK)
        return rc;
    if (!A->carry_done)
        SPMM_CUDA(cudaEventCreateWithFlags(&A->carry_done, cudaEventDisableTiming));
    SPMM_CUDA(cudaEventRecord(A->carry_done, stream));
    A->carry_stream = stream;
    return SPMM_OK;
}

} // namespace spmm
