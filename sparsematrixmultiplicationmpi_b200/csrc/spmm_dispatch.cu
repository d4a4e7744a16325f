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

// the fields every CSR kernel reads
SpmmArgs csr_args(const spmm_csr_s *A, const Request &r)
{
    SpmmArgs args = {};
    if (r.extra)
        args.extra = *r.extra;
    args.rowptr = A->d_rowptr;
    args.colidx = A->d_colidx;
    args.vals = A->d_vals;
    args.B = r.B;
    args.C = r.C;
    args.ldb = r.ldb;
    args.ldc = r.ldc;
    args.row_begin = r.row_begin;
    args.row_end = r.row_end;
    args.nnz_lo = (int)r.nnz_lo;
    args.nnz_hi = (int)r.nnz_hi;
    args.c_row0 = r.c_row0;
    args.kc = r.kc;
    return args;
}

// k range in which AUTO takes the BSR kernel on a handle with a view (DESIGN.md section 4.7, profiles/r3_bsr.md; B200,
// 1000 W): at k = 128 it beat what AUTO runs without the view on fem_blocked b = 3 (254 against 295 us), b = 6 (299 against
// 344 us) and the ten times larger b = 3 matrix (2.22 against 2.31 ms), and lost on b = 4 (292 against 248 us), where the
// tile layout applies. Below k = 64 it lost on every matrix (2-11x at k <= 8: one block row per team is too little
// parallel work per lane), and at k = 64 it lost on two of four.
bool bsr_auto_k(int k) { return k >= 128; }
} // namespace

int resolve_kernel(Form form, int kernel, int *effective)
{
    *effective = kernel;
    // The BSR kernel computes whole block rows into a C of the matrix's shape; the partial forms keep the CSR kernels.
    if (kernel == SPMM_KERNEL_BSR && form != Form::whole)
    {
        set_error("the BSR kernel serves spmm_multiply_device and spmm_multiply_strided_device only");
        return SPMM_ERR_UNSUPPORTED;
    }
    if (kernel == SPMM_KERNEL_AUTO || kernel == SPMM_KERNEL_ROWS || kernel == SPMM_KERNEL_MERGE || kernel == SPMM_KERNEL_BSR)
        return SPMM_OK;
    // the row-range and non-zero-range forms run the row kernel for every other id
    if (form == Form::rows || form == Form::nnz_range)
    {
        *effective = SPMM_KERNEL_ROWS;
        return SPMM_OK;
    }
    // the tiled kernel stages B rows by TMA boxes (not only the rows a window holds); the stream kernel writes whole rows of one C
    SPMM_REQUIRE(kernel == SPMM_KERNEL_TILED ? form != Form::window : kernel == SPMM_KERNEL_STREAM && form == Form::whole,
                 "kernel id not served by this multiply form (include/spmm_b200.h lists the ids of each)");
    return SPMM_OK;
}

// AUTO: merge-path where the schedule picked it; then, for the whole-matrix forms, the stream kernel and the BSR view; then,
// with the scatter form too, the tile layout (built lazily); else the row kernel
static int auto_kernel(spmm_csr_s *A, const Request &r)
{
    if (A->sched.auto_kernel == SPMM_KERNEL_MERGE)
        return SPMM_KERNEL_MERGE;
    // k = 1 on matrices of 4 M non-zeros and more: streamed in nnz order (3.1 against 2.4 TB/s at 10.5 M non-zeros, and
    // bit-identical to the reference); wider k / smaller matrices by spmm_tune_set("stream.kmax" / "stream.min_nnz")
    // (profiles/r1_stream.md)
    const Tuning &t = tuning();
    if (r.form == Form::whole && t.stream != 0 && r.kc <= t.stream_auto_kmax && A->nnz >= t.stream_auto_min_nnz &&
        stream_shape_ok(A, r.B, r.ldb, r.C, r.ldc, r.kc))
        return SPMM_KERNEL_STREAM;
    // a handle with a BSR view, in the k range where its kernel was measured faster; the lazy tile layout is neither
    // counted toward nor built by these launches
    if (r.form == Form::whole && A->bsr_b != 0 && bsr_auto_k(r.kc))
        return SPMM_KERNEL_BSR;
    if (r.form != Form::whole && r.form != Form::scatter)
        return SPMM_KERNEL_ROWS;
    auto_tile_layout(A, r.kc);
    return tiled_auto_ok(A, r) ? SPMM_KERNEL_TILED : SPMM_KERNEL_ROWS;
}

static const char *const STREAM_SHAPE_MSG =
    "stream kernel: k must be 1, 2, 4 or 8 (B 16-byte aligned with an even leading dimension from k = 2), rows of at most 3072 / k non-zeros";

// A handle with 64-bit row offsets: the request in each segment's own rows and non-zeros, segment after segment on `stream`.
// A row lies in one segment, so partial rows of a non-zero range keep their meaning; AUTO decides per segment. Nothing is
// launched unless every segment can serve an explicit STREAM request.
static int multiply_segments(spmm_csr_s *A, const Request &r, int kernel, cudaStream_t stream)
{
    if (kernel == SPMM_KERNEL_TILED || kernel == SPMM_KERNEL_BSR)
    {
        set_error("the tiled and BSR kernels need a layout that is not built for handles with 64-bit row offsets");
        return SPMM_ERR_UNSUPPORTED;
    }
    std::vector<std::pair<spmm_csr_s *, Request>> parts;
    for (spmm_csr_s *S : A->segs)
    {
        const int r0 = std::max(r.row_begin, S->seg_row0), r1 = std::min(r.row_end, S->seg_row0 + S->n_rows);
        if (r0 >= r1)
            continue;
        Request q = r;
        q.row_begin = r0 - S->seg_row0;
        q.row_end = r1 - S->seg_row0;
        q.nnz_lo = std::clamp(r.nnz_lo - S->seg_nnz0, 0LL, S->nnz);
        q.nnz_hi = std::clamp(r.nnz_hi - S->seg_nnz0, q.nnz_lo, S->nnz);
        q.c_row0 = q.row_begin;
        q.C = r.C + (long long)(r0 - r.c_row0) * r.ldc;
        if (kernel == SPMM_KERNEL_STREAM)
            SPMM_REQUIRE(stream_shape_ok(S, q.B, q.ldb, q.C, q.ldc, q.kc), STREAM_SHAPE_MSG);
        parts.emplace_back(S, q);
    }
    for (const auto &[S, q] : parts)
        if (int rc = multiply(S, q, kernel, stream))
            return rc;
    return SPMM_OK;
}

int multiply(spmm_csr_s *A, const Request &r, int kernel, cudaStream_t stream)
{
    SPMM_CUDA(cudaSetDevice(A->device));
    if (A->d_rowptr64)
        return multiply_segments(A, r, kernel, stream);
    // what an explicit request needs from the handle is checked at launch time
    if (kernel == SPMM_KERNEL_BSR)
        SPMM_REQUIRE(A->bsr_b != 0, "BSR kernel requested but spmm_csr_build_bsr was not called (or found no block size)");
    if (kernel == SPMM_KERNEL_STREAM)
        SPMM_REQUIRE(stream_shape_ok(A, r.B, r.ldb, r.C, r.ldc, r.kc), STREAM_SHAPE_MSG);
    if (kernel == SPMM_KERNEL_TILED)
        if (int rc = tiled_check(A, r))
            return rc;
    switch (kernel == SPMM_KERNEL_AUTO ? auto_kernel(A, r) : kernel)
    {
    case SPMM_KERNEL_MERGE: return launch_merge(A, r, stream);
    case SPMM_KERNEL_TILED: return launch_tiled(A, r, stream);
    case SPMM_KERNEL_STREAM: return launch_stream(A, r.B, r.ldb, r.C, r.ldc, r.kc, stream);
    case SPMM_KERNEL_BSR: return launch_bsr(A, r.B, r.ldb, r.C, r.ldc, r.kc, stream);
    default: return launch_rows(A, r, stream);
    }
}

int launch_rows(const spmm_csr_s *A, const Request &r, cudaStream_t stream)
{
    const Tuning &t = tuning();
    const Shape s = pick_shape(r.B, r.ldb, r.C, r.ldc, r.kc);
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
    const bool b_beyond_l2 = (long long)A->n_cols * r.kc * 8 > device_props(A->device).l2_bytes;
    int u = t.rows_unroll > 0 ? t.rows_unroll : (np >= 8 ? 1 : np >= 2 ? 2 : (s.nv >= 4 ? (b_beyond_l2 ? 4 : 2) : 4));

    SpmmArgs args = csr_args(A, r);
    // L2 prefetch only when the operands are 16-byte aligned, B is one contiguous block that starts
    // at column 0 of its rows (no k-slab), and the A arrays are the handle's own (padded) allocations
    const bool aligned = ((uintptr_t)A->d_colidx % 16 == 0) && ((uintptr_t)A->d_vals % 16 == 0) && ((uintptr_t)r.B % 16 == 0);
    args.prefetch = aligned ? (t.rows_prefetch >= 0 ? t.rows_prefetch : 3) : 0;
    // a window of B rows: nothing beyond the rows the column ids name may be touched (no prefetch of "all of B")
    args.b_bytes = (r.ldb == r.kc && r.form != Form::window) ? (long long)A->n_cols * r.ldb * 8 : 0;
    note_kernel("spmm_rows_kernel");
    return s.w == 2 ? launch_rows_w2(A, s.kl, s.nv, np, u, args, s.tiles, A->device, stream)
                    : launch_rows_w1(A, s.kl, s.nv, np, u, args, s.tiles, A->device, stream);
}

int launch_merge(spmm_csr_s *A, const Request &r, cudaStream_t stream)
{
    const Tuning &t = tuning();
    Shape s = pick_shape(r.B, r.ldb, r.C, r.ldc, r.kc);
    // Team shape: pick_shape's (8 lanes x 2 accesses at k = 32). Measured on cfg3 (R-MAT 2^22, k = 32) after the kernel was
    // rebuilt around batches of KL non-zeros (coalesced id/value loads one batch ahead, B rows gathered 4 at a time whatever
    // rows they belong to): 8 x 2 unroll 4 at 80 registers 2.17 ms, 16 x 1 2.34 ms, unroll 8 (127 registers) 4.5 ms
    // (gpurun_out/s5_tune_mb1.jsonl); the row-by-row kernel before it took 3.06-3.50 ms.
    const int u = t.rows_unroll > 0 ? t.rows_unroll : (s.nv >= 4 ? 2 : 4);
    const long long total = (long long)(r.row_end - r.row_begin) + (r.nnz_hi - r.nnz_lo);
    long long items = t.merge_items > 0 ? t.merge_items : 512;
    // enough teams to fill the machine, few enough that the carry rows stay a small fraction of C
    // (a shard of long rows — the first non-zero range of an R-MAT matrix averages 477 per row — is cut less finely: every
    // team inside a row leaves a carry slot and the fix-up walks them in order; measured per range in gpurun_out/s28_*)
    const double avg_row = (double)(r.nnz_hi - r.nnz_lo) / std::max(1, r.row_end - r.row_begin);
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

    SpmmArgs args = csr_args(A, r);
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
