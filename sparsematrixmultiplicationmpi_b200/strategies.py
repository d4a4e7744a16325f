"""The reference's three MPI decompositions as one-process-per-GPU partitions over torch.distributed.

  RowWise          rows of A / C in contiguous blocks        RowWise.cpp:12-126
                   B replicated by broadcast, C gathered      (NCCL broadcast / gather)
  ColumnBlocks     column blocks of A with the matching row   BASELINE.json north_star reading of
                   slab of B; full-size partial C summed by   ColumnWise.cpp:13-131 (SURVEY.md F2)
                   reduce-scatter
  ColumnSlabs      the reference's own reading: B's k columns ColumnWise.cpp:25-48,82-84
                   split across ranks, slabs gathered
  NonZeroRanges    equal ranges of the non-zero stream;       NonZeroElement.cpp:12-120
                   only rows cut by a range boundary are
                   exchanged, peer to peer, and summed in
                   rank order (no dense reduce)

Every class works on torch tensors living on the device of its `compute` engine. `CudaCompute`
(the product) runs the sm_100a kernels through the C-ABI; the CPU tests inject their own engine
on gloo to exercise the partition / exchange logic. There is no CPU engine in the package.

rank/size come from torch.distributed when it is initialised (one process per GPU, launched by
torchrun), else the single-rank degenerate case — exactly how the reference's code behaves at
mpirun -np 1.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

from . import _cabi
from .matrix import DeviceCSR, SparseMatrix


def world(group=None) -> tuple[int, int]:
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def partition_rows(n_rows: int, P: int, r: int) -> tuple[int, int]:
    """RowWise.cpp:26-29: base = N/P, the first N%P ranks take one more row."""
    base, extra = divmod(n_rows, P)
    s = r * base + min(r, extra)
    return s, s + base + (1 if r < extra else 0)


def partition_cols(k: int, P: int, r: int) -> tuple[int, int]:
    """ColumnWise.cpp:25-28: k/P each, the LAST rank also takes all k%P extras."""
    base, extra = divmod(k, P)
    s = r * base
    return s, s + base + (extra if r == P - 1 else 0)


def partition_nnz(nnz: int, P: int, r: int) -> tuple[int, int]:
    """NonZeroElement.cpp:24-39: the first nnz%P ranks take one more element."""
    per, extra = divmod(nnz, P)
    if r < extra:
        s = r * (per + 1)
        return s, s + per + 1
    s = r * per + extra
    return s, s + per


class CudaCompute:
    """Engine of the product path: CSR shards in HBM, multiply through libspmm_b200.so."""

    def __init__(self, device: int | None = None, kernel: str = "auto"):
        if not torch.cuda.is_available():
            raise RuntimeError("sparsematrixmultiplicationmpi_b200 needs a CUDA device (no CPU fallback)")
        _cabi.lib()  # fail loudly if the extension is not built
        self.index = torch.cuda.current_device() if device is None else device
        self.device = torch.device("cuda", self.index)
        self.kernel = kernel

    def upload(self, m: SparseMatrix) -> DeviceCSR:
        return DeviceCSR.from_host(m, self.index)

    def update_values(self, A: DeviceCSR, values: np.ndarray) -> None:
        """New values (host, CSR order) for a shard made by upload(): its schedule and tile layout are kept."""
        A.update_values(values)

    def multiply(self, A: DeviceCSR, B: torch.Tensor, k: int, out: torch.Tensor | None = None) -> torch.Tensor:
        """out[n_rows, k] = A * B[n_cols, k]; contiguous float64 tensors on self.device."""
        assert B.is_cuda and B.dtype == torch.float64 and B.is_contiguous()
        if out is None:
            out = torch.empty((A.n_rows, k), dtype=torch.float64, device=self.device)
        if A.n_rows and k:
            A.multiply(B.data_ptr(), k, out.data_ptr(), self.kernel, torch.cuda.current_stream(self.device).cuda_stream)
        return out

    def column_span(self, A: DeviceCSR) -> tuple[int, int]:
        return A.column_span()

    def multiply_window(self, A: DeviceCSR, window: torch.Tensor, first_row: int, k: int,
                        out: torch.Tensor | None = None) -> torch.Tensor:
        """out = A * B where only the rows [first_row, first_row + len(window)) of B are resident (the block's halo window)."""
        if out is None:
            out = torch.empty((A.n_rows, k), dtype=torch.float64, device=self.device)
        if A.n_rows and k:
            A.multiply_window(window.data_ptr(), first_row, window.shape[0], k, out.data_ptr(),
                              self.kernel if self.kernel in ("auto", "rows", "merge") else "auto",
                              torch.cuda.current_stream(self.device).cuda_stream)
        return out

    def multiply_rows(self, A: DeviceCSR, row_begin: int, row_end: int, B: torch.Tensor, k: int, out: torch.Tensor):
        """out[row_end-row_begin, k] = A[row_begin:row_end, :] * B (a row block of the shard, RowWise.cpp:36-50)."""
        if row_end > row_begin and k:
            A.multiply_rows(row_begin, row_end, B.data_ptr(), k, out.data_ptr(), self.kernel,
                            torch.cuda.current_stream(self.device).cuda_stream)
        return out

    def multiply_slab(self, A: DeviceCSR, B: torch.Tensor, k: int, k_begin: int, k_count: int, out: torch.Tensor):
        """Columns [k_begin, k_begin+k_count) of out = A * B, both with leading dimension k."""
        if A.n_rows and k_count:
            A.multiply_strided(B.data_ptr(), k, out.data_ptr(), k, k_begin, k_count, self.kernel,
                               torch.cuda.current_stream(self.device).cuda_stream)
        return out


def _built_from(plan, m: SparseMatrix):
    """Record the size of the matrix a plan was made from (from_host), for update_values."""
    plan._source = (m.numRows, m.numCols, m.nnz)
    return plan


def _check_same_size(plan, m: SparseMatrix) -> None:
    src = getattr(plan, "_source", None)
    if src is None:
        raise ValueError("update_values needs a plan made by from_host")
    if (m.numRows, m.numCols, m.nnz) != src:
        raise ValueError(f"update_values: matrix is {m.numRows} x {m.numCols} with {m.nnz} non-zeros, "
                         f"the plan was made from {src[0]} x {src[1]} with {src[2]}")


def _gather_rows_to_root(local: torch.Tensor, counts: list[int], k: int, group=None) -> torch.Tensor | None:
    """Gatherv of row blocks to rank 0 (RowWise.cpp:85-87): equal-size padded blocks, trimmed at the root."""
    rank, P = world(group)
    if P == 1:
        return local
    pad_rows = max(counts)
    send = local
    if local.shape[0] != pad_rows:
        send = torch.zeros((pad_rows, k), dtype=local.dtype, device=local.device)
        send[:local.shape[0]] = local
    if rank == 0:
        recv = [torch.empty((pad_rows, k), dtype=local.dtype, device=local.device) for _ in range(P)]
        dist.gather(send, recv, dst=0, group=group)
        return torch.cat([recv[r][:counts[r]] for r in range(P)], dim=0)
    dist.gather(send, None, dst=0, group=group)
    return None


class RowWise:
    """Rank r owns rows [start,end) of A (RowWise.cpp:26-29) and the same rows of C."""

    def __init__(self, compute, n_rows: int, k: int, local_A, group=None):
        self.compute, self.n_rows, self.k, self.A, self.group = compute, n_rows, k, local_A, group
        self.rank, self.P = world(group)
        self.start, self.end = partition_rows(n_rows, self.P, self.rank)
        self.counts = [partition_rows(n_rows, self.P, r)[1] - partition_rows(n_rows, self.P, r)[0]
                       for r in range(self.P)]
        assert local_A.n_rows == self.end - self.start

    @classmethod
    def from_host(cls, compute, m: SparseMatrix, k: int, group=None) -> "RowWise":
        rank, P = world(group)
        s, e = partition_rows(m.numRows, P, rank)
        return _built_from(cls(compute, m.numRows, k, compute.upload(m.row_block(s, e)), group), m)

    def update_values(self, m: SparseMatrix) -> None:
        """New values of the matrix from_host was given: same pattern (the caller's promise, not checked), same size
        (checked). Every rank refreshes its block in place, schedule and tile layout kept; no collective, since every rank
        holds the whole host matrix (as main.cpp leaves it)."""
        _check_same_size(self, m)
        self.compute.update_values(self.A, m.values[m.rowPtr[self.start]:m.rowPtr[self.end]])

    def broadcast_B(self, B: torch.Tensor) -> torch.Tensor:
        """B replicated from rank 0 (main.cpp:137 does this with MPI_Bcast, outside the timed region)."""
        if self.P > 1:
            dist.broadcast(B, src=0, group=self.group)
        return B

    def multiply_local(self, B: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        return self.compute.multiply(self.A, B, self.k, out)

    def gather(self, C_local: torch.Tensor) -> torch.Tensor | None:
        return _gather_rows_to_root(C_local, self.counts, self.k, self.group)

    def all_gather(self, C_local: torch.Tensor) -> torch.Tensor:
        """Full C on every rank (what an iterative caller needs as the next B)."""
        if self.P == 1:
            return C_local
        pad = max(self.counts)
        send = C_local
        if C_local.shape[0] != pad:
            send = torch.zeros((pad, self.k), dtype=C_local.dtype, device=C_local.device)
            send[:C_local.shape[0]] = C_local
        recv = torch.empty((self.P * pad, self.k), dtype=C_local.dtype, device=C_local.device)
        dist.all_gather_into_tensor(recv, send, group=self.group)
        if all(c == pad for c in self.counts):
            return recv
        return torch.cat([recv[r * pad:r * pad + self.counts[r]] for r in range(self.P)], dim=0)

    def run(self, B: torch.Tensor) -> torch.Tensor | None:
        """The reference call: local rows, then Gatherv to rank 0; None on the other ranks."""
        return self.gather(self.multiply_local(B))

    # ---- B row-sharded like C: only the rows of B a block's columns name cross the links (halo exchange) ----
    # The reference replicates all of B on every rank (main.cpp:137); its row loop reads fatVector[colIndices[j]] only
    # (RowWise.cpp:36-50). With B sharded by rows the way C is (rank q owns B[bs_q:be_q], what an iterative caller has
    # after a multiply), a banded block needs its own rows plus a halo of half a bandwidth from its neighbours —
    # kilobytes over NVLink instead of a broadcast of the whole fat vector.
    def halo_plan(self):
        """Column span [lo, hi] of every rank's block (exchanged once) and the B rows every rank owns."""
        if getattr(self, "_halo", None) is None:
            n_cols = self.A.n_cols
            lo, hi = self.compute.column_span(self.A)
            spans = [(lo, hi)]
            if self.P > 1:
                spans = [None] * self.P
                dist.all_gather_object(spans, (lo, hi), group=self.group)
            owners = [partition_rows(n_cols, self.P, q) for q in range(self.P)]
            self._halo = (spans, owners)
        return self._halo

    def window_range(self) -> tuple[int, int]:
        """Rows [w0, w1) of B this rank keeps resident: the rows its block reads and the rows it owns."""
        spans, owners = self.halo_plan()
        lo, hi = spans[self.rank]
        bs, be = owners[self.rank]
        if hi < lo:
            return bs, be
        return min(lo, bs), max(hi + 1, be)

    def alloc_window(self, device=None, dtype=torch.float64) -> tuple[torch.Tensor, torch.Tensor]:
        """(window, own): one buffer for the rows window_range() of B and the view of the rows this rank owns. A caller
        that produces its share of B straight into `own` (e.g. the C of the previous multiply) exchanges halos in place:
        nothing but the halo rows is ever copied."""
        w0, w1 = self.window_range()
        bs, be = self.halo_plan()[1][self.rank]
        window = torch.empty((w1 - w0, self.k), dtype=dtype, device=device if device is not None else self.compute.device)
        return window, window[bs - w0:be - w0]

    def exchange_halo_inplace(self, window: torch.Tensor) -> int:
        """Fill the halo rows of `window` (allocated by alloc_window, own rows already in place) from their owners, peer to
        peer; returns the first row of the window."""
        spans, owners = self.halo_plan()
        w0, w1 = self.window_range()
        lo, hi = spans[self.rank]
        bs, be = owners[self.rank]
        ops = []
        for q in range(self.P):
            if q == self.rank:
                continue
            qs, qe = owners[q]
            a, b = max(lo, qs), min(hi + 1, qe)  # rows I read that q owns
            if b > a:
                ops.append(dist.P2POp(dist.irecv, window[a - w0:b - w0], q, group=self.group))
            qlo, qhi = spans[q]
            a, b = max(qlo, bs), min(qhi + 1, be)  # rows q reads that I own
            if b > a:
                ops.append(dist.P2POp(dist.isend, window[a - w0:b - w0], q, group=self.group))
        if ops:
            for w in dist.batch_isend_irecv(ops):
                w.wait()
        return w0

    def exchange_halo(self, B_own: torch.Tensor) -> tuple[torch.Tensor, int]:
        """B_own = this rank's rows of B (any buffer). Returns (window, first_row): the rows of B this rank's block reads,
        its own part copied in, the rest received peer to peer from their owners. (alloc_window + exchange_halo_inplace
        avoid the local copy.)"""
        window, own = self.alloc_window(B_own.device, B_own.dtype)
        assert B_own.shape[0] == own.shape[0]
        own.copy_(B_own)
        return window, self.exchange_halo_inplace(window)

    def multiply_sharded(self, B_own: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        """C[start:end] from B sharded by rows: halo exchange, then the block multiply on the window."""
        window, first = self.exchange_halo(B_own)
        return self.compute.multiply_window(self.A, window, first, self.k, out)

    # ---- gather fused into the multiply: C rows stored straight into the peers' buffers over NVLink ----
    def _symmetric_C(self, device: torch.device):
        """One (n_rows x k) result buffer per rank, mapped into every rank (torch symmetric memory = CUDA IPC /
        fabric handles over NVLink); cached on the plan."""
        if getattr(self, "_symm", None) is None:
            import torch.distributed._symmetric_memory as symm_mem
            group = self.group if self.group is not None else dist.group.WORLD
            buf = symm_mem.empty((self.n_rows, self.k), dtype=torch.float64, device=device)
            hdl = symm_mem.rendezvous(buf, group)
            self._symm = (buf, hdl)
        return self._symm

    def _scatter(self, B: torch.Tensor, peers: list[int]) -> torch.Tensor:
        buf, hdl = self._symmetric_C(B.device)
        off = self.start * self.k * 8  # this rank's rows start here in every copy of C
        ptrs = [int(hdl.buffer_ptrs[p]) + off for p in peers]
        lo, hi = buf.data_ptr(), buf.data_ptr() + buf.numel() * 8
        if B.data_ptr() < hi and B.data_ptr() + B.numel() * 8 > lo:
            # the previous result fed back as B (an iterative caller): peers would overwrite rows this rank still reads
            B = B.clone()
        # a fast rank must not store into a peer's copy while that peer still reads the previous result
        hdl.barrier(channel=0)
        if self.end > self.start and self.k:
            self.A.multiply_scatter(B.data_ptr(), self.k, ptrs, self.compute.kernel,
                                    torch.cuda.current_stream(B.device).cuda_stream)
        hdl.barrier(channel=0)  # every rank's stores have landed before anybody reads its copy
        return buf

    def multiply_all_gather_p2p(self, B: torch.Tensor) -> torch.Tensor:
        """Full C on every rank without a collective: the multiply kernel stores each finished row piece from
        registers to all P copies of C (its own first, then the peers in ring order so that the NVLink ports
        are used evenly). The returned tensor is the plan's symmetric buffer: it is overwritten by the next call."""
        if self.P == 1:
            return self.multiply_local(B)
        if self.P > 8:
            return self.all_gather(self.multiply_local(B))
        return self._scatter(B, [(self.rank + i) % self.P for i in range(self.P)])

    def run_p2p(self, B: torch.Tensor) -> torch.Tensor | None:
        """The reference call (result on rank 0 only, RowWise.cpp:85-87) with the Gatherv fused into the multiply:
        every rank stores its rows directly into rank 0's buffer."""
        if self.P == 1:
            return self.multiply_local(B)
        buf = self._scatter(B, [0])
        return buf if self.rank == 0 else None

    def multiply_all_gather_overlapped(self, B: torch.Tensor, chunks: int = 4) -> torch.Tensor:
        """Full C on every rank with the gather of row chunk c running over NVLink while chunk c+1 is
        being multiplied: the local rows are cut into `chunks` pieces, each computed straight into its
        slot of a chunk-major send buffer and all-gathered asynchronously as soon as it is ready.
        Needs equal row counts on every rank (pad the matrix otherwise); falls back to all_gather()."""
        if self.P == 1 or len(set(self.counts)) != 1 or chunks <= 1:
            return self.all_gather(self.multiply_local(B))
        rows = self.counts[0]
        cb = -(-rows // chunks)
        out = torch.empty((self.n_rows, self.k), dtype=torch.float64, device=B.device)
        works = []
        stage = []
        for c in range(chunks):
            r0, r1 = min(rows, c * cb), min(rows, (c + 1) * cb)
            if r1 <= r0:
                break
            send = torch.empty((r1 - r0, self.k), dtype=torch.float64, device=B.device)
            self.compute.multiply_rows(self.A, r0, r1, B, self.k, send)
            recv = torch.empty((self.P * (r1 - r0), self.k), dtype=torch.float64, device=B.device)
            works.append(dist.all_gather_into_tensor(recv, send, group=self.group, async_op=True))
            stage.append((r0, r1, recv, send))
        for w in works:
            w.wait()
        view = out.view(self.P, rows, self.k)
        for r0, r1, recv, _ in stage:  # chunk-major -> row-major: one strided copy per chunk
            view[:, r0:r1].copy_(recv.view(self.P, r1 - r0, self.k))
        return out


class ColumnBlocks:
    """Rank r owns columns J_r of A (contiguous, RowWise-style split of numCols) and rows J_r of B.

    Each rank produces a full-size partial C; reduce-scatter(sum) leaves rank r with rows R_r of
    C (contiguous blocks of ceil(N/P) rows, zero padded at the end).
    """

    def __init__(self, compute, n_rows: int, n_cols: int, k: int, local_A, group=None):
        self.compute, self.n_rows, self.n_cols, self.k, self.A, self.group = compute, n_rows, n_cols, k, local_A, group
        self.rank, self.P = world(group)
        self.col_start, self.col_end = partition_rows(n_cols, self.P, self.rank)
        self.block = -(-n_rows // self.P)  # rows of C per rank after the reduce-scatter
        assert local_A.n_rows == n_rows and local_A.n_cols == self.col_end - self.col_start

    @classmethod
    def from_host(cls, compute, m: SparseMatrix, k: int, group=None) -> "ColumnBlocks":
        rank, P = world(group)
        c0, c1 = partition_rows(m.numCols, P, rank)
        keep = (m.colIndices >= c0) & (m.colIndices < c1)
        csum = np.concatenate(([0], np.cumsum(keep, dtype=np.int64)))
        local = SparseMatrix(m.values[keep], m.colIndices[keep] - c0, csum[m.rowPtr].astype(np.int32), m.numRows, c1 - c0)
        return _built_from(cls(compute, m.numRows, m.numCols, k, compute.upload(local), group), m)

    def update_values(self, m: SparseMatrix) -> None:
        """New values of the matrix from_host was given (same pattern, not checked; same size, checked): this rank's column
        block takes the values of its columns, cut from the host matrix as from_host cut them."""
        _check_same_size(self, m)
        keep = (m.colIndices >= self.col_start) & (m.colIndices < self.col_end)
        self.compute.update_values(self.A, m.values[keep])

    def local_B(self, B_full: torch.Tensor) -> torch.Tensor:
        return B_full[self.col_start:self.col_end].contiguous()

    def multiply_local(self, B_local: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        """Partial C, (P*block) x k with the rows past n_rows zero."""
        rows_pad = self.block * self.P
        if out is None:
            out = torch.empty((rows_pad, self.k), dtype=torch.float64, device=B_local.device)
        if rows_pad > self.n_rows:
            out[self.n_rows:].zero_()
        self.compute.multiply(self.A, B_local, self.k, out[:self.n_rows])
        return out

    def reduce_scatter(self, partial: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        if out is None:
            out = torch.empty((self.block, self.k), dtype=partial.dtype, device=partial.device)
        if self.P == 1:
            out.copy_(partial[:self.block])
            return out
        dist.reduce_scatter_tensor(out, partial, op=dist.ReduceOp.SUM, group=self.group)
        return out

    def multiply_reduce_scatter_p2p(self, B_local: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        """This rank's block of C without NCCL: every rank multiplies into a partial C that lives in symmetric memory
        (mapped into all ranks over NVLink), then reads block `rank` of every peer's partial with P2P loads and adds
        them in ascending rank order (spmm_reduce_blocks_device) — deterministic, the oracle's order."""
        if self.P == 1 or self.P > 8 or (self.block * self.k) % 2:
            return self.reduce_scatter(self.multiply_local(B_local), out)
        if getattr(self, "_symm", None) is None:
            import torch.distributed._symmetric_memory as symm_mem
            group = self.group if self.group is not None else dist.group.WORLD
            buf = symm_mem.empty((self.block * self.P, self.k), dtype=torch.float64, device=B_local.device)
            self._symm = (buf, symm_mem.rendezvous(buf, group))
        partial, hdl = self._symm
        if out is None:
            out = torch.empty((self.block, self.k), dtype=torch.float64, device=B_local.device)
        hdl.barrier(channel=0)  # nobody still reads the partial of the previous call
        self.multiply_local(B_local, partial)
        hdl.barrier(channel=0)  # every partial is complete
        off = self.rank * self.block * self.k * 8
        _cabi.reduce_blocks(B_local.device.index, [int(hdl.buffer_ptrs[p]) + off for p in range(self.P)],
                            self.block * self.k, out.data_ptr(), torch.cuda.current_stream(B_local.device).cuda_stream)
        return out

    def multiply_reduce_scatter_push(self, B_local: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        """This rank's block of C with the exchange fused into the multiply: the partial of row block o is not written to
        local memory and reduce-scattered afterwards, it is STORED BY THE SPMM KERNEL straight into slot `rank` of a
        staging buffer on rank o (symmetric memory, peer stores over NVLink / NVSwitch), one launch per destination in
        ring order (rank p starts with block p+1, so every GPU receives from one sender at a time). After one barrier each
        rank adds its P local slots in ascending rank order (spmm_reduce_blocks_device on local pointers): the same
        deterministic sum as the pull variant, with the NVLink traffic overlapped by the arithmetic of the next block and
        no partial C written to and read back from HBM (replaces the collective of ColumnWise.cpp:82-84)."""
        if self.P > 1 and not B_local.is_cuda:
            return self._push_host(B_local, out)
        if self.P == 1 or self.P > 8 or (self.block * self.k) % 2:
            return self.reduce_scatter(self.multiply_local(B_local), out)
        if getattr(self, "_symm_push", None) is None:
            import torch.distributed._symmetric_memory as symm_mem
            group = self.group if self.group is not None else dist.group.WORLD
            buf = symm_mem.empty((self.P, self.block, self.k), dtype=torch.float64, device=B_local.device)
            buf.zero_()  # (rows past n_rows in the last block are never written: they stay zero)
            self._symm_push = (buf, symm_mem.rendezvous(buf, group))
        slots, hdl = self._symm_push
        if out is None:
            out = torch.empty((self.block, self.k), dtype=torch.float64, device=B_local.device)
        stream = torch.cuda.current_stream(B_local.device).cuda_stream
        slot_bytes = self.block * self.k * 8
        hdl.barrier(channel=0)  # nobody still adds up the slots of the previous call
        for step in range(self.P):
            o = (self.rank + 1 + step) % self.P  # the own block last: its stores are local
            r0, r1 = min(self.n_rows, o * self.block), min(self.n_rows, (o + 1) * self.block)
            if r1 > r0:
                self.A.multiply_rows(r0, r1, B_local.data_ptr(), self.k, int(hdl.buffer_ptrs[o]) + self.rank * slot_bytes, "auto", stream)
        hdl.barrier(channel=0)  # every sender's rows have landed in this rank's slots
        base = slots.data_ptr()
        _cabi.reduce_blocks(B_local.device.index, [base + q * slot_bytes for q in range(self.P)], self.block * self.k,
                            out.data_ptr(), stream)
        return out

    def _push_host(self, B_local: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        """The data flow of multiply_reduce_scatter_push on host tensors (gloo): row block o of this rank's partial goes to
        slot `rank` on rank o (send / receive instead of peer stores), the slots are added in ascending rank order."""
        slots = torch.zeros((self.P, self.block, self.k), dtype=torch.float64)
        ops, keep = [], []
        for step in range(self.P):
            o = (self.rank + 1 + step) % self.P
            r0, r1 = min(self.n_rows, o * self.block), min(self.n_rows, (o + 1) * self.block)
            part = slots[self.rank] if o == self.rank else torch.zeros((self.block, self.k), dtype=torch.float64)
            if r1 > r0:
                self.compute.multiply_rows(self.A, r0, r1, B_local, self.k, part[:r1 - r0])
            if o != self.rank:
                keep.append(part)
                ops.append(dist.P2POp(dist.isend, part, o, group=self.group))
        for q in range(self.P):
            if q != self.rank:
                ops.append(dist.P2POp(dist.irecv, slots[q], q, group=self.group))
        for req in dist.batch_isend_irecv(ops):
            req.wait()
        if out is None:
            out = torch.empty((self.block, self.k), dtype=torch.float64)
        out.copy_(slots[0])
        for q in range(1, self.P):
            out += slots[q]
        return out

    def multiply_reduce_scatter_overlapped(self, B_local: torch.Tensor, chunks: int = 4) -> torch.Tensor:
        """Same result as reduce_scatter(multiply_local(B)) — this rank's block of C — but the partial
        C is produced in reduce-scatter chunk order: for chunk c the rows c*cb..(c+1)*cb of EVERY rank's
        block are multiplied into one contiguous (P x cb x k) buffer, whose reduce-scatter over NVLink
        is started asynchronously while chunk c+1 is being multiplied."""
        if self.P == 1 or chunks <= 1:
            return self.reduce_scatter(self.multiply_local(B_local))
        cb = -(-self.block // chunks)
        out = torch.empty((self.block, self.k), dtype=torch.float64, device=B_local.device)
        works, keep = [], []
        for c in range(chunks):
            b0, b1 = min(self.block, c * cb), min(self.block, (c + 1) * cb)
            if b1 <= b0:
                break
            part = torch.empty((self.P, b1 - b0, self.k), dtype=torch.float64, device=B_local.device)
            for p in range(self.P):
                r0, r1 = min(self.n_rows, p * self.block + b0), min(self.n_rows, p * self.block + b1)
                if r1 - r0 < b1 - b0:
                    part[p, max(0, r1 - r0):].zero_()
                self.compute.multiply_rows(self.A, r0, r1, B_local, self.k, part[p, :max(0, r1 - r0)])
            works.append(dist.reduce_scatter_tensor(out[b0:b1], part.view(-1, self.k), op=dist.ReduceOp.SUM,
                                                    group=self.group, async_op=True))
            keep.append(part)
        for w in works:
            w.wait()
        return out

    def run(self, B_local: torch.Tensor) -> torch.Tensor | None:
        mine = self.reduce_scatter(self.multiply_local(B_local))
        counts = [max(0, min(self.block, self.n_rows - r * self.block)) for r in range(self.P)]
        return _gather_rows_to_root(mine[:counts[self.rank]], counts, self.k, self.group)


class ColumnSlabs:
    """The reference's own column-wise strategy: rank r computes columns [s,e) of C (ColumnWise.cpp:25-48)."""

    def __init__(self, compute, k: int, A, group=None):
        self.compute, self.k, self.A, self.group = compute, k, A, group
        self.rank, self.P = world(group)
        self.k_start, self.k_end = partition_cols(k, self.P, self.rank)

    @classmethod
    def from_host(cls, compute, m: SparseMatrix, k: int, group=None) -> "ColumnSlabs":
        return _built_from(cls(compute, k, compute.upload(m), group), m)

    def update_values(self, m: SparseMatrix) -> None:
        """New values of the matrix from_host was given (same pattern, not checked; same size, checked): every rank holds
        the whole matrix and takes all of them."""
        _check_same_size(self, m)
        self.compute.update_values(self.A, m.values)

    def run(self, B: torch.Tensor) -> torch.Tensor | None:
        n = self.A.n_rows
        Cw = torch.zeros((n, self.k), dtype=torch.float64, device=B.device)
        self.compute.multiply_slab(self.A, B, self.k, self.k_start, self.k_end - self.k_start, Cw)
        if self.P == 1:
            return Cw
        # slab gather (ColumnWise.cpp:82-84) + root interleave (:109-126): slabs are disjoint column
        # ranges of zero-initialised buffers, so a sum to the root is exactly the interleave.
        dist.reduce(Cw, dst=0, op=dist.ReduceOp.SUM, group=self.group)
        return Cw if self.rank == 0 else None


class NonZeroRanges:
    """Rank r owns elements [begin,end) of the non-zero stream (NonZeroElement.cpp:24-39).

    Its shard is the CSR of the rows first_row..last_row clipped to that range, so the local
    multiply yields complete rows inside the range and PARTIAL rows at its two ends. A row cut by
    one or more range boundaries is owned by the lowest rank that holds a piece of it; the other
    holders send their k-double partial to the owner, which adds them in rank order.
    """

    def __init__(self, compute, n_rows: int, k: int, local_A, first_row: int, last_row: int, starts_mid_row: bool,
                 group=None):
        self.compute, self.n_rows, self.k, self.A, self.group = compute, n_rows, k, local_A, group
        self.rank, self.P = world(group)
        self.first_row, self.last_row = first_row, last_row
        meta = [first_row, last_row, int(starts_mid_row)]
        if self.P > 1:
            allm = [None] * self.P
            dist.all_gather_object(allm, meta, group=self.group)
        else:
            allm = [meta]
        self.meta = allm
        # owner[r] = rank that owns rank r's first row; ranks with an empty range have last < first
        self.owner_of_first = []
        for r, (f, l, mid) in enumerate(allm):
            o = r
            if l >= f and mid:
                o = r - 1
                while o > 0 and (allm[o][1] < allm[o][0] or (allm[o][0] == f and allm[o][2])):
                    o -= 1
            self.owner_of_first.append(o)

    @staticmethod
    def shard_of(m: SparseMatrix, P: int, r: int):
        """(local SparseMatrix, first_row, last_row, starts_mid_row) of rank r's non-zero range."""
        b, e = partition_nnz(m.nnz, P, r)
        if e <= b:
            return SparseMatrix(np.empty(0), np.empty(0, np.int32), np.zeros(1, np.int32), 0, m.numCols), 0, -1, False
        rp = m.rowPtr.astype(np.int64)
        first = int(np.searchsorted(rp, b, side="right") - 1)
        last = int(np.searchsorted(rp, e - 1, side="right") - 1)
        local_rp = (np.clip(rp[first:last + 2], b, e) - b).astype(np.int32)
        local = SparseMatrix(m.values[b:e], m.colIndices[b:e], local_rp, last - first + 1, m.numCols)
        return local, first, last, bool(b > rp[first])

    @classmethod
    def from_host(cls, compute, m: SparseMatrix, k: int, group=None) -> "NonZeroRanges":
        rank, P = world(group)
        local, first, last, mid = cls.shard_of(m, P, rank)
        return _built_from(cls(compute, m.numRows, k, compute.upload(local), first, last, mid, group), m)

    def update_values(self, m: SparseMatrix) -> None:
        """New values of the matrix from_host was given (same pattern, not checked; same size, checked): this rank's range
        of the non-zero stream, the elements from_host gave it."""
        _check_same_size(self, m)
        b, e = partition_nnz(m.nnz, self.P, self.rank)
        self.compute.update_values(self.A, m.values[b:e])

    def multiply_local(self, B: torch.Tensor) -> torch.Tensor:
        return self.compute.multiply(self.A, B, self.k)

    def fix_boundaries(self, C_local: torch.Tensor) -> torch.Tensor:
        """Peer-to-peer exchange of the cut rows; afterwards every rank holds complete values for the rows it owns."""
        if self.P == 1:
            return C_local
        ops, recv_bufs = [], []
        me = self.rank
        if self.meta[me][1] >= self.meta[me][0] and self.owner_of_first[me] != me:
            ops.append(dist.P2POp(dist.isend, C_local[0].contiguous(), self.owner_of_first[me], group=self.group))
        for r in range(me + 1, self.P):
            if self.meta[r][1] >= self.meta[r][0] and self.owner_of_first[r] == me:
                buf = torch.empty(self.k, dtype=C_local.dtype, device=C_local.device)
                recv_bufs.append((r, buf))
                ops.append(dist.P2POp(dist.irecv, buf, r, group=self.group))
        if ops:
            for w in dist.batch_isend_irecv(ops):
                w.wait()
        for r, buf in recv_bufs:  # ascending rank order: deterministic sum
            C_local[self.meta[r][0] - self.first_row] += buf
        return C_local

    def owned_rows(self) -> tuple[int, int]:
        f, l, _ = self.meta[self.rank]
        if l < f:
            return 0, 0
        return (f + 1, l + 1) if self.owner_of_first[self.rank] != self.rank else (f, l + 1)

    def run(self, B: torch.Tensor) -> torch.Tensor | None:
        C_local = self.fix_boundaries(self.multiply_local(B))
        lo, hi = self.owned_rows()
        mine = C_local[lo - self.first_row:hi - self.first_row] if hi > lo else C_local[:0]
        if self.P == 1:
            out = torch.zeros((self.n_rows, self.k), dtype=torch.float64, device=B.device)
            out[lo:hi] = mine
            return out
        # owned blocks are disjoint row ranges; rows nobody owns are empty rows (zero)
        spans = []
        for r in range(self.P):
            f, l, _ = self.meta[r]
            spans.append((0, 0) if l < f else ((f + 1, l + 1) if self.owner_of_first[r] != r else (f, l + 1)))
        if self.rank == 0:
            out = torch.zeros((self.n_rows, self.k), dtype=torch.float64, device=B.device)
            out[lo:hi] = mine
            ops = [dist.P2POp(dist.irecv, out[a:b], r, group=self.group) for r, (a, b) in enumerate(spans) if r and b > a]
            if ops:
                for w in dist.batch_isend_irecv(ops):
                    w.wait()
            return out
        if hi > lo:
            for w in dist.batch_isend_irecv([dist.P2POp(dist.isend, mine.contiguous(), 0, group=self.group)]):
                w.wait()
        return None
