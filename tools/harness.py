#!/usr/bin/env python
"""Benchmark harness of the SpMM path (north_star item 4): every BASELINE.json config on the GPUs
of one box, GFLOP/s = 2*nnz*k/t and achieved fraction of the HBM roofline (algorithmic bytes =
nnz*12 + (N+1)*4 + 2*N*k*8 per GPU shard), CUDA-event timing over rotating operand sets (cold
L2), beside the reference's CPU code where it fits in a bounded time.

    python tools/harness.py --configs cfg2 --variants           # kernel-variant sweep on cfg2
    python tools/harness.py --configs cfg1,cfg2,cfg3,cfg4,cfg5   # single GPU
    torchrun --nproc-per-node 8 tools/harness.py --configs cfg3,cfg4,cfg5   # row / column / nnz partitions

Writes JSON lines to --out (default gpurun_out/harness.jsonl) and a readable table to stdout.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import sparsematrixmultiplicationmpi_b200 as spmm  # noqa: E402
from sparsematrixmultiplicationmpi_b200 import _cabi, generators as gen  # noqa: E402

L2_BYTES = 126e6
ONLY = ""


def peak_gbs():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        return 6650.0


def abytes(n_rows, nnz, k, b_rows=None):
    return nnz * 12 + (n_rows + 1) * 4 + ((b_rows if b_rows is not None else n_rows) + n_rows) * k * 8


def time_launches(fn, iters, warmup=5):
    """Mean device time per call in ms (CUDA events on the current stream)."""
    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        fn(i)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def operand_sets(make_A, n_cols, n_rows, k, dev, footprint):
    """Enough rotating copies of (A, B, C) that a step never finds its operands in L2 (>= 3 x L2 in flight)."""
    copies = max(1, min(6, int(np.ceil(3 * L2_BYTES / max(footprint, 1)))))
    sets = []
    for s in range(copies):
        A = make_A(s)
        B = torch.randint(1, 101, (n_cols, k), device=dev).double()
        C = torch.empty((n_rows, k), dtype=torch.float64, device=dev)
        sets.append((A, B, C))
    return sets


def run_variants(name, sets, k, variants, iters, emit, nnz, n_rows, extra=None):
    stream = torch.cuda.current_stream().cuda_stream
    pk = peak_gbs()
    import re
    for label, kernel, tune in variants:
        if ONLY and not re.search(ONLY, label):
            continue
        _cabi.tune("reset", 0)
        for key, val in tune.items():
            _cabi.tune(key, val)

        def fn(i):
            A, B, C = sets[i % len(sets)]
            A.multiply(B.data_ptr(), k, C.data_ptr(), kernel, stream)
        try:
            ms = time_launches(fn, iters, warmup=max(5, 10 * len(sets)))  # AUTO builds a handle's tile layout on its 9th multiply: outside the timing
        except Exception as e:  # unsupported shape for this k: report and go on
            emit({"config": name, "k": k, "variant": label, "error": str(e)[:200]})
            continue
        finally:
            _cabi.tune("reset", 0)
        gb = abytes(n_rows, nnz, k) / (ms * 1e-3) / 1e9
        rec = {"config": name, "k": k, "variant": label, "us": ms * 1e3, "gflops": 2.0 * nnz * k / (ms * 1e-3) / 1e9,
               "algo_GBs": gb, "frac_measured_peak": gb / pk, "frac_8TBs": gb / 8000.0, "sets": len(sets)}
        if extra:
            rec.update(extra)
        emit(rec)


def variant_list(k, full):
    v = [("auto", "auto", {}), ("auto pdl=0", "auto", {"tiled.pdl": 0}), ("rows(auto shape)", "rows", {}), ("merge", "merge", {})]
    if k in (1, 2, 4, 8):
        v.append(("stream", "stream", {}))
        v += [(f"stream tile={t}", "stream", {"stream.tile": t}) for t in (256, 512, 1024, 2048, 4096, 8192) if t * k * 8 <= 96 * 1024]
    if not full:
        return v
    for u in (1, 2, 4, 8):
        v.append((f"rows u={u}", "rows", {"rows.unroll": u}))
    for ctas in (1, 2, 3, 4, 6):
        v.append((f"rows ctas/sm={ctas}", "rows", {"rows.ctas_per_sm": ctas}))
    if k >= 16:
        for kl, nv in ((8, 4), (16, 2), (16, 4), (32, 1), (32, 2), (8, 2), (8, 1), (16, 1)):
            if kl * nv * 2 <= max(k, 16) * 1 and (k // 2) % (kl * nv) == 0:
                for u in (2, 4):
                    v.append((f"rows kl={kl} nv={nv} u={u}", "rows", {"rows.kl": kl, "rows.nv": nv, "rows.unroll": u}))
    else:
        for np_ in (1, 2, 4, 8, 16, 32):
            for u in (1, 2, 4):
                v.append((f"rows np={np_} u={u}", "rows", {"rows.np": np_, "rows.unroll": u}))
    for pf in (0, 1, 2, 3):
        v.append((f"rows pf={pf}", "rows", {"rows.prefetch": pf}))
        v.append((f"rows u=4 pf={pf}", "rows", {"rows.prefetch": pf, "rows.unroll": 4}))
    for items in (128, 256, 1024, 2048):
        v.append((f"merge items={items}", "merge", {"merge.items": items}))
    return v


def cfg2(args, emit, dev):
    n, nc, r, c, v, sym = gen.cop20k_A_shaped()
    first = spmm.DeviceCSR.from_coo_host(n, nc, r, c, v, sym, device=dev.index)
    host = first.download()
    emit({"config": "cfg2", "schedule": first.schedule(), "n_rows": n, "nnz": host.nnz})
    for k in [int(x) for x in args.k.split(",")] if args.k else (1, 8, 32, 64):
        fp = abytes(n, host.nnz, k)
        sets = operand_sets(lambda s: spmm.DeviceCSR.from_host(host, dev.index), n, n, k, dev, fp)
        run_variants("cfg2", sets, k, variant_list(k, args.variants), args.iters, emit, host.nnz, n)
        for A, _, _ in sets:
            A.close()
        del sets
        torch.cuda.empty_cache()
        if k >= 2 and k % 2 == 0 and args.tiles:
            for spec in args.tiles.split(","):
                f = [int(x) for x in spec.split("x")]
                T, BR = f[0], f[1]
                thr = f[2] if len(f) > 2 else 0
                depth = f[3] if len(f) > 3 else 0
                ns_cap = f[4] if len(f) > 4 else 0
                pool = f[5] if len(f) > 5 else 0
                ksplit = f[6] if len(f) > 6 else 0
                group = f[7] if len(f) > 7 else 0

                def make(s, T=T, BR=BR, thr=thr, depth=depth, ns_cap=ns_cap, pool=pool, ksplit=ksplit, group=group):
                    A = spmm.DeviceCSR.from_host(host, dev.index)
                    _cabi.tune("reset", 0)
                    _cabi.tune("tiled.thr", thr)
                    _cabi.tune("tiled.depth", depth)
                    _cabi.tune("tiled.ns", ns_cap)
                    _cabi.tune("tiled.pool", pool)
                    _cabi.tune("tiled.ksplit", ksplit)
                    _cabi.tune("tiled.group", group)
                    try:
                        # cut for this k as AUTO cuts it; an explicit ksplit takes the form that reads tiled.ksplit (16-column k-tile)
                        A.build_tiles(T, BR, 0 if ksplit else k)
                    finally:
                        _cabi.tune("reset", 0)
                    return A
                try:
                    sets = operand_sets(make, n, n, k, dev, fp)
                except Exception as e:
                    emit({"config": "cfg2", "k": k, "tiles": spec, "error": str(e)[:200]})
                    continue
                info = sets[0][0].tile_info()
                if not info["rows_per_tile"]:
                    emit({"config": "cfg2", "k": k, "tiles": spec, "error": "no tile shape fits", "info": info})
                    continue
                base = f"tiled {spec} T={info['rows_per_tile']} NS={info['window_slots']}"
                run_variants("cfg2", sets, k, [(base, "tiled", {})], args.iters, emit, host.nnz, n, {"tiles": info})
                for A, _, _ in sets:
                    A.close()
                del sets
                torch.cuda.empty_cache()
    return host


def cfg1(args, emit, dev):
    n, nc, r, c, v, sym = gen.uniform_random(10_000, 10, seed=1)
    A = spmm.DeviceCSR.from_coo_host(n, nc, r, c, v, sym, device=dev.index)
    host = A.download()
    sets = [(A, torch.from_numpy(spmm.generateLargeFatVector(n, 4)).to(dev), torch.empty((n, 4), dtype=torch.float64, device=dev))]
    run_variants("cfg1", sets, 4, variant_list(4, False), args.iters, emit, host.nnz, n, {"note": "launch-latency bound; L2 warm"})
    cpu_reference(emit, "cfg1", host, spmm.generateLargeFatVector(n, 4), 4, [("seq", 1), ("row", 4)])


def cfg3(args, emit, dev, scale=22, ef=16, k=32):
    A = spmm.DeviceCSR.rmat(scale, ef << scale, seed=11, device=dev.index)
    n = A.n_rows
    emit({"config": "cfg3", "schedule": A.schedule(), "n_rows": n, "nnz": A.nnz})
    sets = [(A, torch.randint(1, 101, (n, k), device=dev).double(), torch.empty((n, k), dtype=torch.float64, device=dev))]
    vs = [("auto", "auto", {}), ("rows", "rows", {}), ("merge", "merge", {})]
    if args.variants:
        vs += [(f"merge items={i}", "merge", {"merge.items": i}) for i in (128, 256, 1024, 4096)]
        vs += [(f"rows u={u}", "rows", {"rows.unroll": u}) for u in (2, 4)]
    run_variants("cfg3", sets, k, vs, max(5, args.iters // 10), emit, A.nnz, n)
    return A


def cfg4(args, emit, dev, n=1 << 25, npr=32, hb=4096, k=16):
    A = spmm.DeviceCSR.banded(n, npr, hb, seed=7, device=dev.index)
    sets = [(A, torch.randint(1, 101, (n, k), device=dev).double(), torch.empty((n, k), dtype=torch.float64, device=dev))]
    vs = [("auto", "auto", {}), ("rows", "rows", {}), ("merge", "merge", {})]
    vs += [("rows one chunk per CTA", "rows", {"rows.tile": -1})]
    if args.variants:
        vs += [(f"rows np={p} u={u}", "rows", {"rows.np": p, "rows.unroll": u}) for p in (1, 2, 4) for u in (1, 2, 4)]
        vs += [(f"rows tile={t}", "rows", {"rows.tile": t}) for t in (64, 128, 512, 1024, 4096)]
    run_variants("cfg4", sets, k, vs, max(3, args.iters // 20), emit, A.nnz, n)
    A.close()


def cfg5(args, emit, dev, n=1 << 23, npr=32, k=64):
    A = spmm.DeviceCSR.banded(n, npr, n // 2, seed=9, device=dev.index)  # window = whole row: uniform columns
    sets = [(A, torch.randint(1, 101, (n, k), device=dev).double(), torch.empty((n, k), dtype=torch.float64, device=dev))]
    vs = [("auto", "auto", {}), ("rows", "rows", {}), ("merge", "merge", {})]
    run_variants("cfg5", sets, k, vs, max(3, args.iters // 20), emit, A.nnz, n,
                 {"note": "uniform random columns: B gather is HBM traffic, not L2/L1 hits"})
    A.close()


def cpu_reference(emit, name, host, B, k, runs, budget_s=20.0):
    """The reference's own CPU code (oracle/_ref) on the host cores, bounded."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyoracle
    if not pyoracle.Reference.available():
        emit({"config": name, "cpu_reference": "oracle/_ref not built"})
        return
    ref = pyoracle.Reference("fast")
    for strategy, P in runs:
        t0, times = time.perf_counter(), []
        while len(times) < 5 and time.perf_counter() - t0 < budget_s:
            times.append(ref.spmm(host.numCols, host.rowPtr, host.colIndices, host.values, B, k, strategy, P, want_result=False)[1])
        t = min(times)
        emit({"config": name, "k": k, "cpu_reference": strategy, "P": P, "host_cores": os.cpu_count(),
              "seconds": t, "gflops": 2.0 * host.nnz * k / t / 1e9, "flags": "-O3 -march=x86-64-v3"})


# ---------------------------------------------------------------- multi-GPU (torchrun)
def multi_gpu(args, emit, dev, rank, world):
    eng = spmm.CudaCompute(dev.index)
    stream_sync = torch.cuda.synchronize
    pk = peak_gbs()

    def tmax(ms):
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, iters):
        for _ in range(2):
            fn()
        stream_sync()
        dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        stream_sync()
        dist.barrier()
        return tmax(a.elapsed_time(b) / iters)

    cfgs = args.configs.split(",")
    if "cfg4" in cfgs:  # row blocks of the large banded matrix, B replicated by NCCL broadcast
        n, npr, hb, k = 1 << 25, 32, 4096, 16
        s, e = spmm.partition_rows(n, world, rank)
        A = spmm.DeviceCSR.banded(n, npr, hb, seed=7, device=dev.index, row_begin=s, row_end=e)
        plan = spmm.RowWise(eng, n, k, A)
        B = torch.empty((n, k), dtype=torch.float64, device=dev)
        if rank == 0:
            B.copy_(torch.randint(1, 101, (n, k), device=dev).double())
        t_b = timed(lambda: plan.broadcast_B(B), 5)
        C = torch.empty((e - s, k), dtype=torch.float64, device=dev)
        t_k = timed(lambda: plan.multiply_local(B, C), 10)
        t_g = timed(lambda: plan.all_gather(C), 5)
        t_all = timed(lambda: plan.all_gather(plan.multiply_local(plan.broadcast_B(B), C)), 5)
        t_kg = timed(lambda: plan.all_gather(plan.multiply_local(B, C)), 5)
        t_ov = {c: timed(lambda c=c: plan.multiply_all_gather_overlapped(B, chunks=c), 5) for c in (2, 4, 8)}
        # gather fused into the multiply: C rows stored from registers into every peer's buffer over NVLink
        t_p2p = timed(lambda: plan.multiply_all_gather_p2p(B), 5)
        t_root = timed(lambda: plan.run_p2p(B), 5)
        t_nccl_root = timed(lambda: plan.gather(plan.multiply_local(B, C)), 5)
        nnz = n * npr
        if rank == 0:
            emit({"config": "cfg4", "strategy": "row-wise", "n_gpus": world, "k": k, "kernel_ms": t_k,
                  "broadcast_B_ms": t_b, "all_gather_C_ms": t_g, "bcast+kernel+gather_ms": t_all,
                  "kernel+gather_ms": t_kg, "kernel+gather_overlapped_ms": t_ov,
                  "fused_p2p_all_gather_ms": t_p2p, "fused_p2p_gather_to_root_ms": t_root,
                  "kernel+nccl_gather_to_root_ms": t_nccl_root,
                  "kernel_gflops": 2.0 * nnz * k / (t_k * 1e-3) / 1e9,
                  "kernel_algo_GBs_per_gpu": abytes(e - s, nnz // world, k, b_rows=(e - s) + 2 * hb) / (t_k * 1e-3) / 1e9,
                  "frac_measured_peak_per_gpu": abytes(e - s, nnz // world, k, b_rows=(e - s) + 2 * hb) / (t_k * 1e-3) / 1e9 / pk,
                  "nvlink_GBs_bcast": n * k * 8 / (t_b * 1e-3) / 1e9})
        A.close()
        del B, C
        torch.cuda.empty_cache()
    if "cfg5" in cfgs:  # column blocks, partial C summed by NCCL reduce-scatter
        n, npr, k = 1 << 23, 32, 64
        whole = spmm.DeviceCSR.banded(n, npr, n // 2, seed=9, device=dev.index)
        c0, c1 = spmm.partition_rows(n, world, rank)
        A = whole.column_block(c0, c1)
        whole.close()
        plan = spmm.ColumnBlocks(eng, n, n, k, A)
        Bl = torch.randint(1, 101, (c1 - c0, k), device=dev).double()
        partial = torch.empty((plan.block * world, k), dtype=torch.float64, device=dev)
        mine = torch.empty((plan.block, k), dtype=torch.float64, device=dev)
        t_k = timed(lambda: plan.multiply_local(Bl, partial), 10)
        t_r = timed(lambda: plan.reduce_scatter(partial, mine), 5)
        t_all = timed(lambda: plan.reduce_scatter(plan.multiply_local(Bl, partial), mine), 5)
        t_ov = {c: timed(lambda c=c: plan.multiply_reduce_scatter_overlapped(Bl, chunks=c), 5) for c in (2, 4, 8)}
        t_p2p = timed(lambda: plan.multiply_reduce_scatter_p2p(Bl, mine), 5)
        nnz = n * npr
        if rank == 0:
            emit({"config": "cfg5", "strategy": "column blocks + reduce-scatter", "n_gpus": world, "k": k,
                  "kernel_ms": t_k, "reduce_scatter_ms": t_r, "kernel+reduce_scatter_ms": t_all,
                  "kernel+p2p_rank_order_reduce_ms": t_p2p,
                  "kernel+reduce_scatter_overlapped_ms": t_ov,
                  "gflops_total_overlapped": 2.0 * nnz * k / (min(t_ov.values()) * 1e-3) / 1e9,
                  "gflops_total": 2.0 * nnz * k / (t_all * 1e-3) / 1e9,
                  "kernel_gflops": 2.0 * nnz * k / (t_k * 1e-3) / 1e9,
                  "reduce_scatter_busGBs": (world - 1) / world * n * k * 8 / (t_r * 1e-3) / 1e9})
        A.close()
        del partial, mine, Bl
        torch.cuda.empty_cache()
    if "cfg3" in cfgs:  # non-zero ranges of the R-MAT matrix, boundary rows fixed up peer to peer
        scale, ef, k = 22, 16, 32
        whole = spmm.DeviceCSR.rmat(scale, ef << scale, seed=11, device=dev.index)  # same seed: same matrix on every rank
        n, nnz = whole.n_rows, whole.nnz
        b, e = spmm.partition_nnz(nnz, world, rank)
        first, last = whole.nnz_range_rows(b, e)
        host_rp = whole.download().rowPtr
        B = torch.randint(1, 101, (n, k), device=dev).double()
        plan = spmm.NonZeroRanges(_RangeEngine(whole, b, e, first, last, dev), n, k, _RangeShard(last - first + 1), first,
                                  last, bool(b > host_rp[first]))
        t_k = timed(lambda: plan.multiply_local(B), 10)
        Cl = plan.multiply_local(B)
        t_f = timed(lambda: plan.fix_boundaries(Cl), 5)
        s, e2 = spmm.partition_rows(n, world, rank)
        rows_time = timed(lambda: whole.multiply_rows(s, e2, B.data_ptr(), k, Cl.data_ptr() if Cl.shape[0] >= e2 - s
                                                      else _scratch(e2 - s, k, dev).data_ptr(), "rows"), 10)
        if rank == 0:
            emit({"config": "cfg3", "strategy": "non-zero ranges + P2P boundary rows", "n_gpus": world, "k": k,
                  "kernel_ms": t_k, "boundary_fixup_ms": t_f, "kernel_gflops": 2.0 * nnz * k / (t_k * 1e-3) / 1e9,
                  "row_blocks_rows_kernel_ms": rows_time,
                  "row_blocks_gflops": 2.0 * nnz * k / (rows_time * 1e-3) / 1e9})
        whole.close()


_scratch_buf = {}


def _scratch(rows, k, dev):
    key = (rows, k)
    if key not in _scratch_buf:
        _scratch_buf[key] = torch.empty((rows, k), dtype=torch.float64, device=dev)
    return _scratch_buf[key]


class _RangeShard:
    def __init__(self, n_rows):
        self.n_rows = n_rows


class _RangeEngine:
    """Engine for NonZeroRanges when the whole CSR is resident: the shard is a non-zero range of it."""

    def __init__(self, whole, b, e, first, last, dev):
        self.whole, self.b, self.e, self.first, self.last, self.device = whole, b, e, first, last, dev

    def multiply(self, A, B, k, out=None):
        if out is None:
            out = _scratch(self.last - self.first + 1, k, self.device)
        self.whole.multiply_nnz_range(self.b, self.e, self.first, self.last, B.data_ptr(), k, out.data_ptr(), "auto",
                                      torch.cuda.current_stream().cuda_stream)
        return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="cfg2")
    ap.add_argument("--k", default="")
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--variants", action="store_true")
    ap.add_argument("--cpu", action="store_true", help="also time the reference CPU code on cfg2")
    ap.add_argument("--tiles", default="", help="cfg2: tile layouts to time, e.g. -1x16,64x16,32x8x2x3 (rows_per_tile x box_rows [x box threshold [x depth [x window slots "
                    "[x pool rows [x ksplit [x group]]]]]]; the k-tile is the one AUTO cuts for k)")
    ap.add_argument("--only", default="", help="regex: run only the variants whose label matches")
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "harness.jsonl"))
    args = ap.parse_args()
    global ONLY
    ONLY = args.only
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    fout = open(args.out, "a") if rank == 0 else None

    def emit(rec):
        rec = dict(rec, world=world, ts=time.time())
        if fout:
            fout.write(json.dumps(rec) + "\n")
            fout.flush()
        if rank == 0:
            keys = [k for k in ("config", "k", "variant", "strategy", "us", "kernel_ms", "gflops", "kernel_gflops",
                                "algo_GBs", "frac_measured_peak", "frac_8TBs", "error") if k in rec]
            print("  ".join(f"{k}={rec[k]:.4g}" if isinstance(rec[k], float) else f"{k}={rec[k]}" for k in keys)
                  or json.dumps(rec), flush=True)

    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        multi_gpu(args, emit, dev, rank, world)
        dist.destroy_process_group()
        return
    for name in args.configs.split(","):
        if name == "cfg1":
            cfg1(args, emit, dev)
        elif name == "cfg2":
            host = cfg2(args, emit, dev)
            if args.cpu:
                for k in (1, 8, 32, 64):
                    B = np.random.default_rng(k).integers(1, 101, (host.numRows, k)).astype(np.float64)
                    cpu_reference(emit, "cfg2", host, B, k, [("seq", 1), ("row", os.cpu_count() or 1), ("nnz", os.cpu_count() or 1)], 10.0)
        elif name == "cfg3":
            cfg3(args, emit, dev).close()
        elif name == "cfg3s":
            cfg3(args, emit, dev, scale=20).close()
        elif name == "cfg4":
            cfg4(args, emit, dev)
        elif name == "cfg4s":
            cfg4(args, emit, dev, n=1 << 22)
        elif name == "cfg5":
            cfg5(args, emit, dev)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
