#!/usr/bin/env python
"""bench.py — the headline measurement of the SpMM hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--k 64] [--dump-outputs DIR]

One "step" = one pass C = A*B of the cop20k_A-shaped k=64 SpMM (BASELINE.json configs[1], the
configuration the north_star target is quoted on) over one resident operand set. A and B are seeded,
so the same arguments give the same inputs in every run; --dump-outputs DIR writes the C of the last
timed step as DIR/C.npy (float64; DIR/C_rank<r>.npy per rank at N > 1), a fixed sample of its rows
when it would exceed 64 MB, so that two builds can be compared output for output. It applies to the
GPU path only: --impl reference times the CPU code without keeping its result. With N > 1 (one
process per GPU under torchrun) every rank owns one cop20k_A-shaped diagonal block of a
(N*121,192)-row block-diagonal matrix — the row-wise partition (RowWise.cpp:26-29) of a matrix whose
blocks read only their own rows of B, so no byte has to cross a link (weak scaling, no collective
invented). What the north_star's scaling cases cost WITH their exchange steps is measured in the same
run and printed under "north_star_scaling": the large banded row-partitioned case (cfg4: B sharded by
rows, halo rows exchanged peer to peer, kernel, optional gather of C) and the column-block case (cfg5:
kernel + reduce-scatter of the partial C), each with the 1-GPU time of the same problem beside it, and
"parity_ok": the three strategies on this process group against the oracle on a small matrix.

Printed by rank 0: ONE JSON line with metric / value (GFLOP/s = 2*nnz*k/t, whole job) plus
roofline (algorithmic bytes / kernel time vs the measured HBM copy peak; the kernel name is what the
library reports it launched), e2e (the same multiply through the reference's own C++ entry point:
std::vector<std::vector<double>> in and out, pack / H2D / kernel / D2H / unpack inside the timed region;
"e2e_first_call" adds the upload of A and the layout build, the reference's one-call-per-run pattern
main.cpp:78; "e2e_pinned" is the flat pinned-buffer C-ABI call) and cpu_baseline (the reference's own
CPU code on the host cores). At N = 1 "configs_1gpu" adds the kernel times of BASELINE.json configs 3-5.

--impl reference times the reference's own CPU implementation (oracle/_ref, compiled from the
reference sources; else the oracle port) on the same TOTAL workload (the N-block matrix at --gpus N),
all host threads, rank 0 only.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the benchmark leaves the tree it runs from as it found it: build() never imports oracle/pyoracle.py, so without this
# the first run would add oracle/__pycache__/ to a tree that has just been built
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402

N_ROWS, NNZ = 121_192, 2_624_331
OPERAND_SETS = 4  # rotating resident copies of (A, B, C): 4 x ~175 MB >> 126 MB L2
DUMP_BYTES = 63_000_000  # array bytes --dump-outputs writes over every rank: under 64 MB with the .npy headers


def dump_output(path: str, C: np.ndarray, budget: int) -> None:
    """C as .npy; a fixed, seeded sample of its rows (in row order) when it is larger than `budget` bytes."""
    if C.nbytes > budget:
        keep = budget // (C.shape[1] * C.itemsize)
        C = C[np.sort(np.random.default_rng(0).choice(C.shape[0], keep, replace=False))]
    np.save(path, C)


def algorithmic_bytes(n_rows: int, nnz: int, k: int) -> int:
    """SURVEY.md §8(d): A's CSR arrays + B once + C once."""
    return nnz * 12 + (n_rows + 1) * 4 + 2 * n_rows * k * 8


def measured_peak_gbs() -> tuple[float, str]:
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def recorded_traffic(k: int):
    """(dram bytes per launch of the dominant kernel, where it was recorded): read from the committed ncu --set full
    capture named in profiles/traffic.json — a RECORDED figure, not measured in this run (ncu cannot run inside it)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            d = json.load(f)
            return d.get(f"cop20k_k{k}"), "recorded: " + d.get("source", "profiles/traffic.json")
    except Exception:
        return None, None


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled DURING the timed region (NVML, ~5 ms period)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def stop(self) -> dict:
        self._stop_evt.set()
        self.join(timeout=2)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def build_workload(k: int, seed: int = 20):
    """cop20k_A-shaped records (host) — the same for both arms."""
    from sparsematrixmultiplicationmpi_b200 import generators as gen
    return gen.cop20k_A_shaped(n=N_ROWS, nnz=NNZ, seed=seed)


def block_diagonal_host(n_blocks: int, k: int):
    """Host CSR of the N-block block-diagonal matrix the N ranks of the GPU arm multiply (block r = seed 20 + r)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyoracle
    from sparsematrixmultiplicationmpi_b200.matrix import SparseMatrix
    orc = pyoracle.Oracle()
    rps, cis, vas = [], [], []
    for b in range(n_blocks):
        n, nc, r, c, v, sym = build_workload(k, seed=20 + b)
        rp, ci, va = orc.csr_from_coo(n, r, c, v, sym)  # the reference loader's CSR assembly
        rps.append(rp[1:].astype(np.int64) + b * NNZ if b else rp.astype(np.int64))
        cis.append(ci + b * N_ROWS)
        vas.append(va)
    return SparseMatrix(np.concatenate(vas), np.concatenate(cis).astype(np.int32), np.concatenate(rps).astype(np.int32),
                        n_blocks * N_ROWS, n_blocks * N_ROWS)


def cpu_reference_run(host, B, k, steps, warmup, max_seconds=60.0):
    """The reference's own CPU code on the host cores: row-wise strategy at P = all hardware threads
    (its "mpirun" path on compat MPI) and the sequential function; returns the faster one."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyoracle
    cores = os.cpu_count() or 1
    if pyoracle.Reference.available():
        ref, kind = pyoracle.Reference("fast"), "reference"

        def run(strategy, P):
            return ref.spmm(host.numCols, host.rowPtr, host.colIndices, host.values, B, k, strategy, P,
                            want_result=False)[1]
    else:
        orc, kind = pyoracle.Oracle(), "port"
        cores = 1

        def run(strategy, P):
            t0 = time.perf_counter()
            orc.spmm(host.rowPtr, host.colIndices, host.values, B, k, "seq", 1)
            return time.perf_counter() - t0
    best = {}
    t_begin = time.perf_counter()
    for strategy, P in (("row", cores), ("seq", 1)) if kind == "reference" else (("seq", 1),):
        for _ in range(max(1, warmup)):
            run(strategy, P)
        times = []
        for _ in range(steps):
            times.append(run(strategy, P))
            if time.perf_counter() - t_begin > max_seconds:
                break
        best[(strategy, P)] = statistics.mean(times)
    (strategy, P), t = min(best.items(), key=lambda kv: kv[1])
    # one call of the row-wise function on ONE rank: its flatten / Gatherv / re-nest (RowWise.cpp:63-121) is serial work on the
    # root whatever carries the ranks — the reason its all-cores time does not beat the sequential function at -O3
    one_rank = None
    if kind == "reference" and cores > 1 and time.perf_counter() - t_begin < max_seconds:
        run("row", 1)
        one_rank = run("row", 1)
    flops = 2.0 * host.nnz * k
    blocks = max(1, host.numRows // N_ROWS)
    return {"value": flops / t / 1e9, "unit": "GFLOP/s", "cores": P, "kind": kind,
            "sample": f"full cop20k_A-shaped k={k} multiply ({blocks} diagonal block{'s' if blocks > 1 else ''}), reference {strategy} strategy at P={P} "
                      f"(-O3 -march=x86-64-v3, compat MPI rank-threads), mean of {len(times)} calls",
            "seconds_per_step": t,
            "sequential_gflops": flops / best[("seq", 1)] / 1e9 if ("seq", 1) in best else None,
            "rowwise_all_cores_gflops": flops / best[("row", cores)] / 1e9 if ("row", cores) in best else None,
            "rowwise_one_rank_seconds": one_rank,
            "host_cores": os.cpu_count()}


def entry_lib():
    """libspmm_entry.so: the reference's four C++ entry points + the spmm_entry_run measurement hook."""
    import ctypes as C
    lib = C.CDLL(os.path.join(ROOT, "sparsematrixmultiplicationmpi_b200", "libspmm_entry.so"))
    lib.spmm_entry_run.restype = C.c_int
    lib.spmm_entry_run.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                   C.c_char_p, C.c_int]
    return lib


def entry_run(lib, strategy, P, host, B, k, steps, want_result=False, warmup=10):
    """C++ SparseMatrix + FatVector in, FatVector out, `steps` calls after the first: (first_call_s, mean_s, C or None)."""
    import ctypes as C
    out = np.empty((host.numRows, k)) if want_result else None
    first, mean = C.c_double(), C.c_double()
    err = C.create_string_buffer(512)
    rc = lib.spmm_entry_run(strategy, P, host.numRows, host.numCols, host.nnz, host.rowPtr.ctypes.data,
                            host.colIndices.ctypes.data, host.values.ctypes.data, k, B.ctypes.data,
                            out.ctypes.data if want_result else None, warmup, steps, C.byref(first), C.byref(mean), err, 512)
    if rc:
        raise RuntimeError(err.value.decode() or f"spmm_entry_run status {rc}")
    return first.value, mean.value, out


def main():
    # stdout carries exactly ONE JSON line: everything else this process or its libraries print
    # (NCCL's version banner, torchrun notices) is sent to stderr.
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line: dict) -> None:
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--k", type=int, default=64)
    ap.add_argument("--kernel", default="auto")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip configs_1gpu / north_star_scaling (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the C of the last timed step to DIR as .npy (--impl ours only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the output of the GPU path (--impl ours)")
    k = args.k
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    os.environ.setdefault("SPMM_DEVICE_BASE", str(local_rank))  # the C++ entry points of this process drive this rank's GPU
    # host threads of the pack / unpack pool: the ranks of one box share its cores
    os.environ.setdefault("SPMM_HOST_THREADS", str(max(2, min(16, (os.cpu_count() or 8) // max(1, world)))))
    metric = "SpMM GFLOP/s and HBM GB/s (% roofline) at 1/2/4/8 B200 vs ref CPU MPI"
    n_blocks = max(1, args.gpus if args.impl == "reference" else world)
    config = {"workload": f"cop20k_A-shaped synthetic FEM matrix {N_ROWS}x{N_ROWS}, {NNZ} nnz, k={k}, FP64 "
                          f"(BASELINE.json configs[1]); one such diagonal block per GPU, row-wise partition "
                          f"({n_blocks} block{'s' if n_blocks > 1 else ''} in this run)",
              "n_rows_per_gpu": N_ROWS, "nnz_per_gpu": NNZ, "k": k, "blocks": n_blocks,
              "l2": f"{OPERAND_SETS} rotating resident operand sets (> 126 MB L2) so every step reads cold operands"}

    if args.impl == "reference":
        if rank != 0:
            return
        import sparsematrixmultiplicationmpi_b200  # noqa: F401  (generators only; no GPU work on this arm)
        host = block_diagonal_host(n_blocks, k)  # the same TOTAL work as the GPU arm at this N
        B = np.random.default_rng(1).integers(1, 101, (host.numCols, k)).astype(np.float64)
        steps = min(args.steps, 20 if n_blocks == 1 else 5)
        warm = min(args.warmup, 2 if n_blocks == 1 else 1)
        res = cpu_reference_run(host, B, k, steps, warm, max_seconds=60.0 if n_blocks == 1 else 120.0)
        line = {"impl": "reference", "metric": metric, "value": res["value"], "unit": "GFLOP/s", "n_gpus": args.gpus,
                "steps": steps, "warmup": warm, "ms_per_step": res["seconds_per_step"] * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic", "config": config, "cpu_baseline": res,
                "e2e": {"value": res["value"], "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        emit(line)
        return

    import torch
    import torch.distributed as dist
    import sparsematrixmultiplicationmpi_b200 as spmm
    from sparsematrixmultiplicationmpi_b200 import _cabi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the SpMM path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    stream = torch.cuda.current_stream().cuda_stream

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def tmax(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, iters, warm=2):
        """Mean device ms of fn over `iters` calls: CUDA events on the launching stream, barrier on both sides, max over ranks."""
        for _ in range(warm):
            fn()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        barrier()
        return tmax(a.elapsed_time(b) / iters)

    # ---- operands resident in HBM: OPERAND_SETS copies of this rank's diagonal block ----
    n, nc, r, c, v, sym = build_workload(k, seed=20 + rank)
    first = spmm.DeviceCSR.from_coo_host(n, nc, r, c, v, sym, device=local_rank)
    host = first.download()
    sets = []
    for s in range(OPERAND_SETS):
        A = first if s == 0 else spmm.DeviceCSR.from_host(host, local_rank)
        if args.kernel in ("auto", "tiled"):
            A.build_tiles(-1, 0, k)  # what AUTO does by itself on its first multiply; done here so it is outside any timing
        gen_b = torch.Generator(device=dev)
        gen_b.manual_seed(OPERAND_SETS * rank + s)
        Bd = torch.randint(1, 101, (n, k), device=dev, generator=gen_b).double()
        Cd = torch.empty((n, k), dtype=torch.float64, device=dev)
        sets.append((A, Bd, Cd))
    tiles = sets[0][0].tile_info()
    launches_per_step = 2 if (args.kernel == "merge") else 1

    def step(i):
        A, Bd, Cd = sets[i % OPERAND_SETS]
        A.multiply(Bd.data_ptr(), k, Cd.data_ptr(), args.kernel, stream)

    for i in range(max(args.warmup, 3)):
        step(i)
    kernel_name = (_cabi.lib().spmm_last_kernel_name() or b"").decode()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    t_wall = time.perf_counter()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(args.steps):
        step(i)
    ev1.record()
    barrier()
    wall = time.perf_counter() - t_wall
    clocks = sampler.stop()
    if args.dump_outputs:  # read back now: the L2-warm pass below writes the C of operand set 0 again
        os.makedirs(args.dump_outputs, exist_ok=True)
        dump_output(os.path.join(args.dump_outputs, "C.npy" if world == 1 else f"C_rank{rank}.npy"),
                    sets[(args.steps - 1) % OPERAND_SETS][2].cpu().numpy(), DUMP_BYTES // world)
    ms_per_step = tmax(ev0.elapsed_time(ev1)) / args.steps
    # beside it (SURVEY 8d: "both L2-warm and L2-flushed"): the same launches on ONE operand set, whatever fits stays in L2
    w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0.record()
    for i in range(args.steps):
        step(0)
    w1.record()
    barrier()
    warm_ms_per_step = tmax(w0.elapsed_time(w1)) / args.steps
    flops_per_step = 2.0 * NNZ * k * world
    value = flops_per_step / (ms_per_step * 1e-3) / 1e9

    # ---- roofline of the dominant kernel (this rank's launch) ----
    peak, peak_kind = measured_peak_gbs()
    abytes = algorithmic_bytes(N_ROWS, NNZ, k)
    achieved = abytes / (ms_per_step * 1e-3) / 1e9
    traffic, traffic_source = recorded_traffic(k)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_source, "peak_kind": peak_kind,
                "algorithmic_bytes_per_launch": abytes, "frac_of_8TBs_nominal": achieved / 8000.0,
                "kernel": kernel_name, "tiles": tiles}

    # ---- e2e through the reference's own boundary: C++ SparseMatrix / FatVector objects, the entry point of
    # SparseMatrixFatVectorMultiply.h:14-15 (pack, H2D, kernel, D2H, unpack all inside the timed region) ----
    spmm.clear_cache()
    Bh = np.random.default_rng(7).integers(1, 101, (n, k)).astype(np.float64)
    e2e_steps = max(3, min(args.steps, 20))
    lib = entry_lib()
    barrier()
    first_s, mean_s, _ = entry_run(lib, 0, 1, host, Bh, k, e2e_steps)
    first_s, mean_s = tmax(first_s), tmax(mean_s)
    e2e = {"value": flops_per_step / mean_s / 1e9, "unit": "GFLOP/s", "h2d_bytes_per_step": n * k * 8,
           "d2h_bytes_per_step": n * k * 8, "ms_per_step": mean_s * 1e3,
           "api": "C++ sparseMatrixFatVectorMultiply(const SparseMatrix&, const FatVector&, int) of libspmm_entry.so: "
                  "vector<vector<double>> in and out, A cached in HBM after the first call",
           "host_threads": int(os.environ["SPMM_HOST_THREADS"])}
    e2e_first = {"value": flops_per_step / first_s / 1e9, "unit": "GFLOP/s", "ms": first_s * 1e3,
                 "what": "first call on a new matrix: upload of A (32 MB), CSR row kernel (AUTO builds the tile layout only when a handle "
                         "is multiplied again), transfers as above — the reference's one-call-per-run pattern (main.cpp:78); the page-locked "
                         "staging arena and the kernel modules were set up when libspmm_entry.so was loaded (the place of MPI_Init)"}
    # the flat C-ABI call with pinned host buffers (no pack / unpack): what a caller that owns row-major storage gets
    Bp = torch.randint(1, 101, (n, k)).double().pin_memory()
    Cp = torch.empty((n, k), dtype=torch.float64).pin_memory()
    Bp_np, Cp_np = Bp.numpy(), Cp.numpy()
    A0 = sets[0][0]
    for _ in range(3):
        A0.multiply_host(Bp_np, k, args.kernel if args.kernel in ("auto", "rows", "merge", "tiled") else "auto", Cp_np)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        A0.multiply_host(Bp_np, k, "auto", Cp_np)
    pinned_s = tmax((time.perf_counter() - t0) / e2e_steps)
    e2e_pinned = {"value": flops_per_step / pinned_s / 1e9, "unit": "GFLOP/s", "ms_per_step": pinned_s * 1e3,
                  "api": "spmm_multiply_host(A, B, k, C) with pinned row-major host buffers"}

    extras = {}
    if not args.no_extras:
        try:
            extras = north_star_extras(spmm, torch, dist, dev, rank, world, timed, barrier)
        except Exception as e:  # never lose the headline line to an extra
            extras = {"extras_error": f"{type(e).__name__}: {e}"[:300]}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        Bc = np.random.default_rng(1).integers(1, 101, (n, k)).astype(np.float64)
        cpu = cpu_reference_run(host, Bc, k, steps=5, warmup=1, max_seconds=30.0)

    if rank == 0:
        line = {"metric": metric, "value": value, "unit": "GFLOP/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
                "clocks": clocks, "e2e": e2e, "e2e_first_call": e2e_first, "e2e_pinned": e2e_pinned,
                "gpu_launches": launches_per_step * args.steps,
                "roofline": roofline, "cpu_baseline": cpu, "wall_s_timed_region": wall,
                "l2_warm_ms_per_step": warm_ms_per_step,
                "hbm_gbs_per_gpu": achieved, "kernel_arg": args.kernel}
        line.update(extras)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def north_star_extras(spmm, torch, dist, dev, rank, world, timed, barrier):
    """BASELINE.json configs 3-5 in the same run: kernel times on one GPU (world == 1) or the partitioned strategies with
    their exchange steps and the 1-GPU time of the same problem beside them (world > 1); multi-GPU parity vs the oracle."""
    eng = spmm.CudaCompute(dev.index)
    peak, _ = measured_peak_gbs()

    def gbs(n_rows, nnz, k, ms, b_rows=None):
        b = nnz * 12 + (n_rows + 1) * 4 + ((b_rows if b_rows is not None else n_rows) + n_rows) * k * 8
        return b / (ms * 1e-3) / 1e9

    out = {}
    # ---- cfg4: banded 2^25 rows x 32 per row, k = 16, row blocks (RowWise.cpp:26-29) ----
    n, npr, hb, k = 1 << 25, 32, 4096, 16
    nnz = n * npr

    def cfg4_single():
        with spmm.DeviceCSR.banded(n, npr, hb, seed=7, device=dev.index) as A:
            B = torch.randint(1, 101, (n, k), device=dev).double()
            C = torch.empty((n, k), dtype=torch.float64, device=dev)
            s = torch.cuda.current_stream().cuda_stream
            ms = timed_local(torch, lambda: A.multiply(B.data_ptr(), k, C.data_ptr(), "auto", s), 5)
            del B, C
        torch.cuda.empty_cache()
        return ms

    # ---- cfg5: 2^23 rows x 32 uniformly scattered columns per row, k = 64, column blocks + reduce-scatter ----
    n5, k5 = 1 << 23, 64
    nnz5 = n5 * 32

    def cfg5_single():
        with spmm.DeviceCSR.banded(n5, 32, n5 // 2, seed=9, device=dev.index) as A:
            B = torch.randint(1, 101, (n5, k5), device=dev).double()
            C = torch.empty((n5, k5), dtype=torch.float64, device=dev)
            s = torch.cuda.current_stream().cuda_stream
            ms = timed_local(torch, lambda: A.multiply(B.data_ptr(), k5, C.data_ptr(), "auto", s), 3)
            del B, C
        torch.cuda.empty_cache()
        return ms

    if world == 1:
        with spmm.DeviceCSR.rmat(22, 16 << 22, seed=11, device=dev.index) as A:  # cfg3: R-MAT 4M x 4M, 64M edges, k = 32
            k3 = 32
            B = torch.randint(1, 101, (A.n_rows, k3), device=dev).double()
            C = torch.empty((A.n_rows, k3), dtype=torch.float64, device=dev)
            s = torch.cuda.current_stream().cuda_stream
            ms3 = timed_local(torch, lambda: A.multiply(B.data_ptr(), k3, C.data_ptr(), "auto", s), 5)
            ms3_rows = timed_local(torch, lambda: A.multiply(B.data_ptr(), k3, C.data_ptr(), "rows", s), 3)
            n3, nnz3 = A.n_rows, A.nnz
            del B, C
        torch.cuda.empty_cache()
        ms4, ms5 = cfg4_single(), cfg5_single()
        out["configs_1gpu"] = {
            "cfg3_rmat_4M_64M_k32": {"kernel_ms": ms3, "row_kernel_ms": ms3_rows, "gflops": 2.0 * nnz3 * k3 / (ms3 * 1e-3) / 1e9,
                                    "frac_measured_peak": gbs(n3, nnz3, k3, ms3) / peak, "kernel": "nnz-balanced merge-path (AUTO)"},
            "cfg4_banded_32M_1B_k16": {"kernel_ms": ms4, "gflops": 2.0 * nnz * k / (ms4 * 1e-3) / 1e9,
                                       "frac_measured_peak": gbs(n, nnz, k, ms4) / peak},
            "cfg5_uniform_8M_256M_k64": {"kernel_ms": ms5, "gflops": 2.0 * nnz5 * k5 / (ms5 * 1e-3) / 1e9,
                                         "frac_measured_peak": gbs(n5, nnz5, k5, ms5) / peak}}
        # beside the algorithmic-bytes fraction: what the hardware actually moves per launch (RECORDED ncu traffic of the same
        # kernels, profiles/traffic.json) over this run's time — cfg5 runs at the HBM peak, cfg4 and cfg3 at the L2 -> SM cap
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                rec = json.load(f).get("configs_1gpu", {})
            for name, entry in out["configs_1gpu"].items():
                r = rec.get(name)
                if r:
                    t = entry["kernel_ms"] * 1e-3
                    entry["recorded_traffic"] = {"dram_GBs": r["dram_bytes"] / t / 1e9, "dram_frac_measured_peak": r["dram_bytes"] / t / 1e9 / peak,
                                                 "l2_to_sm_GBs": r["l2_to_sm_bytes"] / t / 1e9, "source": "recorded: " + r["source"]}
        except Exception:
            pass
        return out

    # ---- world > 1 ----
    s0, e0 = spmm.partition_rows(n, world, rank)
    A = spmm.DeviceCSR.banded(n, npr, hb, seed=7, device=dev.index, row_begin=s0, row_end=e0)
    plan = spmm.RowWise(eng, n, k, A)
    window, B_own = plan.alloc_window(dev)  # B sharded by rows like C: the rank's rows live inside its window buffer
    B_own.copy_(torch.randint(1, 101, (e0 - s0, k), device=dev).double())
    C_own = torch.empty((e0 - s0, k), dtype=torch.float64, device=dev)
    w0 = plan.exchange_halo_inplace(window)
    t_halo = timed(lambda: plan.exchange_halo_inplace(window), 5)
    t_kernel = timed(lambda: eng.multiply_window(A, window, w0, k, C_own), 10)
    t_all = timed(lambda: eng.multiply_window(A, window, plan.exchange_halo_inplace(window), k, C_own), 5)
    t_gather = timed(lambda: plan.gather(C_own), 3)
    halo_bytes = (window.shape[0] - (e0 - s0)) * k * 8
    A.close()
    del window, B_own, C_own, plan
    torch.cuda.empty_cache()
    barrier()
    one = cfg4_single() if rank == 0 else 0.0
    barrier()
    one = float(_bcast(torch, dist, dev, one))
    out_cfg4 = {"strategy": "row blocks, B sharded by rows, halo rows exchanged peer to peer (NCCL send/recv over NVLink), C left "
                            "row-sharded", "n_rows": n, "nnz": nnz, "k": k, "kernel_ms": t_kernel, "halo_exchange_ms": t_halo,
                "halo_bytes_per_rank": halo_bytes, "exchange_plus_kernel_ms": t_all, "gather_C_to_root_ms": t_gather,
                "one_gpu_kernel_ms": one, "kernel_speedup_vs_1gpu": one / t_kernel, "all_in_speedup_vs_1gpu": one / t_all,
                "gflops_all_in": 2.0 * nnz * k / (t_all * 1e-3) / 1e9,
                "frac_measured_peak_per_gpu": gbs(e0 - s0, nnz // world, k, t_kernel, b_rows=(e0 - s0) + 2 * hb) / peak}

    whole = spmm.DeviceCSR.banded(n5, 32, n5 // 2, seed=9, device=dev.index)
    c0, c1 = spmm.partition_rows(n5, world, rank)
    Ab = whole.column_block(c0, c1)
    whole.close()
    planb = spmm.ColumnBlocks(eng, n5, n5, k5, Ab)
    Bl = torch.randint(1, 101, (c1 - c0, k5), device=dev).double()
    partial = torch.empty((planb.block * world, k5), dtype=torch.float64, device=dev)
    mine = torch.empty((planb.block, k5), dtype=torch.float64, device=dev)
    t_k5 = timed(lambda: planb.multiply_local(Bl, partial), 5)
    t_rs = timed(lambda: planb.reduce_scatter(partial, mine), 3)
    t_all5 = timed(lambda: planb.reduce_scatter(planb.multiply_local(Bl, partial), mine), 3)
    try:
        t_p2p = timed(lambda: planb.multiply_reduce_scatter_p2p(Bl, mine), 3)
    except Exception as e:
        t_p2p = None
        out["cfg5_p2p_error"] = str(e)[:200]
    try:
        t_push = timed(lambda: planb.multiply_reduce_scatter_push(Bl, mine), 3)
    except Exception as e:
        t_push = None
        out["cfg5_push_error"] = str(e)[:200]
    planb._symm = planb._symm_push = None
    Ab.close()
    del partial, mine, Bl, planb
    torch.cuda.empty_cache()
    barrier()
    one5 = cfg5_single() if rank == 0 else 0.0
    barrier()
    one5 = float(_bcast(torch, dist, dev, one5))
    best5 = min(x for x in (t_all5, t_p2p, t_push) if x)
    out_cfg5 = {"strategy": "column blocks of A, partial C summed by reduce-scatter over NVLink", "n_rows": n5, "nnz": nnz5,
                "k": k5, "kernel_ms": t_k5, "reduce_scatter_nccl_ms": t_rs, "kernel_plus_reduce_scatter_nccl_ms": t_all5,
                "kernel_plus_p2p_rank_order_reduce_ms": t_p2p, "fused_peer_store_multiply_plus_local_reduce_ms": t_push,
                "one_gpu_kernel_ms": one5,
                "kernel_speedup_vs_1gpu": one5 / t_k5, "all_in_speedup_vs_1gpu": one5 / best5,
                "reduce_scatter_bus_GBs": (world - 1) / world * n5 * k5 * 8 / (t_rs * 1e-3) / 1e9}
    # ---- cfg3: R-MAT 2^22, 2^26 edges, k = 32 — equal non-zero ranges (NonZeroElement.cpp:24-39), only the rows cut by a
    # range boundary exchanged peer to peer; beside it the same matrix in equal ROW blocks (one rank gets the hub rows) ----
    k3 = 32
    whole = spmm.DeviceCSR.rmat(22, 16 << 22, seed=11, device=dev.index)  # same seed: the same matrix on every rank
    n3, nnz3 = whole.n_rows, whole.nnz
    b3, e3 = spmm.partition_nnz(nnz3, world, rank)
    first, last = whole.nnz_range_rows(b3, e3)
    rp3 = whole.download().rowPtr
    B3 = torch.randint(1, 101, (n3, k3), device=dev).double()
    C3 = torch.empty((last - first + 1, k3), dtype=torch.float64, device=dev)

    class RangeOfWhole:  # the rank's shard is a non-zero range of the resident CSR: no second copy of the matrix
        device = dev

        def multiply(self, A_, B_, k_, out_=None):
            whole.multiply_nnz_range(b3, e3, first, last, B_.data_ptr(), k_, C3.data_ptr(), "auto", torch.cuda.current_stream().cuda_stream)
            return C3

    class RowsOf:
        n_rows = last - first + 1

    plan3 = spmm.NonZeroRanges(RangeOfWhole(), n3, k3, RowsOf(), first, last, bool(b3 > rp3[first]))
    t_k3 = timed(lambda: plan3.multiply_local(B3), 5)
    Cl = plan3.multiply_local(B3)
    t_f3 = timed(lambda: plan3.fix_boundaries(Cl), 3)
    t_all3 = timed(lambda: plan3.fix_boundaries(plan3.multiply_local(B3)), 5)
    rs, re_ = spmm.partition_rows(n3, world, rank)
    Cr = torch.empty((re_ - rs, k3), dtype=torch.float64, device=dev)
    t_rows3 = timed(lambda: whole.multiply_rows(rs, re_, B3.data_ptr(), k3, Cr.data_ptr(), "rows", torch.cuda.current_stream().cuda_stream), 2, warm=1)
    Cfull = torch.empty((n3, k3), dtype=torch.float64, device=dev)
    one3 = timed_local(torch, lambda: whole.multiply(B3.data_ptr(), k3, Cfull.data_ptr(), "auto", torch.cuda.current_stream().cuda_stream), 5) if rank == 0 else 0.0
    barrier()
    one3 = float(_bcast(torch, dist, dev, one3))
    whole.close()
    del B3, C3, Cr, Cfull, Cl
    torch.cuda.empty_cache()
    out_cfg3 = {"strategy": "equal non-zero ranges, rows cut by a range boundary fixed up peer to peer in rank order", "n_rows": n3,
                "nnz": nnz3, "k": k3, "kernel_ms": t_k3, "boundary_fixup_ms": t_f3, "kernel_plus_fixup_ms": t_all3,
                "one_gpu_kernel_ms": one3, "kernel_speedup_vs_1gpu": one3 / t_k3, "all_in_speedup_vs_1gpu": one3 / t_all3,
                "equal_row_blocks_row_kernel_ms": t_rows3}

    # ---- the reference's own reading of column-wise (ColumnWise.cpp:25-48): B's k columns split across the ranks, on cfg2 ----
    n2, nc2, r2, c2, v2, sym2 = build_workload(64)
    with spmm.DeviceCSR.from_coo_host(n2, nc2, r2, c2, v2, sym2, device=dev.index) as A2:
        slabs = spmm.ColumnSlabs(eng, 64, A2)
        B2 = torch.randint(1, 101, (n2, 64), device=dev).double()
        C2 = torch.zeros((n2, 64), dtype=torch.float64, device=dev)
        t_slab_k = timed(lambda: eng.multiply_slab(A2, B2, 64, slabs.k_start, slabs.k_end - slabs.k_start, C2), 20, warm=12)
        t_slab_all = timed(lambda: slabs.run(B2), 5)
        one_slab = timed_local(torch, lambda: A2.multiply(B2.data_ptr(), 64, C2.data_ptr(), "auto", torch.cuda.current_stream().cuda_stream), 20, warm=12)
    out_slabs = {"strategy": "k-slabs of B (the reference's reading): every rank multiplies all of A by k/P columns, slabs gathered on the root",
                 "matrix": "cfg2", "k": 64, "kernel_ms": t_slab_k, "kernel_plus_gather_ms": t_slab_all, "one_gpu_kernel_ms_this_rank": one_slab}

    out["north_star_scaling"] = {"cfg4_banded_32M_1B_k16": out_cfg4, "cfg5_uniform_8M_256M_k64": out_cfg5,
                                 "cfg3_rmat_4M_64M_k32": out_cfg3, "cfg2_column_slabs_k64": out_slabs}
    out["parity_ok"] = multi_gpu_parity(spmm, torch, dist, dev, rank, world)
    return out


def timed_local(torch, fn, iters, warm=2):
    """Mean device ms on this rank only (no barrier: the other ranks are idle)."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def _bcast(torch, dist, dev, x):
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    dist.broadcast(t, src=0)
    return t.item()


def multi_gpu_parity(spmm, torch, dist, dev, rank, world) -> bool:
    """The three strategies on THIS process group (NCCL over NVLink) against the oracle on a small cop20k_A-shaped
    matrix: |x - ref| <= 1e-12 |ref| per entry (the north_star tolerance). The oracle is the checker only."""
    from sparsematrixmultiplicationmpi_b200 import generators as gen
    n, nc, r, c, v, sym = gen.cop20k_A_shaped(n=20_000, nnz=420_001, nx=27, ny=27, seed=4)
    k = 16
    with spmm.DeviceCSR.from_coo_host(n, nc, r, c, v, sym, device=dev.index) as A:
        host = A.download()
    B = np.random.default_rng(3).integers(1, 101, (n, k)).astype(np.float64)
    Bd = torch.from_numpy(B).to(dev)
    eng = spmm.CudaCompute(dev.index)
    results = {}
    row = spmm.RowWise.from_host(eng, host, k)
    bs, be = spmm.partition_rows(n, world, rank)
    results["row_wise_halo"] = row.gather(row.multiply_sharded(Bd[bs:be].contiguous()))
    results["row_wise_p2p"] = row.run_p2p(Bd)
    blk = spmm.ColumnBlocks.from_host(eng, host, k)
    results["column_blocks"] = blk.run(blk.local_B(Bd))
    # the fused variant (the kernel stores every row block into its owner's slots over NVLink, local rank-order sum)
    counts = [max(0, min(blk.block, n - r_ * blk.block)) for r_ in range(world)]
    from sparsematrixmultiplicationmpi_b200.strategies import _gather_rows_to_root
    results["column_blocks_fused_peer_stores"] = _gather_rows_to_root(
        blk.multiply_reduce_scatter_push(blk.local_B(Bd))[:counts[rank]], counts, k, None)
    results["non_zero_ranges"] = spmm.NonZeroRanges.from_host(eng, host, k).run(Bd)
    torch.cuda.synchronize()
    ok = True
    if rank == 0:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import pyoracle
        ref = pyoracle.Oracle().spmm(host.rowPtr, host.colIndices, host.values, B, k)
        for name, t in results.items():
            got = t.cpu().numpy()
            good = got.shape == ref.shape and bool(np.all(np.abs(got - ref) <= 1e-12 * np.abs(ref)))
            if not good:
                print(f"bench.py: multi-GPU parity FAILED for {name}", file=sys.stderr)
            ok = ok and good
    flag = torch.tensor([1.0 if ok else 0.0], dtype=torch.float64, device=dev)
    dist.broadcast(flag, src=0)
    for A_ in (row.A, blk.A):
        A_.close()
    return bool(flag.item() == 1.0)


if __name__ == "__main__":
    main()
