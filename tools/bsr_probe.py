#!/usr/bin/env python
"""Where the BSR kernel (spmm_bsr.cu) wins: fem_blocked matrices with b = 3, 4, 6 at cfg2's size and one b = 3 matrix ten
times larger (B at k = 64 is 620 MB, far beyond the 126 MB L2), k in {1, 2, 3, 4, 8, 16, 32, 33, 64, 128}, arms
  rows    SPMM_KERNEL_ROWS
  tiled   SPMM_KERNEL_TILED after build_tiles(-1, 0, k) (even k)
  stream  SPMM_KERNEL_STREAM (k = 1, 2, 4, 8)
  auto    AUTO on handles without a view, after 12 calls (its lazy tile layout exists)
  bsr     SPMM_KERNEL_BSR after build_bsr(b)
Operand sets (A handle, B, C) are rotated so that their total exceeds the L2, as bench.py does; each figure is CUDA events
around >= 200 launches after a warm-up of every set. Reports time, GFLOP/s (2 nnz k / t) and bench.py's algorithmic-bytes
fraction (A's CSR arrays + B once + C once over the HBM peak), the check time of spmm_csr_build_bsr, and checks every arm's
C against BSR's to 1e-12 relative. One JSON line per figure on stdout (and in --out).

  python tools/bsr_probe.py [--reps 200] [--out FILE] [--skip-large]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

import sparsematrixmultiplicationmpi_b200 as spmm
from sparsematrixmultiplicationmpi_b200 import _cabi, generators as gen

KS = [1, 2, 3, 4, 8, 16, 32, 33, 64, 128]
MATRICES = [  # name, b, mesh nodes, node-level entries
    ("fem3", 3, 40_397, 291_592),
    ("fem4", 4, 30_298, 164_020),
    ("fem6", 6, 20_199, 72_898),
    ("fem3_x10", 3, 403_970, 2_915_920),
]
L2_BYTES = 126 << 20
OUT = None


def emit(**d):
    line = json.dumps(d)
    print(line, flush=True)
    if OUT:
        OUT.write(line + "\n")
        OUT.flush()


def measured_peak_gbs():
    """The HBM peak bench.py divides by (MEASURED_PEAKS.json, else its fallback)."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def algorithmic_bytes(n_rows, nnz, k):
    """bench.py's formula: A's CSR arrays + B once + C once."""
    return nnz * 12 + (n_rows + 1) * 4 + 2 * n_rows * k * 8


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, timeout=60).stdout.strip()
    return out.splitlines()[0] if out else "unknown"


def last_kernel():
    return (_cabi.lib().spmm_last_kernel_name() or b"").decode()


def event_ms(fn, reps):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    for i in range(reps):
        fn(i)
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps


def main():
    global OUT
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--out", default=None)
    ap.add_argument("--skip-large", action="store_true")
    args = ap.parse_args()
    OUT = open(args.out, "a") if args.out else None
    peak, peak_src = measured_peak_gbs()
    emit(card=card(), hbm_peak_gbs=peak, hbm_peak_source=peak_src, reps=args.reps)
    cur = torch.cuda.current_stream().cuda_stream
    for name, b, nodes, node_nnz in MATRICES:
        if args.skip_large and nodes > 100_000:
            continue
        n, nc, r, c, v, sym = gen.fem_blocked(b, nodes, node_nnz, 20)
        with spmm.DeviceCSR.from_coo_host(n, nc, r, c, v, sym, 0) as A0:
            host = A0.download()
        del r, c, v
        nnz = host.nnz
        a_bytes = nnz * 12 + (n + 1) * 4
        # the check pass of spmm_csr_build_bsr: explicit b and the search over 6..2, median of 5
        with spmm.DeviceCSR.from_host(host, 0) as A0:
            for mode in (b, -1):
                ts = []
                for _ in range(6):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    got = A0.build_bsr(mode)
                    ts.append((time.perf_counter() - t0) * 1e3)
                assert got == b, (name, mode, got)
                emit(matrix=name, b=b, what="build_bsr", block_dim=mode, ms_median=float(np.median(ts[1:])))
        for k in KS:
            set_bytes = a_bytes + 2 * n * k * 8
            n_sets = int(min(8, max(2, -(-3 * L2_BYTES // set_bytes))))
            rng = np.random.default_rng(k)
            Bs = [torch.from_numpy(rng.random((nc, k)) + 0.5).cuda() for _ in range(n_sets)]
            Cs = [torch.empty((n, k), dtype=torch.float64, device="cuda") for _ in range(n_sets)]
            X = [spmm.DeviceCSR.from_host(host, 0) for _ in range(n_sets)]  # explicit kernels; BSR view on
            P = [spmm.DeviceCSR.from_host(host, 0) for _ in range(n_sets)]  # AUTO without a view
            for h in X:
                assert h.build_bsr(b) == b
            arms = ["rows", "bsr", "auto"]
            if k % 2 == 0:
                tiles = [h.build_tiles(-1, 0, k) for h in X]
                if tiles[0]["rows_per_tile"] > 0:
                    arms.append("tiled")
            if k in (1, 2, 4, 8):
                arms.append("stream")
            results = {}
            for arm in arms:
                hs = P if arm == "auto" else X
                kern = arm

                def launch(i):
                    j = i % n_sets
                    hs[j].multiply(Bs[j].data_ptr(), k, Cs[j].data_ptr(), kern, cur)

                try:
                    for i in range(12 * n_sets):  # warm-up; AUTO builds its lazy layout on the 9th call of a handle
                        launch(i)
                    torch.cuda.synchronize()
                except _cabi.SpmmError as e:
                    emit(matrix=name, b=b, k=k, arm=arm, skipped=str(e))
                    continue
                kname = last_kernel()
                ms = event_ms(launch, max(args.reps, n_sets))
                launch(0)
                torch.cuda.synchronize()
                results[arm] = Cs[0].cpu().numpy()
                t = ms * 1e-3
                emit(matrix=name, b=b, n_rows=n, nnz=nnz, k=k, arm=arm, kernel=kname, us=ms * 1e3,
                     gflops=2.0 * nnz * k / t / 1e9, alg_frac=algorithmic_bytes(n, nnz, k) / t / 1e9 / peak,
                     operand_sets=n_sets, set_mb=set_bytes / 1e6)
            ref = results.get("bsr")
            for arm, got in results.items():
                # per entry |x - bsr| <= 1e-12 |bsr| (the empty rows of the mesh give exact zeros in every arm)
                err, scale = np.abs(got - ref), np.abs(ref)
                ok = bool((err <= 1e-12 * scale).all())
                rel = float(np.max(err[scale > 0] / scale[scale > 0]))
                emit(matrix=name, k=k, arm=arm, check="max_rel_vs_bsr", value=rel, ok=ok)
            for h in X + P:
                h.close()
            del Bs, Cs, results
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
