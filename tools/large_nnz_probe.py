#!/usr/bin/env python
"""What segmentation costs: handles with 64-bit row offsets (spmm_csr_create_device64) against int32 handles, time per
non-zero of one multiply, timed with CUDA events. One JSON line per figure; profiles/r3_large_nnz.md holds a run.

Matrices (banded, 33 entries per row):
  big64     2^26 rows, 2,214,592,512 non-zeros, 64-bit handle (3 segments of at most 2^30)
  half64    2^25 rows of the same closed form, 64-bit handle (2 segments)
  half32    the same 2^25 rows as an int32 handle: the same matrix as half64, without segments
  banded32  spmm_gen_banded(2^25, 33, half bandwidth 16): the library's own banded generator, int32 handle
Closed form: columns (r + j - 16) mod n, values 1 + ((33 r + j) mod 7) / 8, j = 0..32. Each timed launch uses the next
of two (B, C) pairs; every operand is larger than the 126 MB of L2, so nothing is re-read from L2 across launches.

  python tools/large_nnz_probe.py [--reps 10] [--out large_nnz.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

import sparsematrixmultiplicationmpi_b200 as spmm
from sparsematrixmultiplicationmpi_b200 import _cabi

W = 33
KS = (1, 8, 16)
KERNELS = ("auto", "rows", "merge")
OUT = None


def emit(**d):
    line = json.dumps(d)
    print(line, flush=True)
    if OUT:
        with open(OUT, "a") as f:
            f.write(line + "\n")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out.splitlines()[0]
    except Exception as e:
        return f"nvidia-smi failed: {e}"


def closed_form(n, rowptr_dtype):
    """rowptr, colidx, vals of the banded closed form on the device, built in row chunks."""
    nnz = n * W
    rowptr = torch.arange(n + 1, dtype=torch.int64, device="cuda") * W
    colidx = torch.empty(nnz, dtype=torch.int32, device="cuda")
    vals = torch.empty(nnz, dtype=torch.float64, device="cuda")
    j = torch.arange(W, dtype=torch.int64, device="cuda")
    step = 1 << 22
    for r0 in range(0, n, step):
        r = torch.arange(r0, min(n, r0 + step), dtype=torch.int64, device="cuda")[:, None]
        colidx[r0 * W:(r0 + r.shape[0]) * W] = ((r + j - 16) % n).to(torch.int32).reshape(-1)
        vals[r0 * W:(r0 + r.shape[0]) * W] = (1.0 + ((W * r + j) % 7).to(torch.float64) / 8.0).reshape(-1)
    torch.cuda.empty_cache()
    return rowptr.to(rowptr_dtype), colidx, vals


def handle_of(name, n):
    """(DeviceCSR, arrays it borrows)"""
    import ctypes as C
    if name == "banded32":
        return spmm.DeviceCSR.banded(n, W, 16), None
    wide = name.endswith("64")
    rp, ci, va = closed_form(n, torch.int64 if wide else torch.int32)
    if wide:
        return spmm.DeviceCSR.from_csr64(rp, ci, va, n, n, copy=False), (rp, ci, va)
    h = C.c_void_p()
    _cabi.check(_cabi.lib().spmm_csr_create_device(0, n, n, n * W, C.c_void_p(rp.data_ptr()), C.c_void_p(ci.data_ptr()),
                                                   C.c_void_p(va.data_ptr()), 0, C.byref(h)))
    return spmm.DeviceCSR(h.value, owner=(rp, ci, va)), (rp, ci, va)


def time_handle(name, A, pairs, reps):
    stream = torch.cuda.current_stream().cuda_stream
    n = A.n_rows
    for k in KS:
        views = [(B[:n * k].view(n, k), Cm[:n * k].view(n, k)) for B, Cm in pairs]
        for kernel in KERNELS:
            def launch(i):
                B, Cm = views[i % len(views)]
                A.multiply(B.data_ptr(), k, Cm.data_ptr(), kernel, stream)
            for i in range(3):
                launch(i)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            s.record()
            for i in range(reps):
                launch(i)
            e.record()
            torch.cuda.synchronize()
            ms = s.elapsed_time(e) / reps
            emit(matrix=name, n_rows=n, nnz=A.nnz, k=k, kernel=kernel, ran=_cabi.lib().spmm_last_kernel_name().decode(),
                 ms=ms, ns_per_nnz=ms * 1e6 / A.nnz)


def main():
    global OUT
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    OUT = args.out
    if OUT:
        os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
    assert torch.cuda.is_available(), "this probe measures on a CUDA device"
    free, total = torch.cuda.mem_get_info()
    emit(card=card(), device=torch.cuda.get_device_name(0), free_gib=free / 2**30, total_gib=total / 2**30)
    big = 1 << 26
    kmax = max(KS)
    # two (B, C) pairs at the widest k; narrower k use a contiguous prefix. Element e of B is (3 e) mod 11 - 5
    pairs = []
    step = 1 << 26
    for _ in range(2):
        B = torch.empty(big * kmax, dtype=torch.float64, device="cuda")
        for e0 in range(0, B.numel(), step):
            e = torch.arange(e0, min(B.numel(), e0 + step), dtype=torch.int64, device="cuda")
            B[e0:e0 + e.numel()] = ((3 * e) % 11 - 5).to(torch.float64)
        pairs.append((B, torch.empty(big * kmax, dtype=torch.float64, device="cuda")))
    torch.cuda.empty_cache()
    results = {}
    for name, n in (("big64", big), ("half64", big // 2), ("half32", big // 2), ("banded32", big // 2)):
        A, keep = handle_of(name, n)
        time_handle(name, A, pairs, args.reps)
        if name in ("half64", "half32"):
            Cm = torch.empty((n, 8), dtype=torch.float64, device="cuda")
            A.multiply(pairs[0][0][:n * 8].data_ptr(), 8, Cm.data_ptr(), "rows")
            results[name] = Cm.cpu()
            del Cm
        A.close()
        del A, keep
        torch.cuda.empty_cache()
    emit(check="half64 and half32 give the same C at k = 8 (row kernel), bit for bit",
         equal=bool(torch.equal(results["half64"], results["half32"])))


if __name__ == "__main__":
    main()
