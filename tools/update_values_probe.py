#!/usr/bin/env python
"""Cost of new values for a resident matrix on cfg2 (cop20k_A-shaped, k = 64, tile layout built the way AUTO builds it):
the device and host forms of spmm_csr_update_values_*, the path they replace (close + from_host + build_tiles), the multiply
before and after an update, and 50 time steps of (update, multiply) against (new handle, multiply). One JSON line per figure.

  python tools/update_values_probe.py [--reps 200] [--steps 50]
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

K = 64


def emit(**d):
    print(json.dumps(d), flush=True)


def measured_peak_gbs():
    """The HBM peak bench.py divides by (MEASURED_PEAKS.json, else its fallback)."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def power_limit_w():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except Exception:
        return None


def event_ms(fn, reps):
    """Mean device time of fn() over reps launches, CUDA events around the whole batch."""
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    for i in range(reps):
        fn(i)
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps


def wall_ms(fn, reps):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(reps):
        fn(i)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--steps", type=int, default=50)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this probe measures on a CUDA device"
    stream = torch.cuda.current_stream().cuda_stream
    emit(device=torch.cuda.get_device_name(0), power_limit_w=power_limit_w())

    n, nc, r, c, v, sym = gen.cop20k_A_shaped()
    with spmm.DeviceCSR.from_coo_host(n, nc, r, c, v, sym, device=0) as A0:
        host = A0.download()
    nnz = host.nnz
    rng = np.random.default_rng(1)
    B = torch.from_numpy(rng.integers(1, 101, (n, K)).astype(np.float64)).cuda()
    Cm = torch.empty((n, K), dtype=torch.float64, device="cuda")

    def new_host(i):
        return spmm.SparseMatrix(0.5 + np.random.default_rng(100 + i).random(nnz), host.colIndices, host.rowPtr, n, n)

    A = spmm.DeviceCSR.from_host(host, 0)
    info = A.build_tiles(-1, 0, K)

    def mult(_=0):
        A.multiply(B.data_ptr(), K, Cm.data_ptr(), "auto", stream)

    for _ in range(20):
        mult()
    before_ms = event_ms(mult, args.reps)
    before_kernel = _cabi.lib().spmm_last_kernel_name().decode()
    emit(what="multiply before update", ms=before_ms, kernel=before_kernel, tile_info=info, n=n, nnz=nnz, k=K)

    # device form: sources rotated over more than the 126 MB of L2, so that each update reads its source from HBM
    n_src = int(np.ceil(160e6 / (8 * nnz)))
    srcs = [torch.from_numpy(0.5 + np.random.default_rng(200 + i).random(nnz)).cuda() for i in range(n_src)]
    upd = lambda i: A.update_values(srcs[i % n_src], stream)
    for i in range(2 * n_src):
        upd(i)
    dev_ms = event_ms(upd, args.reps)
    moved = 3 * 8 * nnz  # each value read once, written to the CSR array and to the layout
    peak, peak_src = measured_peak_gbs()
    gbs = moved / dev_ms / 1e6
    emit(what="device-form update", ms=dev_ms, bytes=moved, gbs=gbs, hbm_peak_gbs=peak, peak_source=peak_src,
         frac_of_peak=gbs / peak, sources=n_src, source_bytes_total=n_src * 8 * nnz,
         note="sources rotated over more than L2 (126 MB); the two destinations (2 x 8 nnz bytes) are the same every call")
    p = C.c_void_p()
    _cabi.check(_cabi.lib().spmm_csr_device_ptrs(A.handle, None, None, C.byref(p)))

    class View:
        __cuda_array_interface__ = {"shape": (nnz,), "typestr": "<f8", "data": (p.value, False), "version": 3}
    own = torch.as_tensor(View(), device="cuda")
    inplace_ms = event_ms(lambda i: A.update_values(own, stream), args.reps)
    emit(what="device-form update, values edited in place (layout only)", ms=inplace_ms, bytes=2 * 8 * nnz,
         gbs=2 * 8 * nnz / inplace_ms / 1e6, note="source and destination together 42 MB: partly L2-resident")

    # host form: wall clock to completion
    pinned = torch.empty(nnz, dtype=torch.float64).pin_memory().numpy()
    pinned[:] = 0.5 + np.random.default_rng(300).random(nnz)
    pageable = 0.5 + np.random.default_rng(301).random(nnz)
    for name, src in (("pinned", pinned), ("pageable", pageable)):
        A.update_values(src)
        ms = wall_ms(lambda i: A.update_values(src), 20)
        emit(what=f"host-form update ({name} source)", ms=ms, bytes_over_pcie=8 * nnz, gbs_pcie=8 * nnz / ms / 1e6)

    after_ms = event_ms(mult, args.reps)
    after_kernel = _cabi.lib().spmm_last_kernel_name().decode()
    emit(what="multiply after update", ms=after_ms, kernel=after_kernel, tile_info=A.tile_info(),
         same_kernel=after_kernel == before_kernel, same_layout=A.tile_info() == info)

    # the path the update replaces: a new handle (upload + schedule) and the layout AUTO would build
    def rebuild(i):
        nonlocal A
        A.close()
        A = spmm.DeviceCSR.from_host(host, 0)
        A.build_tiles(-1, 0, K)
    rebuild_ms = wall_ms(rebuild, 5)
    emit(what="close + from_host + build_tiles(-1, 0, 64)", ms=rebuild_ms)

    # 50 time steps of an iterative caller: new values from the host each step, then one multiply
    mats = [new_host(i) for i in range(args.steps)]
    for m in mats[:3]:
        A.update_values(m.values)
        mult()
    upd_step = wall_ms(lambda i: (A.update_values(mats[i].values), mult()), args.steps)
    upd_kernel = _cabi.lib().spmm_last_kernel_name().decode()
    dsrc = [torch.from_numpy(m.values).cuda() for m in mats[:n_src]]
    dev_step = wall_ms(lambda i: (A.update_values(dsrc[i % n_src], stream), mult()), args.steps)
    A.close()
    state = {"A": None}

    def fresh_step(i):
        if state["A"] is not None:
            state["A"].close()
        state["A"] = spmm.DeviceCSR.from_host(mats[i], 0)
        state["A"].multiply(B.data_ptr(), K, Cm.data_ptr(), "auto", stream)
    fresh_step(0)
    fresh_ms = wall_ms(fresh_step, args.steps)
    fresh_kernel = _cabi.lib().spmm_last_kernel_name().decode()
    state["A"].close()
    emit(what=f"{args.steps} steps of (host-form update, multiply)", ms_per_step=upd_step, kernel=upd_kernel)
    emit(what=f"{args.steps} steps of (device-form update, multiply)", ms_per_step=dev_step, kernel=upd_kernel,
         note="sources already on the device")
    emit(what=f"{args.steps} steps of (new handle from_host, multiply)", ms_per_step=fresh_ms, kernel=fresh_kernel)


if __name__ == "__main__":
    main()
