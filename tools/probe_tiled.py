#!/usr/bin/env python
"""Where the tiled kernel's time goes on cfg2 (cop20k_A shape): cold / warm operands and launch knobs side by side.

    python tools/probe_tiled.py [--k 64] [--iters 200] [--out gpurun_out/probe_tiled.jsonl]

Every line: the mean launch time (CUDA events, `iters` back-to-back launches) of the tiled kernel with
  * all operands rotating over 4 resident sets (cold: what bench.py times),
  * the same B for every launch (B stays in L2; A's layout and C rotate),
  * one operand set only (everything that fits stays in L2),
for each setting of the launch knobs given by --knobs (comma separated key=value groups joined by '+').
Results are checked against the row kernel once per knob setting (max relative difference printed).
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import sparsematrixmultiplicationmpi_b200 as spmm  # noqa: E402
from sparsematrixmultiplicationmpi_b200 import _cabi, generators as gen  # noqa: E402


def timed(fn, iters, warmup=12):
    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        fn(i)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--k", type=int, default=64)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--sets", type=int, default=4)
    ap.add_argument("--knobs", default="")
    ap.add_argument("--build", default="", help="build knobs, e.g. tiled.depth=3+tiled.group=2 (applied while the layouts are built)")
    ap.add_argument("--tile", default="-1x0", help="rows_per_tile x box_rows of the layout")
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "probe_tiled.jsonl"))
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    k = args.k
    n, nc, r, c, v, sym = gen.cop20k_A_shaped()
    first = spmm.DeviceCSR.from_coo_host(n, nc, r, c, v, sym, device=0)
    host = first.download()
    T, BR = [int(x) for x in args.tile.split("x")]
    sets = []
    _cabi.tune("reset", 0)
    for kv in [x for x in args.build.split("+") if x]:
        key, val = kv.split("=")
        _cabi.tune(key, int(val))
    for s in range(args.sets):
        A = spmm.DeviceCSR.from_host(host, 0)
        A.build_tiles(T, BR, k)
        sets.append((A, torch.randint(1, 101, (n, k), device=dev).double(), torch.empty((n, k), dtype=torch.float64, device=dev)))
    _cabi.tune("reset", 0)
    info = sets[0][0].tile_info()
    stream = torch.cuda.current_stream().cuda_stream
    ref = torch.empty((n, k), dtype=torch.float64, device=dev)
    sets[0][0].multiply(sets[0][1].data_ptr(), k, ref.data_ptr(), "rows", stream)
    out = open(args.out, "a")
    for group in args.knobs.split(","):
        _cabi.tune("reset", 0)
        for kv in [x for x in group.split("+") if x]:
            key, val = kv.split("=")
            _cabi.tune(key, int(val))

        def cold(i):
            A, B, C = sets[i % len(sets)]
            A.multiply(B.data_ptr(), k, C.data_ptr(), "tiled", stream)

        def warm_b(i):
            A, _, C = sets[i % len(sets)]
            A.multiply(sets[0][1].data_ptr(), k, C.data_ptr(), "tiled", stream)

        def one_set(i):
            A, B, C = sets[0]
            A.multiply(B.data_ptr(), k, C.data_ptr(), "tiled", stream)

        rec = {"k": k, "knobs": group or "default", "build": args.build, "tiles": info,
               "cold_us": timed(cold, args.iters), "warm_B_us": timed(warm_b, args.iters), "one_set_us": timed(one_set, args.iters)}
        torch.cuda.synchronize()
        C0 = sets[0][2]
        rec["max_rel_diff_vs_rows"] = float(((C0 - ref).abs() / ref.abs().clamp_min(1e-300)).max())
        print(json.dumps(rec), flush=True)
        out.write(json.dumps(rec) + "\n")
    _cabi.tune("reset", 0)
    out.close()


if __name__ == "__main__":
    main()
