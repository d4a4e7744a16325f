"""bench.py's command line: the reference arm runs on host cores only, so its JSON contract is checked here without a
GPU; --dump-outputs is checked against the oracle on the GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import REL_TOL, ROOT, assert_close_rel


def test_reference_arm_prints_one_contract_line():
    """Times the compiled reference where oracle/_ref is built, else the oracle's restatement of it."""
    import pyoracle
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, res.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1
    assert d["unit"] == "GFLOP/s" and d["higher_is_better"] is True and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert d["vs_baseline"] is None and "workload" in d["config"] and "k=64" in d["config"]["workload"]
    assert d["value"] > 0 and d["ms_per_step"] > 0
    # 2 * nnz * k / t on the full cfg2 multiply
    assert abs(d["value"] - 2 * 2624331 * 64 / (d["ms_per_step"] * 1e-3) / 1e9) <= 1e-6 * d["value"]
    cb = d["cpu_baseline"]
    kind = "reference" if pyoracle.Reference.available() else "port"
    assert cb["kind"] == kind and cb["cores"] >= 1 and cb["sample"] and cb["value"] == d["value"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    assert d.get("gpu_launches", 0) == 0


def test_dump_output_samples_rows_above_the_budget(tmp_path):
    import bench
    C = np.arange(1000 * 8, dtype=np.float64).reshape(1000, 8)
    bench.dump_output(str(tmp_path / "full.npy"), C, C.nbytes)
    assert np.array_equal(np.load(tmp_path / "full.npy"), C)
    for name in ("a", "b"):
        bench.dump_output(str(tmp_path / f"{name}.npy"), C, 100 * 8 * 8)
    a, b = np.load(tmp_path / "a.npy"), np.load(tmp_path / "b.npy")
    assert a.shape == (100, 8) and np.array_equal(a, b)  # the same rows every time
    rows = a[:, 0] / 8
    assert np.all(np.diff(rows) > 0) and np.array_equal(a, C[rows.astype(int)])


@pytest.mark.parametrize("args", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_rejects_bad_arguments(args):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=120)
    assert res.returncode == 2 and not res.stdout, res.stderr[-1000:]


@pytest.mark.gpu
def test_bench_dump_outputs_is_the_product(oracle, tmp_path):
    """--dump-outputs writes the C of the last timed step: A (seed 20) times the seeded B of that step's operand set."""
    import torch
    from sparsematrixmultiplicationmpi_b200 import generators as gen
    steps, k = 3, 64
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--no-extras",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    d = json.loads(res.stdout)
    assert d["steps"] == steps and d["gpu_launches"] == steps
    assert os.listdir(tmp_path) == ["C.npy"]
    got = np.load(tmp_path / "C.npy")
    n, _, r, c, v, sym = gen.cop20k_A_shaped(seed=20)
    rp, ci, va = oracle.csr_from_coo(n, r, c, v, sym)
    g = torch.Generator(device="cuda")
    g.manual_seed((steps - 1) % 4)  # operand set of the last step, rank 0
    B = torch.randint(1, 101, (n, k), device="cuda", generator=g).double().cpu().numpy()
    assert got.dtype == np.float64 and got.shape == (n, k)
    assert_close_rel(got, oracle.spmm(rp, ci, va, B, k), tol=REL_TOL)  # positive A and B: no cancellation


def test_plot_tool_writes_the_four_families(tmp_path):
    """tools/plot_results.py: execution time, speed-up, performance, efficiency (the reference notebook's families) as SVG."""
    out = tmp_path / "plots"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "plot_results.py"), os.path.join(ROOT, "profiles", "r1_results.csv"),
                          "--matrix", "cfg1", "--out", str(out)], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr[-1000:]
    names = sorted(os.listdir(out))
    for family in ("execution_time", "speedup", "performance", "efficiency"):
        assert any(family in n for n in names), names
    assert open(out / names[0]).read().startswith("<svg")
