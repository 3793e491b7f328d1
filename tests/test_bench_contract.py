"""bench.py's JSON contract, checked on CPU through the reference arm; the CUDA arm's output dump needs a GPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*extra, env=None):
    e = dict(os.environ)
    e.update(env or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, env=e,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    return lines


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    lines = run_bench("--impl", "reference", "--steps", "2", "--warmup", "1", "--cpu-cols", "1500")
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "nnz/s" and d["unit"] == "nnz/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None and d["dtype"] == "f64"
    assert d["data"] == "synthetic" and "workload" in d["config"] and d["config"]["workload"].startswith("C2")
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] == 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": "nnz/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    lines = run_bench("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", "--cpu-cols", "500",
                      env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert lines == []


def test_cuda_arm_refuses_to_run_without_a_gpu():
    import torch

    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_steps_results(tmp_path):
    """--dump-outputs writes what the timed step returned: the four reductions of the seeded workload, in float64,
    within the parity bar of the oracle's results on the same matrix."""
    import numpy as np

    from oracle import oracle
    from rcppsparse_b200 import synth

    lines = run_bench("--steps", "3", "--warmup", "1", "--scale", "0.01", "--no-transpose", "--no-products", "--no-e2e",
                      "--no-cpu-baseline", "--no-parity", "--dump-outputs", str(tmp_path))
    assert json.loads(lines[-1])["steps"] == 3
    spec = synth.config("C2", 0.01)
    i, p, x = synth.generate_host(spec)
    args = (i, p, x, spec.nrow, spec.ncol)
    chk = oracle.best()
    assert sorted(f.name for f in tmp_path.iterdir()) == ["colMeans.npy", "colSums.npy", "rowMeans.npy", "rowSums.npy"]
    for op in ("colSums", "rowSums", "colMeans", "rowMeans"):
        got = np.load(tmp_path / f"{op}.npy")
        assert got.dtype == np.float64
        oracle.assert_within(op, got, getattr(chk, op)(*args), *args)


def test_value_before_row_copy_arithmetic():
    """bench.py reports, next to the steady-state value, what the same step does while the row sums are still on
    the scatter kernels; the helper only swaps the row ops' times."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    ops = ("colSums", "rowSums", "colMeans", "rowMeans")
    per_op = {"colSums": 0.1, "rowSums": 0.1, "colMeans": 0.1, "rowMeans": 0.1}
    v = mod.value_before_row_copy(ops, 10**8, per_op, 0.5)
    assert abs(v - 4e8 / 1.2e-3) < 1e-3 * v
    assert mod.value_before_row_copy(("colSums",), 10**8, per_op, 0.5) == 1e8 / 1e-4
