#!/usr/bin/env python
"""colVars / rowVars beside colMeans / rowMeans at C2 (1M x 100k, d = 1e-3, 10^8 entries), device forms.

    python tools/vars_bench.py [--config C2] [--reps 10] [--warmup 3] [--out profiles/r06/vars.jsonl]

The matrix is generated on the device.  Every op is timed with CUDA events around its device-form call on the mirror's
stream: `warmup` calls first, then the median and the best of `reps` calls.  Two layouts:
  * "csc": the CSC arrays, the row-ordered copy pinned off (rowVars / rowMeans on the path row_path() reports);
  * "row copy": the same mirror with its row-ordered copy built (rowVars / rowMeans sweep it like a column sum).
For every op the line holds its bytes and the rate they give over the 7.7 TB/s of a B200's HBM3e:
  * compulsory: every array once and the output once (sb200_algorithmic_bytes; colVars 8N + 4(n+1) + 8n);
  * two_pass: what the two passes must move: x (and for rows on the CSC arrays i) read twice, p read twice, the means
    written, read back, and the output written.
The inputs (1.2 GB) exceed the 126 MB L2, which is not flushed between calls.  Before timing, colVars / rowVars of the
first columns / rows are checked against a float64 two-pass on the host.  Every line records the card and its power
limit.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
HBM_BYTES_PER_S = 7.7e12  # NVIDIA B200 data sheet, one GPU


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def timed(fn, reps, warmup, stream):
    import torch

    for _ in range(warmup):
        fn()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        fn()
        b.record(stream)
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return statistics.median(ms), min(ms)


def host_vars(i, p, x, n, m, axis):
    """float64 two-pass variances of the first m columns (axis 0: i, p, x of those columns) or of rows 0 .. m-1 (axis 1:
    all entries, grouped by row)."""
    group = np.repeat(np.arange(len(p) - 1), np.diff(p)) if axis == 0 else i
    keep = group < m
    g, v = group[keep], x[keep]
    cnt = np.bincount(g, minlength=m)
    mean = np.bincount(g, weights=v, minlength=m) / n
    S = np.bincount(g, weights=(v - mean[g]) ** 2, minlength=m)
    return (S + (n - cnt) * mean * mean) / (n - 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="C2")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06", "vars.jsonl"))
    a = ap.parse_args()
    import torch

    from rcppsparse_b200 import DeviceMatrix, synth

    if not torch.cuda.is_available():
        raise SystemExit("vars_bench: no CUDA device (the measurement needs the GPU; there is no CPU fallback)")
    assert a.reps >= 10 and a.warmup >= 3
    gpu = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    out = open(a.out, "a")

    def emit(d):
        d = dict(d, card=gpu)
        print(json.dumps(d), flush=True)
        out.write(json.dumps(d) + "\n")

    spec = synth.config(a.config)
    D = DeviceMatrix.synth(spec)
    stream = torch.cuda.current_stream()
    D.set_stream(stream.cuda_stream)
    N, nrow, ncol = D.nnz, D.nrow, D.ncol
    D.row_companion(-1)

    # correctness first: the first 2000 columns / the rows of the first 4000 columns' entries against a host two-pass
    cv = torch.empty(ncol, dtype=torch.float64, device="cuda")
    rv = torch.empty(nrow, dtype=torch.float64, device="cuda")
    D.col_vars_dev(cv)
    D.row_vars_dev(rv)
    D.sync()
    i, p, x = D.download_columns(0, 2000)
    want = host_vars(i, p, x, nrow, 2000, 0)
    col_err = float(np.max(np.abs(cv[:2000].cpu().numpy() - want) / np.abs(want)))
    i, p, x = D.download_columns()
    want = host_vars(i, p, x, ncol, 4000, 1)
    row_err = float(np.max(np.abs(rv[:4000].cpu().numpy() - want) / np.abs(want)))
    del i, p, x
    emit({"config": a.config, "check": "against a float64 two-pass on the host", "colVars_max_rel_diff": col_err,
          "rowVars_max_rel_diff": row_err})
    assert col_err < 1e-12 and row_err < 1e-12

    col_compulsory = D.algorithmic_bytes("col_vars")
    col_two_pass = 16 * N + 8 * (ncol + 1) + 24 * ncol
    for layout in ("csc", "row copy"):
        if layout == "row copy":
            D.row_companion(1)
        row_path = D.row_path()
        if layout == "csc":
            row_compulsory, row_two_pass = D.algorithmic_bytes("row_vars"), 24 * N + 24 * nrow
        else:
            row_compulsory, row_two_pass = D.algorithmic_bytes("row_sums_companion"), 16 * N + 8 * (nrow + 1) + 24 * nrow
        ops = [("colMeans", lambda: D.col_sums_dev(cv, float(nrow)), D.algorithmic_bytes("col_means"), None),
               ("colVars", lambda: D.col_vars_dev(cv), col_compulsory, col_two_pass),
               ("rowMeans", lambda: D.row_sums_dev(rv, float(ncol)),
                D.algorithmic_bytes("row_means" if layout == "csc" else "row_means_companion"), None),
               ("rowVars", lambda: D.row_vars_dev(rv), row_compulsory, row_two_pass)]
        if layout == "row copy":
            ops = [o for o in ops if o[0].startswith("row")]  # the column ops do not read the copy
        for name, fn, compulsory, two_pass in ops:
            med, best = timed(fn, a.reps, a.warmup, stream)
            line = {"config": a.config, "nrow": nrow, "ncol": ncol, "nnz": N, "layout": layout, "op": name,
                    "row_path": row_path if name.startswith("row") else None, "reps": a.reps, "warmup": a.warmup,
                    "ms_median": round(med, 4), "ms_best": round(best, 4), "compulsory_bytes": compulsory,
                    "compulsory_frac_of_hbm_peak_at_median": round(compulsory / (med * 1e-3) / HBM_BYTES_PER_S, 3)}
            if two_pass is not None:
                line.update(two_pass_bytes=two_pass, two_pass_frac_of_hbm_peak_at_median=round(two_pass / (med * 1e-3) / HBM_BYTES_PER_S, 3))
            emit(line)
    D.close()
    out.close()


if __name__ == "__main__":
    main()
