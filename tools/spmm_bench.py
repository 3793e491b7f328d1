#!/usr/bin/env python
"""Sparse x dense block on one GPU: one spmm(_t)_dev call against k spmv(_t)_dev calls on the same mirror.

    python tools/spmm_bench.py [--configs C2,C4] [--ks 1,2,4,8,16,32,64] [--reps 10] [--out profiles/r03/spmm.jsonl]

Matrices are generated on the device.  For each (config, op, k) and regime it times, with CUDA events on the handle's
stream (>= 3 warm-ups, >= 10 timed calls, median and best):
  spmm_t_dev / spmm_dev on the CSC arrays, spmm_dev on the row-ordered copy, k calls of spmv(_t)_dev in the same
  regime, and (reference only) k calls on the resident band-major companions.
Algorithmic bytes 12N + 4(n+1) + 8 nrow k + 8 ncol k against the measured HBM rate, FP64 operations 2Nk.  The timed
outputs are checked against the k single-vector results of the same run (|delta| <= 1e-12 * sum |a b|, the sums from a
mirror of |A|), C2 at k = 8 against the CPU checker, and one non-resident Matrix.spmm from pageable numpy is timed
against 8 Matrix.spmv calls.  One JSON line per measurement.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_GBS = 6530.0  # measured on this project's B200 (DESIGN.md section 5)


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


def abs_mirror(D):
    """A mirror of |A| (same structure, absolute values) for the error bars; built column block by column block."""
    import torch

    from rcppsparse_b200 import DeviceMatrix

    xa = torch.empty(max(D.nnz, 1), dtype=torch.float64, device="cuda")
    pos, step = 0, 50_000
    for c0 in range(0, D.ncol, step):
        _, _, x = D.download_columns(c0, min(D.ncol, c0 + step))
        xa[pos:pos + len(x)] = torch.from_numpy(np.abs(x)).cuda()
        pos += len(x)
    d_i, d_p, _ = D.device_arrays()
    torch.cuda.synchronize()
    return DeviceMatrix.adopt(d_i, d_p, xa[:D.nnz], D.nrow, D.ncol)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="C2,C4")
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--ks", default="1,2,4,8,16,32,64")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03", "spmm.jsonl"))
    a = ap.parse_args()
    import torch

    from oracle import oracle
    from rcppsparse_b200 import Matrix, DeviceMatrix, synth

    if not torch.cuda.is_available():
        raise SystemExit("spmm_bench: no CUDA device (the measurement needs the GPU; there is no CPU fallback)")
    reps, warmup = max(10, a.reps), max(3, a.warmup)
    ks = [int(k) for k in a.ks.split(",")]
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    out = open(a.out, "a")
    gpu = card()

    def emit(rec):
        rec = dict(rec, gpu=gpu)
        print(json.dumps(rec), flush=True)
        out.write(json.dumps(rec) + "\n")
        out.flush()

    stream = torch.cuda.current_stream()
    for cfg in a.configs.split(","):
        spec = synth.config(cfg, a.scale)
        D = DeviceMatrix.synth(spec)
        D.set_stream(stream.cuda_stream)
        Dabs = abs_mirror(D)
        Dabs.set_stream(stream.cuda_stream)
        Dabs.row_companion(-1)
        Dabs.band_companion(0, -1)
        N, nrow, ncol = D.nnz, D.nrow, D.ncol
        base = {"config": cfg, "workload": spec.name, "nnz": N, "nrow": nrow, "ncol": ncol}
        g = torch.Generator(device="cuda").manual_seed(7)

        def check(op, Y, Yk, B, k):
            """Y (k x rows, i.e. column-major) against the k single-vector results, bar from the |A| mirror."""
            feed = torch.empty_like(Y)
            (Dabs.spmm_t_dev if op == "spmv_t" else Dabs.spmm_dev)(B.abs().contiguous(), k, feed)
            torch.cuda.synchronize()
            bad = ((Y - Yk).abs() > 1e-12 * feed) & torch.isfinite(feed)
            return int(bad.sum().item())

        def products(regime, ops):
            for k in ks:
                for op in ops:
                    rows_in, rows_out = (nrow, ncol) if op == "spmv_t" else (ncol, nrow)
                    B = torch.randn((k, rows_in), generator=g, device="cuda", dtype=torch.float64)
                    Y = torch.empty((k, rows_out), device="cuda", dtype=torch.float64)
                    Yk = torch.empty_like(Y)
                    spmm = D.spmm_t_dev if op == "spmv_t" else D.spmm_dev
                    spmv = D.spmv_t_dev if op == "spmv_t" else D.spmv_dev
                    med, best = timed(lambda: spmm(B, k, Y), reps, warmup, stream)

                    def k_calls():
                        for j in range(k):
                            spmv(B[j], Yk[j])

                    kmed, kbest = timed(k_calls, reps, warmup, stream)
                    nbytes = 12 * N + 4 * (ncol + 1) + 8 * nrow * k + 8 * ncol * k
                    emit(dict(base, op="spmm_t" if op == "spmv_t" else "spmm", regime=regime, k=k, ms_median=round(med, 4),
                              ms_best=round(best, 4), k_calls_ms_median=round(kmed, 4), k_calls_ms_best=round(kbest, 4),
                              speedup_median=round(kmed / med, 3), algorithmic_bytes=nbytes,
                              frac_hbm=round(nbytes / (HBM_GBS * 1e6) / med, 3), fp64_ops=2 * N * k,
                              gflops=round(2 * N * k / (med * 1e6), 1), bad_entries=check(op, Y, Yk, B, k)))
                    del B, Y, Yk

        # (a) and (c) on the CSC arrays: no cached layout serves either product
        D.row_companion(-1)
        D.band_companion(0, -1)
        products("csc", ("spmv_t", "spmv"))
        # (b) A B on the row-ordered copy, against k A v on the same copy
        D.row_companion(0)
        t0 = time.perf_counter()
        D.row_companion(1)
        torch.cuda.synchronize()
        emit(dict(base, build="row_companion", ms=round((time.perf_counter() - t0) * 1e3, 2)))
        D.band_companion(1, -1)  # A v stays the gather sweep of the copy
        products("row-companion", ("spmv",))
        # (d) reference only: k single-vector calls on the resident band-major companions
        for which, op in ((0, "spmv_t"), (1, "spmv")):
            t0 = time.perf_counter()
            D.band_companion(which, 0)
            D.band_companion(which, 1)
            torch.cuda.synchronize()
            emit(dict(base, build=f"band_companion({which})", ms=round((time.perf_counter() - t0) * 1e3, 2)))
            spmv = D.spmv_t_dev if op == "spmv_t" else D.spmv_dev
            rows_in, rows_out = (nrow, ncol) if op == "spmv_t" else (ncol, nrow)
            for k in ks:
                B = torch.randn((k, rows_in), generator=g, device="cuda", dtype=torch.float64)
                Yk = torch.empty((k, rows_out), device="cuda", dtype=torch.float64)

                def k_calls():
                    for j in range(k):
                        spmv(B[j], Yk[j])

                kmed, kbest = timed(k_calls, reps, warmup, stream)
                emit(dict(base, op=op, regime="band-major companion, k calls (reference)", k=k, k_calls_ms_median=round(kmed, 4),
                          k_calls_ms_best=round(kbest, 4)))
                del B, Yk

        if cfg == "C2":
            # the CPU checker at k = 8, and the one-shot path: a non-resident Matrix from pageable numpy
            i, p, x = D.download_columns()
            args = (i, p, x, nrow, ncol)
            chk = oracle.best()
            k = 8
            Bh = np.asfortranarray(np.round(np.random.default_rng(8).standard_normal((ncol, k)), 3))
            Bth = np.asfortranarray(np.round(np.random.default_rng(9).standard_normal((nrow, k)), 3))
            worst = 0.0
            D.row_companion(-1)
            Y, Yt = D.spmm(Bh), D.spmm_t(Bth)
            for j in range(k):
                worst = max(worst, oracle.assert_within("spmv", Y[:, j], chk.spmv(*args, Bh[:, j]), *args, v=Bh[:, j]))
                worst = max(worst, oracle.assert_within("spmv_t", Yt[:, j], chk.spmv_t(*args, Bth[:, j]), *args, v=Bth[:, j]))
            emit(dict(base, check=f"{chk.kind} checker, k = 8, spmm and spmm_t on the CSC arrays", worst_err_over_sum_abs=worst))
            A = Matrix(x, i, p, np.array([nrow, ncol], np.int32))
            for name, fn in (("Matrix.spmm(B), k = 8", lambda: A.spmm(Bh)),
                             ("8 x Matrix.spmv(v)", lambda: [A.spmv(Bh[:, j]) for j in range(k)])):
                fn()
                wall = []
                for _ in range(3):
                    t0 = time.perf_counter()
                    fn()
                    wall.append((time.perf_counter() - t0) * 1e3)
                emit(dict(base, one_shot=name, wall_ms_median=round(statistics.median(wall), 2), wall_ms_best=round(min(wall), 2)))
            del A
        Dabs.close()
        D.close()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
    out.close()


if __name__ == "__main__":
    main()
