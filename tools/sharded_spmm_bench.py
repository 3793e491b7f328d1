#!/usr/bin/env python
"""Block products on several GPUs of one process: sb200_sharded_spmm / sb200_sharded_spmm_t through ShardedHostMatrix.

    python tools/sharded_spmm_bench.py [--configs C2,C4] [--c4-scale 0.25] [--ks 8,16,64] [--worlds 1,2,4,8]
                                       [--shared-worlds 2] [--reps 10] [--warmup 3] [--out profiles/r04/sharded_spmm.jsonl]

The matrices are generated on the device and downloaded once: the host form takes host arrays.  C4 runs at a stated
column scale (--c4-scale; its full 24 GB of i/x would have to sit in host memory beside B and Y).  For every
(config, W, regime, op, k) one JSON line holds:
  * wall_ms_median / wall_ms_best: the host-form call, B and Y pageable numpy arrays, >= 3 warm-ups, >= 10 timed calls;
  * device_ms_median: the device part, from every block's operand resident to every result piece complete, CUDA-event
    time per device, max over devices (the library reports it under SB200_TRACE=1), median over the timed calls;
  * reduce_bytes_per_device: 8 nrow k (W - 1) / W, what A B's reduce reads over peer memory per device;
  * bad_entries: outputs outside 1e-12 * sum |a b| of the W = 1 result of the same run (sum |a b| from a handle of |A|),
    summed over every call of the series (warm-ups, timed calls and traced calls; checked after the clock stops);
    checked_calls says how many.
Regimes: "csc" (every block on its CSC arrays; A B with L2 reductions) and "rows" (every block with its row-ordered
copy).  W runs over distinct GPUs as far as the machine has them; --shared-worlds adds handles whose W blocks share
GPU 0 (every multi-block code path, no extra hardware: a measure of the split's overhead, not of scaling).
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def device_parts(fn, n):
    """n calls of fn with SB200_TRACE=1, the library's stderr captured: the 'device part' of each call, in ms."""
    sys.stderr.flush()
    with tempfile.TemporaryFile() as f:
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        os.environ["SB200_TRACE"] = "1"
        try:
            for _ in range(n):
                fn()
        finally:
            del os.environ["SB200_TRACE"]
            os.dup2(saved, 2)
            os.close(saved)
        f.seek(0)
        text = f.read().decode(errors="replace")
    return [float(m) for m in re.findall(r"device part ([0-9.]+) ms", text)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="C2,C4")
    ap.add_argument("--c4-scale", type=float, default=0.25)
    ap.add_argument("--ks", default="8,16,64")
    ap.add_argument("--worlds", default="1,2,4,8")
    ap.add_argument("--shared-worlds", default="2")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04", "sharded_spmm.jsonl"))
    a = ap.parse_args()
    import torch

    from rcppsparse_b200 import DeviceMatrix, ShardedHostMatrix, _lib, synth

    if not torch.cuda.is_available():
        raise SystemExit("sharded_spmm_bench: no CUDA device (the measurement needs the GPU; there is no CPU fallback)")
    reps, warmup = max(10, a.reps), max(3, a.warmup)
    ks = [int(k) for k in a.ks.split(",")]
    n_dev = _lib.device_count()
    placements = [("distinct", w) for w in (int(s) for s in a.worlds.split(",")) if w <= n_dev]
    placements += [("shared", w) for w in (int(s) for s in a.shared_worlds.split(",") if s)]
    assert placements and placements[0] == ("distinct", 1), "the W = 1 handle comes first: it gives the reference results"
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    out = open(a.out, "a")
    gpu = card()

    def emit(rec):
        rec = dict(rec, gpu=gpu, gpus_present=n_dev)
        print(json.dumps(rec), flush=True)
        out.write(json.dumps(rec) + "\n")
        out.flush()

    for cfg in a.configs.split(","):
        scale = a.c4_scale if cfg == "C4" else 1.0
        spec = synth.config(cfg, scale)
        with DeviceMatrix.synth(spec) as D:
            i, p, x = D.download_columns()
        nrow, ncol, N = spec.nrow, spec.ncol, len(x)
        base = {"config": cfg, "scale": scale, "workload": spec.name, "nnz": N, "nrow": nrow, "ncol": ncol}
        rng = np.random.default_rng(11)
        operands = {(op, k): np.asfortranarray(rng.standard_normal(((ncol if op == "spmm" else nrow), k))) for op in ("spmm", "spmm_t")
                    for k in ks}
        with ShardedHostMatrix(i, p, np.abs(x), nrow, ncol, 1) as Sabs:
            feed = {(op, k): getattr(Sabs, op)(np.abs(B)) for (op, k), B in operands.items()}
        ref = {}
        for placement, W in placements:
            devices = [0] * W if placement == "shared" else None
            with ShardedHostMatrix(i, p, x, nrow, ncol, W, devices=devices) as S:
                for regime in ("csc", "rows"):
                    for w in range(W):  # csc: drop the copy and never build it; rows: build it now
                        for action in ((-1,) if regime == "csc" else (0, 1)):
                            S.block(w).row_companion(action)
                    for op in ("spmm", "spmm_t"):
                        for k in ks:
                            B = operands[(op, k)]
                            f = getattr(S, op)
                            tol = 1e-12 * feed[(op, k)]
                            seen = {"bad": 0, "calls": 0}

                            def check(Y):
                                if (op, k) not in ref:  # the first call of the W = 1 handle
                                    ref[(op, k)] = Y
                                seen["bad"] += int(np.count_nonzero(np.abs(Y - ref[(op, k)]) > tol))
                                seen["calls"] += 1

                            for _ in range(warmup):
                                check(f(B))
                            ms = []
                            for _ in range(reps):
                                t0 = time.perf_counter()
                                Y = f(B)
                                ms.append((time.perf_counter() - t0) * 1e3)
                                check(Y)
                            dev = device_parts(lambda: check(f(B)), reps)
                            emit(dict(base, placement=placement, W=W, regime=regime, op=op, k=k,
                                      wall_ms_median=round(statistics.median(ms), 3), wall_ms_best=round(min(ms), 3),
                                      device_ms_median=round(statistics.median(dev), 3) if dev else None,
                                      device_ms_best=round(min(dev), 3) if dev else None,
                                      reduce_bytes_per_device=(8 * nrow * k * (W - 1) // W) if op == "spmm" else 0,
                                      operand_bytes=8 * B.size, result_bytes=8 * Y.size, reps=reps, warmup=warmup,
                                      bad_entries=seen["bad"], checked_calls=seen["calls"]))
        del operands, feed, ref


if __name__ == "__main__":
    main()
