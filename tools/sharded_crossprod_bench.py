#!/usr/bin/env python
"""crossprod() on several GPUs of one process: sb200_sharded_crossprod through ShardedHostMatrix, beside the one-GPU
sb200_crossprod.

    python tools/sharded_crossprod_bench.py [--shapes C1,C2cut] [--worlds 1,2,4,8] [--shared-worlds 2]
                                            [--out profiles/r05/sharded_crossprod.jsonl]

Shapes: C1 (10k x 10k, d = 0.01, 800 MB result) and C2's structure cut to 40 000 columns (1M x 40k, d = 1e-3, 12.8 GB
result).  The matrices are generated on the device and downloaded once: the host forms take host arrays.  For every
(shape, path, W, out) one JSON line holds:
  * wall_ms_median / wall_ms_best: the host-form call into `out`, a pageable numpy array or pinned host memory;
  * device_ms_median: the device part.  Sharded: from the first push of the row gather to every slab complete,
    CUDA-event time per device, max over devices (the library reports it under SB200_TRACE=1).  One GPU:
    sb200_crossprod_dev into a device buffer between CUDA events (zero-fill, atomics and mirror pass);
  * bits_equal_w1: the result of every sharded series equals the sharded W = 1 result bit for bit (NaN-free data);
    the one-GPU path, which adds in another order, reports max_rel_diff_w1 instead.
Paths: "one-gpu" (sb200_crossprod on a resident mirror that keeps its row-ordered copy), "distinct" (W blocks on GPUs
0 .. W-1, as far as the machine has them) and "shared" (W blocks on GPU 0: the split's overhead, not scaling).
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
    return [float(m) for m in re.findall(r"sharded crossprod: device part ([0-9.]+) ms", text)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="C1,C2cut")
    ap.add_argument("--worlds", default="1,2,4,8")
    ap.add_argument("--shared-worlds", default="2")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05", "sharded_crossprod.jsonl"))
    a = ap.parse_args()
    import torch

    from rcppsparse_b200 import DeviceMatrix, ShardedHostMatrix, _lib, synth

    if not torch.cuda.is_available():
        raise SystemExit("sharded_crossprod_bench: no CUDA device (the measurement needs the GPU; there is no CPU fallback)")
    n_dev = _lib.device_count()
    placements = [("distinct", w) for w in (int(s) for s in a.worlds.split(",")) if w <= n_dev]
    placements += [("shared", w) for w in (int(s) for s in a.shared_worlds.split(",") if s)]
    assert placements and placements[0] == ("distinct", 1), "the W = 1 handle comes first: it gives the reference result"
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    out_file = open(a.out, "a")
    gpu = card()

    def emit(rec):
        rec = dict(rec, gpu=gpu, gpus_present=n_dev)
        print(json.dumps(rec), flush=True)
        out_file.write(json.dumps(rec) + "\n")
        out_file.flush()

    for shape in a.shapes.split(","):
        spec = synth.config("C1") if shape == "C1" else synth.config("C2", 0.4)
        reps, warmup = (10, 3) if shape == "C1" else (3, 1)  # a C2cut call moves 12.8 GB to the host
        with DeviceMatrix.synth(spec) as D:
            i, p, x = D.download_columns()
        nrow, ncol, N = spec.nrow, spec.ncol, len(x)
        base = {"shape": shape, "workload": spec.name, "nnz": N, "nrow": nrow, "ncol": ncol,
                "result_bytes": 8 * ncol * ncol, "reps": reps, "warmup": warmup}
        row_len = np.bincount(i, minlength=nrow).astype(np.float64)
        base["pairs"] = int((row_len * row_len).sum())  # products the sharded sweep forms in all (full columns)
        outs = {"pageable": np.empty((ncol, ncol)), "pinned": torch.empty((ncol, ncol), dtype=torch.float64, pin_memory=True).numpy()}
        ref = None

        def timed(f, out):
            for _ in range(warmup):
                f(out)
            ms = []
            for _ in range(reps):
                t0 = time.perf_counter()
                f(out)
                ms.append((time.perf_counter() - t0) * 1e3)
            return ms

        # sharded, W = 1 first (the reference bits), then every other placement
        for placement, W in placements:
            devices = [0] * W if placement == "shared" else None
            with ShardedHostMatrix(i, p, x, nrow, ncol, W, devices=devices) as S:
                L, h = _lib.lib(), S._h
                equal = {"ok": True, "calls": 0}

                def call(out):
                    _lib.check(L.sb200_sharded_crossprod(h, out.ctypes.data))

                for kind, out in outs.items():
                    ms = timed(call, out)
                    if ref is None:
                        ref = out.copy()
                    equal["ok"] &= bool(np.array_equal(out.view(np.uint64), ref.view(np.uint64)))
                    equal["calls"] += 1
                    dev = device_parts(lambda: call(out), reps) if kind == "pageable" else []
                    emit(dict(base, path="sharded", placement=placement, W=W, out=kind,
                              wall_ms_median=round(statistics.median(ms), 3), wall_ms_best=round(min(ms), 3),
                              device_ms_median=round(statistics.median(dev), 3) if dev else None,
                              device_ms_best=round(min(dev), 3) if dev else None, bits_equal_w1=equal["ok"]))
                    out.fill(0.0)
        # one GPU, today's path: a resident mirror (its row-ordered copy is built on the first call and kept)
        with DeviceMatrix.from_host(i, p, x, nrow, ncol) as M:
            for kind, out in outs.items():
                ms = timed(lambda o: _lib.check(_lib.lib().sb200_crossprod(M._h, o.ctypes.data)), out)
                step = max(1, ncol // 16)  # in column chunks: no second full-size temporary
                rel = max(float(np.max(np.abs(out[c:c + step] - ref[c:c + step]), initial=0.0)) for c in range(0, ncol, step))
                rel /= max(1e-300, float(np.max(np.abs(ref))))
                dev = []
                if kind == "pageable":
                    d = torch.empty((ncol, ncol), dtype=torch.float64, device="cuda:0")
                    for _ in range(warmup):
                        M.crossprod_dev(d)
                    torch.cuda.synchronize()
                    for _ in range(reps):
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        M.crossprod_dev(d)
                        torch.cuda.synchronize()  # the mirror runs on its own stream: wait for it before the end event
                        e1.record()
                        e1.synchronize()
                        dev.append(e0.elapsed_time(e1))
                    del d
                emit(dict(base, path="one-gpu", placement="sb200_crossprod", W=1, out=kind,
                          wall_ms_median=round(statistics.median(ms), 3), wall_ms_best=round(min(ms), 3),
                          device_ms_median=round(statistics.median(dev), 3) if dev else None,
                          device_ms_best=round(min(dev), 3) if dev else None, max_rel_diff_w1=rel))
        del outs, ref


if __name__ == "__main__":
    main()
