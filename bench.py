#!/usr/bin/env python
"""bench.py — the driver's benchmark contract for the RcppSparse hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own serial CPU code
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results to DIR/<op>.npy

`value` (BASELINE.json configs[1], SURVEY.md 8d "C2"): 1,000,000 x 100,000 uniform rsparsematrix-style
dgCMatrix, density 1e-3 (~1e8 stored entries, FP64 values, int32 indices), synthetic, generated straight into
HBM by the integer-exact recipe of rcppsparse_b200/synth.py.  One STEP = one pass of the four reductions the
config names — colSums, rowSums, colMeans, rowMeans (reference RcppSparse.h:131-156) — over the device-resident
matrix; value = 4 * nnz / step time.  At N > 1 (torchrun, one rank per GPU) every rank owns a C2-sized column
block (weak scaling); column results are assembled and row results summed by the library's exchange kernels
over NVLink peer memory, each op's exchange running beside the next op's sweep (the last op's beside the first
sweep of the next step); every result of every timed step is complete before the closing barrier.

The other three hot ops run on THEIR OWN BASELINE configs in the same run and are reported in
`roofline_by_op` next to the C2 reductions (same K/W, CUDA events on the launching stream, inputs >> L2):
  * transpose (RcppSparse.h:375-385) on C3, 30k x 1M power-law columns + row popularity, ~1.5e9 entries (N = 1), and — the
    other transpose path, two stream splits — on the tall C2 and C4 (`transpose@C2`, `transpose@C4`);
  * A v and A^T v (iterator idiom, shapes of RcppSparse.h:140-142 / 133-135) on C4, 2^20 x 2M power-law columns,
    ~2.0e9 entries — at N > 1 the SAME matrix split into nnz-balanced column blocks (strong scaling; `c4_strong`
    carries per-op times, the NVLink term and, measured in the same run on rank 0's GPU, the one-GPU time).
Every sharded op is checked against the oracle on a small block before anything is timed (`parity`).

Resident-mirror layouts: the library serves rowSums/rowMeans/A v from a row-ordered copy and both products from
band-major companions that it builds once for mirrors that keep being asked (sparse_b200.h).  The steady state
measured here is that regime; the first-call regime (scatter kernel / L2-gather sweep) and the one-off build
times are reported beside it (`row_companion`, `products.first_calls`).

Other keys: `per_op`, `roofline` (slowest op of the C2 step), `e2e` (the same step through the host-buffer C
ABI from pinned memory, every step: upload i/p/x + four results back; `.pageable` = from ordinary host arrays,
`.one_op_per_upload` = one upload per op as a lone .Call would pay, `.transpose` = sb200_transpose with host
buffers), `cpu_baseline` (reference code on a bounded column block), `clocks`, `gpu_launches`.
The JSON line is the LAST line of stdout (NCCL may print its banner before it when NCCL_DEBUG is set).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

OPS = ("colSums", "rowSums", "colMeans", "rowMeans")
ABI_OP = {"colSums": "col_sums", "rowSums": "row_sums", "colMeans": "col_means", "rowMeans": "row_means",
          "spmv": "spmv", "spmv_t": "spmv_t", "transpose": "transpose"}
METRIC = "nnz/s"
NOMINAL_HBM_GBS = 8000.0  # BASELINE.json metric: "% of 8 TB/s"
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback
NVLINK_GBS = 770.0  # measured peer copy per direction (B200_PROFILING.md)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C2", help="workload of `value`: C1|C2|C3|C4 (default C2 = BASELINE configs[1])")
    ap.add_argument("--scale", type=float, default=1.0, help="column-count scale of every workload (tests)")
    ap.add_argument("--ops", default=",".join(OPS), help="ops of the `value` step; also spmv,spmv_t,transpose")
    ap.add_argument("--cpu-cols", type=int, default=25000, help="columns of the block timed on the CPU (b200 arm's cpu_baseline)")
    ap.add_argument("--ref-seconds", type=float, default=150.0, help="reference arm: CPU budget for all steps (bounds the sample)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-transpose", action="store_true", help="skip the C3 transpose section")
    ap.add_argument("--no-products", action="store_true", help="skip the C4 A v / A^T v section")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run oracle check of the sharded ops")
    ap.add_argument("--no-n1-inrun", action="store_true", help="N > 1: do not time the whole C4 matrix on rank 0's GPU")
    ap.add_argument("--big-steps", type=int, default=0, help="steps of the C3/C4 sections (default: --steps, at most 50)")
    ap.add_argument("--exchange", default=None, choices=["p2p", "nccl"],
                    help="N > 1: the library's peer-memory exchange kernels (default) or NCCL collectives")
    ap.add_argument("--overlap", action="store_true",
                    help="N > 1 with --exchange nccl: leave each op's collective in flight under the next op's sweep")
    ap.add_argument("--no-row-companion", action="store_true",
                    help="keep rowSums/rowMeans on the scatter kernels (no row-ordered copy of the resident mirror)")
    ap.add_argument("--no-band-companion", action="store_true",
                    help="keep A^T v / A v on the L2-gather sweeps (no band-major companions)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step to DIR/<op>.npy (float64, at most 64 MB in all) so that "
                         "two builds run with the same arguments can be compared output for output")
    return ap.parse_args()


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, arrays):
    """Write every array as out_dir/<name>.npy in float64.  An array longer than its equal share of DUMP_BYTES is
    replaced by the entries at a fixed, seeded sample of positions (the same positions for the same length)."""
    os.makedirs(out_dir, exist_ok=True)
    share = (DUMP_BYTES // max(len(arrays), 1) - 4096) // 8  # 4096: room for the .npy header
    for name, a in arrays.items():
        a = np.asarray(a).ravel()
        if a.size > share:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def value_before_row_copy(ops, nnz, per_op_ms, scatter_ms):
    """Throughput of the same step with rowSums/rowMeans still on the scatter kernels (a mirror's first 8 row-sum
    calls, and adopted device arrays): the timed ops' own times, with each row op replaced by the scatter time
    measured before the row-ordered copy was built."""
    total_ms = sum(scatter_ms if op in ("rowSums", "rowMeans") else per_op_ms[op] for op in ops)
    return len(ops) * nnz / (total_ms * 1e-3) if total_ms > 0 else None


def profile_traffic(kernel, workload):
    """dram bytes per launch of `kernel` on `workload` from the committed ncu capture, if any."""
    path = os.path.join(ROOT, "profiles", "dominant_kernel_traffic.json")
    try:
        k = json.load(open(path))["kernels"][kernel]
        if k.get("workload", "C2") != workload:
            return None
        return k["dram_bytes_per_launch"]
    except Exception:
        return None


def roofline_entry(op, workload, kernel, ab, ms, peak, nnz, extra=None):
    gbs = ab / (ms * 1e-3) / 1e9
    d = {"op": op, "workload": workload, "kernel": kernel, "bound": "hbm", "ms_per_launch": ms,
         "algorithmic_bytes_per_launch": int(ab), "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
         "frac_of_nominal_8TBps": gbs / NOMINAL_HBM_GBS, "nnz_per_s": nnz / (ms * 1e-3),
         "traffic": profile_traffic(kernel, workload)}
    if extra:
        d.update(extra)
    return d


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index
        self.t0 = self.t1 = None

    def start(self):
        """Started well before the timed region (nvidia-smi needs ~1 s to produce its first line)."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def wait_first_sample(self, timeout=5.0):
        t_end = time.perf_counter() + timeout
        while self.proc and not self.rows and time.perf_counter() < t_end:
            time.sleep(0.02)

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                pass
        inside = [r for (t, r) in self.rows if self.t0 is not None and self.t0 <= t <= self.t1 + 0.05]
        where = "during the timed region"
        if not inside:  # region shorter than one sampling period: take the samples right around it
            inside = [r for (t, r) in self.rows if self.t0 is not None and abs(t - self.t0) < 0.5]
            where = "within 0.5 s of the timed region (region shorter than the sampling period)"
        sm, mx, reasons = [], [], set()
        for r in inside:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                                  ("sw_power_cap", 8)):
                    if r[col].lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "sampled": where}


# =====================================================================================================
# reference arm: the reference's own serial CPU code (oracle/_ref when it was built from
# /root/reference, else the C port of the same loops) on the same workload
# =====================================================================================================
def cpu_block(spec, n_cols):
    """Columns [0, n_cols) of the workload as host arrays, generated in slabs (the recipe is per column)."""
    from rcppsparse_b200 import synth

    n_cols = max(1, min(n_cols, spec.ncol))
    slab = 10000
    if n_cols <= slab:
        i, p, x = synth.generate_host(spec, 0, n_cols)
        return i, p, x, spec.nrow, n_cols
    parts = [synth.generate_host(spec, c, min(c + slab, n_cols)) for c in range(0, n_cols, slab)]
    i = np.concatenate([q[0] for q in parts])
    x = np.concatenate([q[2] for q in parts])
    p = np.zeros(n_cols + 1, np.int64)
    at, base = 0, 0
    for q in parts:
        n = q[1].shape[0] - 1
        p[at:at + n + 1] = q[1].astype(np.int64) + base
        at += n
        base += int(q[1][-1])
    return i, p.astype(np.int32), x, spec.nrow, n_cols


def time_cpu(ops, block, reps):
    """Best-of-reps wall time of each op on the block; returns (checker kind, {op: seconds}, nnz)."""
    from oracle import oracle
    from rcppsparse_b200 import synth

    chk = oracle.best()  # the line's `kind` says which checker ran
    i, p, x, nrow, ncol = block
    v_c, v_r = synth.dense_vector(1, ncol), synth.dense_vector(2, nrow)
    out = {}
    for op in ops:
        best = float("inf")
        for _ in range(reps):
            t0 = time.perf_counter()
            if op == "spmv":
                chk.spmv(i, p, x, nrow, ncol, v_c)
            elif op == "spmv_t":
                chk.spmv_t(i, p, x, nrow, ncol, v_r)
            elif op == "transpose":
                chk.transpose(i, p, x, nrow, ncol)
            else:
                getattr(chk, op)(i, p, x, nrow, ncol)
            best = min(best, time.perf_counter() - t0)
        out[op] = best
    return chk.kind, out, int(x.shape[0])


def run_reference(args, ops):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # other ranks exit 0 without work
    from rcppsparse_b200 import synth

    spec = synth.config(args.workload, args.scale)
    # The whole matrix when all steps fit the CPU budget (the driver's --steps 20 --warmup 5 does: ~1.4 s per
    # step on one core), else a bounded column sample of it.  --cpu-cols overrides (tests).
    n_steps = args.steps + max(1, min(args.warmup, 3))
    est_step_s = 1.45 * (spec.ncol / 100000.0) * (len(ops) / 4.0)  # C2: ~1.4 s for the four reductions on one core
    cols = spec.ncol
    if est_step_s * n_steps > args.ref_seconds:
        cols = max(1000, int(spec.ncol * args.ref_seconds / (est_step_s * n_steps)))
    if args.cpu_cols != 25000:
        cols = min(cols, args.cpu_cols)
    cols = min(cols, spec.ncol)
    block = cpu_block(spec, cols)
    nnz = int(block[2].shape[0])
    for _ in range(max(1, min(args.warmup, 3))):
        time_cpu(ops, block, 1)
    kind = "port"
    step_s = []
    for _ in range(args.steps):
        kind, t, _ = time_cpu(ops, block, 1)
        step_s.append(sum(t.values()))
    step = float(np.median(step_s))
    value = len(ops) * nnz / step
    whole = cols == spec.ncol
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "nnz/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": step * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(spec, args, ops, nnz_per_rank=nnz if whole else None),
        "cpu_baseline": {"value": value, "unit": "nnz/s", "cores": 1, "kind": kind,
                         "sample": (f"the whole workload ({nnz} stored entries)" if whole else
                                    f"columns [0,{block[4]}) of the workload ({nnz} stored entries)") +
                                   f", {len(ops)} ops per step, serial (the reference hot path has no parallel pragma)"},
        "e2e": {"value": value, "unit": "nnz/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def workload_config(spec, args, ops, nnz_per_rank):
    return {"workload": spec.name, "nrow": spec.nrow, "ncol_per_gpu": spec.ncol, "nnz_per_gpu": nnz_per_rank,
            "ops_per_step": list(ops), "values": "f64", "indices": "int32", "seed": spec.seed,
            "parallelism": f"column-sharded x{args.gpus}" if args.gpus > 1 else "single GPU",
            "l2": "inputs (1.2 GB/rank at C2, 18 GB at C3, 24 GB at C4) exceed the 126 MB L2; no explicit flush",
            "also_measured": "transpose on C3 and A v / A^T v on C4: roofline_by_op, c4_strong"}


# =====================================================================================================
# this repo's arm
# =====================================================================================================
class Ctx:
    pass


def time_calls(ctx, fn, steps, warmup):
    """Device time per call of fn (CUDA events on the launching stream around exactly `steps` calls, after
    `warmup` untimed ones, barrier + synchronize on both sides, max over ranks); returns (mean ms, min ms)."""
    import torch
    import torch.distributed as dist

    for _ in range(max(3, warmup)):
        fn()
    ctx.barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    ctx.barrier()
    total = ev[0][0].elapsed_time(ev[-1][1])
    per = [a.elapsed_time(b) for a, b in ev]
    t = torch.tensor([total / steps, float(np.min(per))], dtype=torch.float64, device=ctx.dev)
    if ctx.world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0].item()), float(t[1].item())


def in_run_parity(ctx, args):
    """Every op of the column-sharded matrix against the oracle on a small C4-shaped block, through the same
    exchange layer and the same cached layouts the timed sections use; returns the worst |err| / sum|terms|."""
    import torch
    import torch.distributed as dist

    from oracle import oracle
    from rcppsparse_b200 import DeviceMatrix, shard, synth

    spec = synth.powerlaw_spec(40_000, 6_000, 180.0, 4321, row_levels=0, name="parity block")
    i, p, x = synth.generate_host(spec)
    bounds = shard.split_columns_by_nnz(p, ctx.world)
    c0, c1 = bounds[ctx.rank], bounds[ctx.rank + 1]
    D = DeviceMatrix.synth(spec, c0, c1, device=ctx.local_rank)
    S = shard.ShardedMatrix(shard.GpuLocal(D), bounds, ctx.rank, device=ctx.dev, exchange=args.exchange)
    chk = oracle.best()
    a = (i, p, x, spec.nrow, spec.ncol)
    v_c, v_r = synth.dense_vector(1, spec.ncol), synth.dense_vector(2, spec.nrow)
    d_vc, d_vr = torch.from_numpy(v_c).to(ctx.dev), torch.from_numpy(v_r).to(ctx.dev)
    worst = {}

    def check(tag):
        for op, run, want, v in (("colSums", S.colSums, chk.colSums(*a), None), ("colMeans", S.colMeans, chk.colMeans(*a), None),
                                 ("rowSums", S.rowSums, chk.rowSums(*a), None), ("rowMeans", S.rowMeans, chk.rowMeans(*a), None),
                                 ("spmv", lambda: S.spmv(d_vc), chk.spmv(*a, v_c), v_c),
                                 ("spmv_t", lambda: S.spmv_t(d_vr), chk.spmv_t(*a, v_r), v_r)):
            got = run().cpu().numpy()
            worst[op] = max(worst.get(op, 0.0), oracle.assert_within(op, got, want, *a, v=v))

    check("first-call kernels")
    if not args.no_row_companion:
        D.row_companion(1)
    if not args.no_band_companion:
        D.band_companion(0, 1)
        D.band_companion(1, 1)
    check("cached layouts")
    if ctx.world == 1:  # the transpose is per GPU in this benchmark
        T = D.transpose_dev()
        ti, tp, tx = T.download_columns()
        wi, wp, wx = chk.transpose(*a)
        assert np.array_equal(tp, wp) and np.array_equal(ti, wi) and np.array_equal(tx.view(np.uint64), wx.view(np.uint64)), \
            "transpose differs from the oracle"
        T.close()
    if ctx.world > 1:
        S.close()
    D.close()
    ok = torch.tensor([1], dtype=torch.int32, device=ctx.dev)
    if ctx.world > 1:
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    return {"parity_checked": True, "checker": chk.kind, "block": f"{spec.nrow} x {spec.ncol} power-law columns, {x.shape[0]} entries, "
            f"{ctx.world} column block(s)", "tolerance": "1e-12 * sum|terms| per entry; transpose bit-exact (N = 1)",
            "worst_err_over_sum_abs_terms": worst, "layouts": "first-call kernels and cached layouts both checked"}


TRANSPOSE_KERNELS = {"C3": "transpose_bitrank_kernel", "C2": "split_kernel<1> + split_kernel<2>", "C4": "split_kernel<1> + split_kernel<2>"}


def section_transpose(ctx, args, peak, steps, warmup, cfg="C3"):
    """CSC -> CSR transpose on C3 (BASELINE configs[2]) — or on the tall C2 / C4, which take the two-split path — on this
    rank's GPU: sb200_transpose_dev, result kept in HBM."""
    import torch

    from rcppsparse_b200 import DeviceMatrix, synth

    spec = synth.config(cfg, args.scale)
    # every call allocates its result (12 B/entry) from the library's pool; start from an empty pool so that the blocks a
    # previous section left behind (other sizes) do not push the allocator onto its slow paths mid-measurement
    from rcppsparse_b200 import _lib
    _lib.lib().sb200_trim(ctx.local_rank)
    t0 = time.perf_counter()
    D = DeviceMatrix.synth(spec, device=ctx.local_rank)
    D.set_stream(torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    gen_s = time.perf_counter() - t0
    keep = []

    def run_alloc():
        keep.clear()  # the previous result goes back to the pool before the next one is allocated
        keep.append(D.transpose_dev())

    def run():
        D.transpose_into(keep[0])  # the same transpose into the result that exists: no allocation, same kernels

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run_alloc()
    e1.record()
    torch.cuda.synchronize()
    first_ms = e0.elapsed_time(e1)
    # the allocating form (what Matrix::transpose() is): median over a few calls — multi-GB blocks going through the
    # pool every call show up as occasional allocator spikes of 0.1-1 s at C4, which say nothing about the kernels
    alloc_ms = []
    for _ in range(min(steps, 9)):
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record()
        run_alloc()
        eb.record()
        eb.synchronize()
        alloc_ms.append(ea.elapsed_time(eb))
    ms, ms_min = time_calls(ctx, run, steps, warmup)
    # size-independent check at full size: the result's column sums are the source's row sums, entry count kept
    T = keep[0]
    ok = T.nnz == D.nnz and T.nrow == D.ncol and T.ncol == D.nrow
    a = torch.empty(D.nrow, dtype=torch.float64, device=ctx.dev)
    b = torch.empty(D.nrow, dtype=torch.float64, device=ctx.dev)
    T.set_stream(torch.cuda.current_stream().cuda_stream)
    T.col_sums_dev(a)
    D.row_companion(-1)
    D.row_sums_dev(b)
    torch.cuda.synchronize()
    scale = float(b.abs().max().item()) or 1.0
    drift = float((a - b).abs().max().item()) / scale
    ab = D.algorithmic_bytes("transpose")
    entry = roofline_entry("transpose", cfg, TRANSPOSE_KERNELS.get(cfg, "transpose"), ab, ms, peak, D.nnz,
                           {"ms_min": ms_min, "first_call_ms": first_ms, "nnz": D.nnz,
                            "allocating_form_ms": {"median": float(np.median(alloc_ms)), "min": float(np.min(alloc_ms)),
                                                   "max": float(np.max(alloc_ms)), "calls": len(alloc_ms)},
                            "what": "sb200_transpose_into: (cached) plan + placement kernel(s) into the result of an earlier "
                                    "sb200_transpose_dev; allocating_form_ms = sb200_transpose_dev itself (result and, on the two-split "
                                    "path's first call, the 16 B/entry record stream from the pool + the result's tile plans); "
                                    "first_call_ms includes building the plan",
                            "check": {"shape_and_nnz_ok": bool(ok), "colSums(T) vs rowSums(A) max rel diff": drift}})
    info = {"workload": spec.name, "nnz": D.nnz, "generate_s": gen_s, "steps": steps}
    keep.clear()
    D.close()
    return entry, info


def c4_bounds(spec, world):
    """nnz-balanced column blocks of the C4 matrix, from the recipe's column lengths (same on every rank)."""
    from rcppsparse_b200 import synth

    lens = np.concatenate([synth.column_lengths(spec, np.arange(c, min(c + 250000, spec.ncol), dtype=np.uint64))
                           for c in range(0, spec.ncol, 250000)])
    p = np.zeros(spec.ncol + 1, np.int64)
    np.cumsum(lens, out=p[1:])
    from rcppsparse_b200 import shard

    return shard.split_columns_by_nnz(p, world), int(p[-1])


def time_products(ctx, args, D, S, v_col, v_row, steps, warmup):
    """ms per call of A v and A^T v: through the sharded matrix S (exchange included) or, S = None, on D alone."""
    import torch

    out_r = torch.empty(max(D.nrow, 1), dtype=torch.float64, device=ctx.dev)
    out_c = torch.empty(max(D.ncol, 1), dtype=torch.float64, device=ctx.dev)
    if S is not None:
        fns = {"spmv": lambda: S.spmv(v_col), "spmv_t": lambda: S.spmv_t(v_row)}
    else:
        fns = {"spmv": lambda: D.spmv_dev(v_col, out_r), "spmv_t": lambda: D.spmv_t_dev(v_row, out_c)}
    res = {}
    for op, fn in fns.items():
        res[op] = time_calls(ctx, fn, steps, warmup)
    return res


def build_product_layouts(args, D):
    """Row-ordered copy + both band-major companions of a resident mirror (what the library does on its own after
    8 calls of each kind), timed: the first build grows the memory pool (the driver maps tens of GB), a rebuild with
    the pool warm is the cost of the passes themselves."""
    import torch

    out = {}
    if args.no_band_companion:
        return out

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3

    out["band_companion_AT_v_build_ms"] = timed(lambda: D.band_companion(0, 1))
    D.band_companion(0, 0)
    out["band_companion_AT_v_rebuild_ms_pool_warm"] = timed(lambda: D.band_companion(0, 1))
    out["row_copy_plus_band_companion_A_v_build_ms"] = timed(lambda: D.band_companion(1, 1))
    D.band_companion(1, 0)
    out["band_companion_A_v_rebuild_ms_pool_warm"] = timed(lambda: D.band_companion(1, 1))
    out["layouts_mask"] = D.layouts()
    out["extra_hbm_bytes"] = D.layout_bytes()
    out["matrix_bytes"] = 12 * D.nnz + 4 * (D.ncol + 1)
    return out


def section_products(ctx, args, peak, steps, warmup):
    """A v and A^T v on C4 (BASELINE configs[3]): the same 2.0e9-entry matrix on 1 GPU or split into nnz-balanced
    column blocks over the ranks (strong scaling), exchange included."""
    import torch

    from rcppsparse_b200 import DeviceMatrix, shard, synth

    spec = synth.config("C4", args.scale)
    bounds, nnz_total = c4_bounds(spec, ctx.world)
    c0, c1 = bounds[ctx.rank], bounds[ctx.rank + 1]
    t0 = time.perf_counter()
    D = DeviceMatrix.synth(spec, c0, c1, device=ctx.local_rank)
    torch.cuda.synchronize()
    gen_s = time.perf_counter() - t0
    local = shard.GpuLocal(D)
    S = shard.ShardedMatrix(local, bounds, ctx.rank, device=ctx.dev, exchange=args.exchange) if ctx.world > 1 else None
    v_col = torch.empty(spec.ncol, dtype=torch.float64, device=ctx.dev)
    v_row = torch.empty(spec.nrow, dtype=torch.float64, device=ctx.dev)
    D.synth_vector_dev(spec.seed, 0, spec.ncol, v_col)
    D.synth_vector_dev(spec.seed + 7, 0, spec.nrow, v_row)
    v_loc = v_col[c0:c1] if ctx.world > 1 else v_col

    info = {"workload": spec.name, "nnz_total": nnz_total, "nnz_this_rank": D.nnz, "generate_s": gen_s, "steps": steps}
    # first-call regime: scatter / L2-gather kernels on the CSC arrays (what a mirror's first 8 calls run)
    D.row_companion(-1)
    D.band_companion(0, -1)
    first = time_products(ctx, args, D, None, v_loc, v_row, min(steps, 5), 3)
    info["first_calls"] = {op: {"ms": first[op][0], "row_path": D.row_path()} for op in first}
    D.row_companion(0)
    D.band_companion(0, 0)
    info["layouts"] = build_product_layouts(args, D)
    res = time_products(ctx, args, D, S, v_col if S is not None else v_loc, v_row, steps, warmup)
    ab_local = D.algorithmic_bytes("spmv")
    m, n = spec.nrow, spec.ncol
    ab_total = 12 * nnz_total + 4 * (n + 1) + 8 * n + 8 * m
    kern = "bandsweep_kernel" if not args.no_band_companion else "sweep_kernel<SPMV_T>"
    entries = {}
    for op in ("spmv", "spmv_t"):
        ms, ms_min = res[op]
        e = roofline_entry(op, "C4", kern + (" over the row-ordered copy's companion" if op == "spmv" else ""),
                           ab_total / ctx.world, ms, peak, nnz_total / ctx.world,
                           {"ms_min": ms_min, "nnz_per_s_all_gpus": nnz_total / (ms * 1e-3),
                            "first_call_ms": info["first_calls"][op]["ms"],
                            "bytes_note": "SURVEY.md 8(d): 12N + 4(n+1) + 8n + 8m of the whole matrix / n_gpus; this rank's own block is "
                                          f"{ab_local} bytes"})
        if ctx.world > 1:
            coll = 8 * m if op == "spmv" else 8 * n
            e["nvlink"] = {"what": "row-indexed partials summed over ranks (8m bytes in, 8m out per GPU)" if op == "spmv" else
                                   "column slices gathered on every rank (8n bytes received per GPU)",
                           "bytes_per_gpu": coll, "floor_us_at_770GBps": coll / (NVLINK_GBS * 1e9) * 1e6,
                           "hbm_floor_us": ab_total / ctx.world / (peak * 1e9) * 1e6}
            e["frac"] = (ab_total / ctx.world / (peak * 1e9) + coll / (NVLINK_GBS * 1e9)) / (ms * 1e-3)
            e["frac_note"] = "(HBM floor of the block + NVLink term) / measured time"
        entries[op] = e
    if S is not None:
        S.close()
    D.close()
    return entries, info


def section_products_n1_inrun(ctx, args, peak, steps, warmup):
    """N > 1: the whole C4 matrix on rank 0's GPU, same kernels, no exchange — the one-GPU time the strong-scaling
    speed-up is taken against, measured in the same run on the same box (other ranks wait at the barrier)."""
    import torch

    from rcppsparse_b200 import DeviceMatrix, synth

    out = None
    if ctx.rank == 0:
        try:
            spec = synth.config("C4", args.scale)
            D = DeviceMatrix.synth(spec, device=ctx.local_rank)
            D.set_stream(torch.cuda.current_stream().cuda_stream)
            v_col = torch.empty(spec.ncol, dtype=torch.float64, device=ctx.dev)
            v_row = torch.empty(spec.nrow, dtype=torch.float64, device=ctx.dev)
            D.synth_vector_dev(spec.seed, 0, spec.ncol, v_col)
            D.synth_vector_dev(spec.seed + 7, 0, spec.nrow, v_row)
            build_product_layouts(args, D)
            one = Ctx()
            one.world, one.dev = 1, ctx.dev
            one.barrier = torch.cuda.synchronize
            res = time_products(one, args, D, None, v_col, v_row, min(steps, 10), 3)
            out = {op: res[op][0] for op in res}
            D.close()
        except Exception as e:  # never lose the line
            out = {"error": f"{type(e).__name__}: {e}"}
    ctx.barrier()
    return out


def run_b200(args, ops):
    import torch
    import torch.distributed as dist

    from rcppsparse_b200 import DeviceMatrix, _lib, shard, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: bench.py measures the CUDA path and has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    ctx = Ctx()
    ctx.world, ctx.rank, ctx.local_rank, ctx.dev = world, rank, local_rank, dev

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ctx.barrier = barrier
    peak, peak_src = measured_peak()
    big_steps = args.big_steps if args.big_steps > 0 else min(args.steps, 50)

    # ---- parity first: nothing is timed on kernels that disagree with the oracle ------------------------------
    parity = None
    if not args.no_parity:
        parity = in_run_parity(ctx, args)

    spec = synth.config(args.workload, args.scale)
    c0, c1 = rank * spec.ncol, (rank + 1) * spec.ncol  # weak scaling: every rank generates its own block
    D = DeviceMatrix.synth(spec, c0, c1, device=local_rank)
    nnz = D.nnz
    local = shard.GpuLocal(D)  # binds the handle to torch's current stream
    bounds = [k * spec.ncol for k in range(world + 1)]
    S = shard.ShardedMatrix(local, bounds, rank, device=dev, exchange=args.exchange)
    v_col = torch.empty(S.ncol, dtype=torch.float64, device=dev)
    v_row = torch.empty(S.nrow, dtype=torch.float64, device=dev)
    D.synth_vector_dev(spec.seed, 0, S.ncol, v_col)
    D.synth_vector_dev(spec.seed + 7, 0, S.nrow, v_row)
    T_keep = []

    # p2p: the exchange kernels of op k run on the window's stream beside the sweep of op k+1 (always);
    # nccl: only with --overlap (measured slower: the NCCL kernel waits for SM resources behind the sweep)
    overlap = world > 1 and (S.exchange == "p2p" or args.overlap)

    def run_op(op):
        """Launch op; with more than one rank its collective is left in flight (async NCCL) so that the next
        op's sweep overlaps it — every step waits for all of its results before it ends."""
        if op == "spmv":
            return S.spmv(v_col, async_op=overlap)
        if op == "spmv_t":
            return S.spmv_t(v_row, async_op=overlap)
        if op == "transpose":
            T_keep.clear()
            T_keep.append(D.transpose_dev())  # local block only (the sharded exchange is ShardedMatrix.transpose)
            return None
        return getattr(S, op)(async_op=overlap)

    def wait_all(pend):
        for r in pend or ():
            if r is not None:
                r.wait()

    last = {}  # op -> what its call in the latest step returned (a tensor, a Pending, or None for the transpose)

    def run_step(marks=None, prev=None):
        """One step.  With overlapped exchanges the results of the PREVIOUS step are waited for after this step's
        first sweep has been launched (its last exchange then runs beside that sweep instead of ending the step
        alone); the caller waits for the last step's results before the closing barrier.  Returns what is pending."""
        pend = []
        for k, op in enumerate(ops):
            last[op] = run_op(op)
            pend.append(last[op])
            if k == 0:
                wait_all(prev)
            if marks is not None:
                marks[k + 1].record()
        if marks is not None:
            marks[len(ops) + 1].record()
        return pend if overlap else None

    # ---- row sums of a resident mirror -------------------------------------------------------------------------
    # The library serves rowSums/rowMeans with its scatter kernel until a mirror has been asked for them more than
    # SB200_ROW_COMPANION_AFTER (8) times, then from a row-ordered copy of x (sparse_b200.h).  The steady state of
    # this benchmark is the second regime; the first is timed here, with the one-off cost of the switch, so that
    # the line carries both.
    row_companion = None
    if any(op in ("rowSums", "rowMeans") for op in ops):
        out_r = torch.empty(max(D.nrow, 1), dtype=torch.float64, device=dev)
        if args.no_row_companion:
            D.row_companion(-1)
        path0 = D.row_path()
        for _ in range(2):
            D.row_sums_dev(out_r)
        torch.cuda.synchronize()
        pre = []
        for _ in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            D.row_sums_dev(out_r)
            e1.record()
            e1.synchronize()
            pre.append(e0.elapsed_time(e1))
        ab0 = D.algorithmic_bytes("row_sums")
        row_companion = {"scatter_path": path0, "scatter_ms_per_call": float(np.median(pre)),
                         "scatter_GBps": ab0 / (float(np.median(pre)) * 1e-3) / 1e9, "scatter_algorithmic_bytes": ab0,
                         "policy": "row-ordered copy after 8 row-sum calls on a mirror that owns its arrays",
                         "built": False}
        if not args.no_row_companion:
            try:
                t0 = time.perf_counter()
                D.row_companion(1)  # what the 9th call would do on its own; explicit so that it is timed, and so that
                torch.cuda.synchronize()  # it precedes the warm-up whatever --warmup is
                build_ms = (time.perf_counter() - t0) * 1e3
                # again with the pool warm and the transpose plan on the handle (what a refresh of the values costs):
                D.row_companion(0)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                D.row_companion(1)
                torch.cuda.synchronize()
                rebuild_ms = (time.perf_counter() - t0) * 1e3
                row_companion.update(built=True, build_ms=build_ms, rebuild_ms_pool_warm=rebuild_ms,
                                     build_note="build_ms: first transpose in the process (kernel load, transpose plan, the "
                                                "pool growing by the copy and the transpose's scratch); rebuild: the same call "
                                                "with the pool warm and the plan cached",
                                     extra_hbm_bytes=12 * nnz + 4 * (D.nrow + 1))
                saved = row_companion["scatter_ms_per_call"]
                row_companion["break_even_calls_after_threshold"] = None
                row_companion["_saved_ms"] = saved
            except Exception as e:
                row_companion["error"] = f"{type(e).__name__}: {e}"
        del out_r

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    pend = None
    for _ in range(max(args.warmup, 3)):
        pend = run_step(prev=pend)
    wait_all(pend)
    pend = None
    barrier()
    if rank == 0:
        sampler.wait_first_sample()
    launches0 = _lib.lib().sb200_launch_count()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(len(ops) + 2)] for _ in range(args.steps)]
    barrier()
    sampler.mark_begin()
    t_wall0 = time.perf_counter()
    for s in range(args.steps):
        ev[s][0].record()
        pend = run_step(ev[s], prev=pend)
    wait_all(pend)  # every result of every timed step is complete before the closing barrier
    tail_ev = torch.cuda.Event(enable_timing=True)
    tail_ev.record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    sampler.mark_end()
    launches = _lib.lib().sb200_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        outs = {}
        for op in ops:
            if op == "transpose":
                outs.update(zip(("transpose_i", "transpose_p", "transpose_x"), T_keep[0].download_columns()))
            else:
                r = last[op]
                outs[op] = (r.tensor if isinstance(r, shard.Pending) else r).cpu().numpy()
        dump_outputs(args.dump_outputs, outs)

    total_ms = ev[0][0].elapsed_time(tail_ev)  # device time of exactly K steps on the launching stream, last results included
    per_op_ms = {op: float(np.mean([ev[s][k].elapsed_time(ev[s][k + 1]) for s in range(args.steps)]))
                 for k, op in enumerate(ops)}
    per_op_min = {op: float(np.min([ev[s][k].elapsed_time(ev[s][k + 1]) for s in range(args.steps)]))
                  for k, op in enumerate(ops)}
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    nnz_all = torch.tensor([nnz], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(nnz_all, op=dist.ReduceOp.SUM)
    nnz_total = int(nnz_all.item())
    on_copy = D.row_path() == "row-companion"
    row_path_final = D.row_path()
    ab_of = {op: D.algorithmic_bytes(ABI_OP[op] + ("_companion" if on_copy and op in ("rowSums", "rowMeans") else "")) for op in ops}
    ab_csc = {op: D.algorithmic_bytes(ABI_OP[op]) for op in ops}

    # ---- e2e: the host-buffer C ABI, upload + results every step (N = 1 only) -------------------------------
    e2e = None
    if world == 1 and not args.no_e2e and rank == 0:
        try:
            e2e = measure_e2e(args, ops, D, nnz, local_rank)
        except Exception as e:  # never lose the device-resident line
            e2e = {"value": None, "unit": "nnz/s", "error": f"{type(e).__name__}: {e}"}
    elif world > 1:
        e2e = {"value": None, "unit": "nnz/s", "note": "measured at N=1 (host-buffer C ABI is per process)"}

    if world > 1:
        S.close()  # raises if an exchange barrier ever timed out
    T_keep.clear()
    D.close()

    # ---- the other hot ops on their own configs ----------------------------------------------------------------
    by_op, sections = {}, {}
    if not args.no_transpose and world == 1:
        try:
            by_op["transpose@C3"], sections["transpose"] = section_transpose(ctx, args, peak, big_steps, args.warmup)
        except Exception as e:
            sections["transpose"] = {"error": f"{type(e).__name__}: {e}"}
        for cfg in ("C2", "C4"):  # the tall configs: two stable stream splits (transpose_split.cu)
            try:
                by_op[f"transpose@{cfg}"], sections[f"transpose_{cfg}"] = section_transpose(ctx, args, peak, max(3, big_steps // 2), args.warmup, cfg)
            except Exception as e:
                sections[f"transpose_{cfg}"] = {"error": f"{type(e).__name__}: {e}"}
    c4_strong = None
    if not args.no_products:
        try:
            entries, info = section_products(ctx, args, peak, big_steps, args.warmup)
            by_op["spmv@C4"], by_op["spmv_t@C4"] = entries["spmv"], entries["spmv_t"]
            sections["products"] = info
            if world > 1:
                n1 = None if args.no_n1_inrun else section_products_n1_inrun(ctx, args, peak, big_steps, args.warmup)
                c4_strong = {"n_gpus": world, "nnz_total": info["nnz_total"], "scaling": "strong",
                             "ms": {op: entries[op]["ms_per_launch"] for op in entries},
                             "nnz_per_s": {op: entries[op]["nnz_per_s_all_gpus"] for op in entries},
                             "one_gpu_ms_same_run": n1,
                             "speedup_vs_n1": ({op: n1[op] / entries[op]["ms_per_launch"] for op in entries}
                                               if n1 and "error" not in n1 else None)}
        except Exception as e:
            sections["products"] = {"error": f"{type(e).__name__}: {e}"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    ms_per_step = total_ms / args.steps
    value = len(ops) * nnz_total / (ms_per_step * 1e-3)
    per_op = {}
    row_kernel = ("sweep_kernel<COLSUM> over the row-ordered copy" if on_copy else
                  "band_scatter_kernel" if row_path_final == "banded" else "rowsum_stream_kernel")
    kernel_of = {"rowSums": row_kernel, "rowMeans": row_kernel, "colSums": "sweep_kernel<COLSUM>",
                 "colMeans": "sweep_kernel<COLSUM>", "spmv": "sweep_kernel<SPMV>", "spmv_t": "sweep_kernel<SPMV_T>",
                 "transpose": "transpose_bitrank_kernel"}
    wl = args.workload.upper()
    for op in ops:
        ab = ab_of[op]
        gbs = ab / (per_op_ms[op] * 1e-3) / 1e9
        per_op[op] = {"ms": per_op_ms[op], "ms_min": per_op_min[op], "nnz_per_s_per_gpu": nnz / (per_op_ms[op] * 1e-3),
                      "algorithmic_bytes": ab, "achieved_GBps": gbs, "frac_of_measured": gbs / peak,
                      "frac_of_nominal_8TBps": gbs / NOMINAL_HBM_GBS}
        extra = {"ms_min": per_op_min[op]}
        if on_copy and op in ("rowSums", "rowMeans") and row_companion:
            # the same op on the reference-shaped CSC arrays (SURVEY 8d: 12N + 8m), before the row-ordered copy exists
            extra["on_csc_arrays"] = {"kernel": "band_scatter_kernel" if row_companion["scatter_path"] == "banded" else "rowsum_stream_kernel",
                                      "ms": row_companion["scatter_ms_per_call"], "algorithmic_bytes": ab_csc[op],
                                      "frac": ab_csc[op] / (row_companion["scatter_ms_per_call"] * 1e-3) / 1e9 / peak}
            extra["bytes_note"] = "on the row-ordered copy: 8N + 4(m+1) + 8m"
        by_op[f"{op}@{wl}"] = roofline_entry(op, wl, kernel_of[op], ab, per_op_ms[op], peak, nnz, extra)
    dom = max(ops, key=lambda o: per_op_ms[o])
    roofline = {"bound": "hbm", "kernel": kernel_of[dom], "op": dom, "achieved": per_op[dom]["achieved_GBps"], "peak": peak,
                "peak_source": peak_src, "unit": "GB/s", "frac": per_op[dom]["achieved_GBps"] / peak,
                "frac_of_nominal_8TBps": per_op[dom]["achieved_GBps"] / NOMINAL_HBM_GBS,
                "algorithmic_bytes_per_launch": per_op[dom]["algorithmic_bytes"], "ms_per_launch": per_op_ms[dom],
                "timed": "CUDA events on the launching stream around the op (zero-fill + kernel), mean over the timed steps",
                "traffic": profile_traffic(kernel_of[dom], wl) if args.scale == 1.0 else None,
                "scope": "slowest op of the C2 step; every op on its own config is in roofline_by_op"}
    if row_companion is not None:
        row_companion["scatter_frac_of_measured"] = row_companion["scatter_GBps"] / peak
        saved = row_companion.pop("_saved_ms", None)
        if row_companion.get("built") and saved is not None:
            gain = saved - float(np.mean([per_op_ms[o] for o in ops if o in ("rowSums", "rowMeans")]))
            # the build as a resident mirror pays it (pool warm); the first transpose of a process also loads the kernels
            # and grows the pool, which no later build does
            warm = row_companion.get("rebuild_ms_pool_warm", row_companion["build_ms"])
            row_companion["break_even_calls_after_threshold"] = (warm / gain) if gain > 0 else None
            row_companion["break_even_calls_first_build_of_process"] = (row_companion["build_ms"] / gain) if gain > 0 else None
        else:
            row_companion.pop("break_even_calls_after_threshold", None)
        if world == 1 and row_companion.get("built"):
            row_companion["value_before_row_copy"] = value_before_row_copy(ops, nnz, per_op_ms, row_companion["scatter_ms_per_call"])

    line = {
        "metric": METRIC, "value": value, "unit": "nnz/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": workload_config(spec, args, ops, nnz), "per_op": per_op, "roofline": roofline,
        "roofline_by_op": by_op, "sections": sections, "c4_strong": c4_strong, "parity": parity,
        "row_path": row_path_final, "row_companion": row_companion,
        "exchange": (None if world == 1 else
                     "libsparse_b200 kernels over NVLink peer memory (cudaIpc window): P2P stores of each rank's slice for "
                     "column results, rank-ordered P2P reduction for row results, flag barriers; op k's exchange runs beside op k+1's "
                     "sweep (the last op's beside the next step's first sweep), all results complete inside the timed region" if S.exchange == "p2p" else
                     "NCCL all-gather / all-reduce" + (", left in flight under the next op's sweep" if overlap else "")),
        "gpu_launches": int(launches), "clocks": clocks, "wall_s_timed_region": t_wall, "e2e": e2e,
    }

    # ---- cpu_baseline: the reference's serial code on a bounded block, rank 0, N = 1 only ------------------------
    if world == 1 and not args.no_cpu_baseline:
        try:
            block = cpu_block(spec, args.cpu_cols)
            kind, t_cpu, nnz_cpu = time_cpu(ops, block, 3)
            cpu_step = sum(t_cpu.values())
            line["cpu_baseline"] = {
                "value": len(ops) * nnz_cpu / cpu_step, "unit": "nnz/s", "cores": 1, "kind": kind,
                "host_cores_available": os.cpu_count(),
                "sample": f"columns [0,{block[4]}) of the workload ({nnz_cpu} stored entries), best of 3 per op, serial",
                "per_op_nnz_per_s": {op: nnz_cpu / t_cpu[op] for op in ops}}
        except Exception as e:
            line["cpu_baseline"] = {"value": None, "unit": "nnz/s", "error": f"{type(e).__name__}: {e}"}
    sys.stdout.flush()
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def measure_e2e(args, ops, D, nnz, device):
    """Same step through the reference-facing host-buffer entry points: every step uploads i/p/x from
    pinned host memory into a fresh mirror (what one .Call from R pays), runs the ops, and reads every
    result vector back to host."""
    import torch

    from rcppsparse_b200 import DeviceMatrix

    i, p, x = D.download_columns()
    hi = torch.from_numpy(i).pin_memory()
    hp = torch.from_numpy(p).pin_memory()
    hx = torch.from_numpy(x).pin_memory()
    del i, p, x
    v_c = np.ones(D.ncol)
    v_r = np.ones(D.nrow)
    host_fn = {"colSums": "col_sums", "rowSums": "row_sums", "colMeans": "col_means", "rowMeans": "row_means"}

    # results land in caller-owned pinned buffers, as the inputs leave from pinned buffers (the C ABI takes the
    # caller's pointer either way; fresh pageable vectors would add their first-touch page faults to every step)
    res = {op: torch.empty(D.ncol if op in ("colSums", "colMeans", "spmv_t") else D.nrow, dtype=torch.float64).pin_memory()
           for op in ops if op != "transpose"}

    def run_ops(M, which, outs):
        for op in which:
            if op in host_fn:
                getattr(M, host_fn[op])(out=outs[op])
            elif op == "spmv":
                M.spmv(v_c)
            elif op == "spmv_t":
                M.spmv_t(v_r)
            elif op == "transpose":
                M.transpose_host()

    def step():
        with DeviceMatrix.from_host(hi, hp, hx, D.nrow, D.ncol, device=device, validate=True) as M:
            run_ops(M, ops, res)

    def timed(fn, n):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(n):
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t0)
        return float(np.median(ts)), ts

    dt, times = timed(step, args.e2e_steps)
    h2d = 12 * nnz + 4 * (D.ncol + 1)
    d2h = sum(8 * (D.ncol if op in ("colSums", "colMeans", "spmv_t") else D.nrow) for op in ops if op != "transpose")
    out = {"value": len(ops) * nnz / dt, "unit": "nnz/s", "ms_per_step": dt * 1e3, "h2d_bytes_per_step": int(h2d),
           "d2h_bytes_per_step": int(d2h), "steps": args.e2e_steps, "ms_all_steps": [round(t * 1e3, 3) for t in times],
           "what": "per step: sb200_matrix_create from pinned host buffers (values upload overlapped with structure check "
                   "and plans) + the host-buffer ops (results copied back into pinned host buffers) + destroy; wall clock, "
                   "median step"}
    # one upload per op: what a lone .Call(columnSums, A) pays (the Exporter builds a fresh Matrix per call,
    # reference src/RcppExports.cpp:20)
    try:
        def step1():
            for op in ops:  # the drop-in header's per-call mirror: SB200_LAZY_ROWS, `i` goes up only if the op reads it
                with DeviceMatrix.from_host(hi, hp, hx, D.nrow, D.ncol, device=device, validate=True, lazy_rows=True) as M:
                    run_ops(M, (op,), res)

        dt1, _ = timed(step1, max(2, args.e2e_steps // 2))
        h2d1 = sum((12 if op in ("rowSums", "rowMeans", "spmv", "spmv_t", "transpose") else 8) * nnz + 4 * (D.ncol + 1) for op in ops)
        out["one_op_per_upload"] = {"value": len(ops) * nnz / dt1, "ms_per_step": dt1 * 1e3,
                                    "h2d_bytes_per_step": int(h2d1), "d2h_bytes_per_step": int(d2h),
                                    "what": "a fresh mirror from pinned buffers for EVERY op of the step, created as the drop-in header "
                                            "creates its per-call mirror (SB200_LAZY_ROWS: colSums / colMeans never read `i`, so they "
                                            "upload x and p only; the row ops upload everything)"}
    except Exception as e:
        out["one_op_per_upload"] = {"value": None, "error": f"{type(e).__name__}: {e}"}
    # the same step from PAGEABLE arrays (what an R caller owns): staged through pinned chunks by worker threads
    try:
        pi, pp, px = hi.numpy().copy(), hp.numpy().copy(), hx.numpy().copy()
        pres = {op: np.empty(res[op].shape[0]) for op in res}

        def pstep():
            with DeviceMatrix.from_host(pi, pp, px, D.nrow, D.ncol, device=device, validate=True) as M:
                run_ops(M, [op for op in ops if op in host_fn], pres)

        pdt, _ = timed(pstep, max(2, args.e2e_steps // 2))
        out["pageable"] = {"value": len(ops) * nnz / pdt, "ms_per_step": pdt * 1e3,
                           "what": "same step with pageable host arrays for inputs and results"}

        # transpose with host buffers (sb200_transpose): upload + device transpose + p'/i'/x' back into host vectors
        tp = np.empty(D.nrow + 1, np.int32)
        ti = np.empty(nnz, np.int32)
        tx = np.empty(nnz, np.float64)
        from rcppsparse_b200 import _lib as L
        from rcppsparse_b200.matrix import _ptr

        def tstep():
            with DeviceMatrix.from_host(pi, pp, px, D.nrow, D.ncol, device=device, validate=True) as M:
                L.check(L.lib().sb200_transpose(M._h, _ptr(tp), _ptr(ti), _ptr(tx)))

        tdt, _ = timed(tstep, max(2, args.e2e_steps // 2))
        out["transpose"] = {"value": nnz / tdt, "unit": "nnz/s", "ms_per_step": tdt * 1e3, "h2d_bytes_per_step": int(h2d),
                            "d2h_bytes_per_step": int(12 * nnz + 4 * (D.nrow + 1)), "workload": "the `value` workload (C2)",
                            "what": "sb200_matrix_create from pageable arrays + sb200_transpose into pageable host vectors + destroy"}
    except Exception as e:
        out.setdefault("pageable", {"value": None, "error": f"{type(e).__name__}: {e}"})
        out.setdefault("transpose", {"value": None, "error": f"{type(e).__name__}: {e}"})
    return out


def main():
    args = parse_args()
    ops = tuple(o for o in args.ops.split(",") if o)
    for o in ops:
        if o not in ABI_OP:
            raise SystemExit(f"unknown op {o}")
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes the CUDA path's results; the reference arm times a column sample")
        run_reference(args, tuple(o for o in ops if o != "transpose") or OPS)
    else:
        run_b200(args, ops)


if __name__ == "__main__":
    main()
