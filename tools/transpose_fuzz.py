#!/usr/bin/env python
"""Randomised shapes through every transpose path against the oracle (bit for bit).  python tools/transpose_fuzz.py [N] [SEED]"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import oracle  # noqa: E402  (a checker: this is a test tool, not product code)
from rcppsparse_b200 import DeviceMatrix, synth  # noqa: E402


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 40
    rng = np.random.default_rng(int(sys.argv[2]) if len(sys.argv) > 2 else 7)
    chk = oracle.best()
    done = 0
    for k in range(n):
        nrow = int(10 ** rng.uniform(0, 6.6))
        ncol = int(10 ** rng.uniform(0, 4.7))
        target = 10 ** rng.uniform(2, float(os.environ.get("FUZZ_MAX_LOG10", "6.7")))
        dens = min(1.0, target / (nrow * ncol))
        if rng.random() < 0.5:
            spec = synth.uniform_spec(nrow, ncol, dens, 100 + k)
        else:
            spec = synth.powerlaw_spec(nrow, ncol, max(0.05, dens * nrow), 100 + k, row_levels=int(rng.integers(0, 6)),
                                       empty_permille=int(rng.integers(0, 500)))
        i, p, x = synth.generate_host(spec)
        want = chk.transpose(i, p, x, spec.nrow, spec.ncol)
        for path, extra in (("split", {}), ("split", {"SB200_SPLIT_SHIFT": str(int(rng.integers(0, 12)))}), ("place", {}), ("banded", {}), (None, {})):
            for key in ("SB200_TRANSPOSE_PATH", "SB200_SPLIT_SHIFT"):
                os.environ.pop(key, None)
            if path:
                os.environ["SB200_TRANSPOSE_PATH"] = path
            os.environ.update(extra)
            if "SB200_SPLIT_SHIFT" in extra and (spec.nrow >> int(extra["SB200_SPLIT_SHIFT"])) >= 3072:
                continue
            with DeviceMatrix.from_host(i, p, x, spec.nrow, spec.ncol) as D:
                for _ in range(2):
                    ti, tp, tx = D.transpose_host()
                    ok = np.array_equal(tp, want[1]) and np.array_equal(ti, want[0]) and np.array_equal(
                        tx.view(np.uint64), want[2].view(np.uint64))
                    if not ok:
                        print("MISMATCH", spec.name, spec.nrow, spec.ncol, len(x), path, extra)
                        sys.exit(1)
            done += 1
        print(f"ok {k}: {spec.nrow} x {spec.ncol}, {len(x)} entries", flush=True)
    print(f"transpose fuzz: {done} runs bit-exact")


if __name__ == "__main__":
    main()
