"""Builds rcppsparse_b200/libsparse_b200.so (and the tools) in-tree with nvcc for sm_100a.

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.  nvcc
cross-compiles here without a GPU.  Rebuilds only when a source is newer than the output.
"""
from __future__ import annotations

import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
OBJ = os.path.join(PKG, "build")
LIB = os.path.join(PKG, "libsparse_b200.so")
MICROBENCH = os.path.join(PKG, "microbench")

LIB_SOURCES = ["capi.cu", "blockcache.cu", "sweep.cu", "scan.cu", "validate.cu", "bands.cu", "transpose.cu", "transpose_split.cu", "bmc.cu", "synth.cu", "exchange.cu", "sharded.cu", "extract.cu", "crossprod.cu", "spmm.cu", "hostcopy.cu", "vars.cu"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xptxas", "-v",
              "--expt-relaxed-constexpr"] + ARCH


def nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: libsparse_b200 can only be built with the CUDA toolkit")
    return exe


def _deps():
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(ROOT, "include", "sparse_b200.h"))
    return hdrs


def _stale(out: str, srcs) -> bool:
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    return any(os.path.getmtime(s) > t for s in srcs)


def _compile(src: str, obj: str, log_dir: str) -> str:
    cmd = [nvcc()] + NVCC_FLAGS + ["-c", src, "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    with open(os.path.join(log_dir, os.path.basename(src) + ".ptxas.log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
    return obj


def build_library(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    deps = _deps()
    jobs = []
    for name in LIB_SOURCES:
        src = os.path.join(CSRC, name)
        obj = os.path.join(OBJ, name.replace(".cu", ".o"))
        if force or _stale(obj, [src] + deps):
            jobs.append((src, obj))
    if jobs:
        if verbose:
            print(f"[build] nvcc sm_100a: {', '.join(os.path.basename(s) for s, _ in jobs)}", file=sys.stderr)
        with cf.ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            for fut in [ex.submit(_compile, s, o, OBJ) for s, o in jobs]:
                fut.result()
    objs = [os.path.join(OBJ, n.replace(".cu", ".o")) for n in LIB_SOURCES]
    if force or jobs or _stale(LIB, objs):
        cmd = [nvcc(), "-shared", "-o", LIB] + objs + ARCH
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


def build_microbench(force: bool = False) -> str:
    src = os.path.join(CSRC, "microbench.cu")
    if not os.path.exists(src):
        return ""
    if force or _stale(MICROBENCH, [src] + _deps()):
        cmd = [nvcc(), "-O3", "-std=c++17", "-lineinfo"] + ARCH + [src, "-o", MICROBENCH]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on microbench:\n{r.stdout}\n{r.stderr}")
    return MICROBENCH


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose=True))
    mb = build_microbench(force="--force" in sys.argv)
    if mb:
        print(mb)
