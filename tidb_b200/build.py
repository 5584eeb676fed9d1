"""Builds tidb_b200/csrc/libtidbgpu.so in-tree with nvcc for sm_100a (B200 only, no other arch).

    python -m tidb_b200.build            # incremental
    python -m tidb_b200.build --force

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "build")
LIB = os.path.join(CSRC, "libtidbgpu.so")
SOURCES = ["runtime.cu", "join.cu", "agg.cu", "vec.cu", "partition.cu", "codec.cu", "topn.cu", "sort.cu"]
HEADERS = ["common.cuh", "join_kernels.cuh", "partition_kernels.cuh", "tma.cuh", "agg_update.cuh", os.path.join("..", "..", "include", "tidbgpu.h")]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "--expt-relaxed-constexpr"]


def nvcc() -> str:
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found")
    return p


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]
    srcs = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    jobs = []
    for s in srcs:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJ, s.replace(".cu", ".o"))
        if force or _stale(obj, [src] + hdrs):
            jobs.append((src, obj))

    def compile_one(job):
        src, obj = job
        cmd = [nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        return r.stderr

    with ThreadPoolExecutor(max_workers=8) as ex:
        logs = list(ex.map(compile_one, jobs))
    if verbose:
        for l in logs:
            print(l)
    objs = [os.path.join(OBJ, s.replace(".cu", ".o")) for s in srcs]
    if force or jobs or _stale(LIB, objs):
        cmd = [nvcc(), "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart_static", "-lpthread", "-ldl", "-lrt"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
