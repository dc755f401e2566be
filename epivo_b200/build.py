"""Build libepivo_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with
the repo snapshot to the GPU box)."""
from __future__ import annotations

import concurrent.futures
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "csrc", "build")
LIB = os.path.join(HERE, "libepivo_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
         "-Xcompiler", "-fPIC", "-Xptxas", "-v"]
# FMA contraction is on: every place that must reproduce OpenCV's un-fused arithmetic bit for bit
# (Sampson error, K-normalisation) spells its operations with __dmul_rn / __dadd_rn / __fma_rn.


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(verbose: bool = False, force: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    srcs = sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(HERE, "..", "include", "epivo_b200.h"))
    jobs = []
    for s in srcs:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJ, s[:-3] + ".o")
        if force or _stale(obj, [src] + hdrs):
            jobs.append((src, obj))

    def run(job):
        src, obj = job
        p = subprocess.run([NVCC, *FLAGS, "-c", src, "-o", obj], capture_output=True, text=True)
        return src, p

    with concurrent.futures.ThreadPoolExecutor(max_workers=8) as ex:
        for src, p in ex.map(run, jobs):
            if verbose or p.returncode:
                sys.stderr.write(f"== nvcc {os.path.basename(src)}\n{p.stdout}{p.stderr}\n")
            if p.returncode:
                raise RuntimeError(f"nvcc failed on {src}")
            log = os.path.join(OBJ, os.path.basename(src)[:-3] + ".ptxas.log")
            with open(log, "w") as f:
                f.write(p.stderr)
    objs = [os.path.join(OBJ, s[:-3] + ".o") for s in srcs]
    if jobs or _stale(LIB, objs):
        p = subprocess.run([NVCC, "-shared", "-o", LIB, *objs, "-lcudart"], capture_output=True, text=True)
        if p.returncode:
            sys.stderr.write(p.stdout + p.stderr)
            raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv))
