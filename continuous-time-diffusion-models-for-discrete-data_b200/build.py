"""Build recipe for libctdd_b200.so (hand-written sm_100a kernels + the C ABI of include/ctdd.h).

nvcc cross-compiles for sm_100a without a GPU; objects are compiled in parallel and linked into a shared
library that lives IN-TREE next to this file (git-ignored, but it travels to the GPU box with the snapshot).
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
BUILD = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libctdd_b200.so")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17", "--expt-extended-lambda", "--expt-relaxed-constexpr",
    "-Xcompiler", "-fPIC", "-I", INCLUDE,
]


def _sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _headers():
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hs += [os.path.join(INCLUDE, f) for f in os.listdir(INCLUDE) if f.endswith(".h")]
    return hs


def _newer(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu under csrc/ for sm_100a and link libctdd_b200.so. Returns the library path."""
    os.makedirs(BUILD, exist_ok=True)
    srcs, hdrs = _sources(), _headers()
    jobs = []
    for s in srcs:
        o = os.path.join(BUILD, os.path.basename(s)[:-3] + ".o")
        if force or _newer(o, [s] + hdrs + [os.path.abspath(__file__)]):
            jobs.append((s, o))

    def compile_one(job):
        s, o = job
        cmd = [NVCC] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {s}:\n{r.stdout}\n{r.stderr}")
        return r.stderr

    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            for log in ex.map(compile_one, jobs):
                if verbose and log:
                    sys.stderr.write(log)
    objs = [os.path.join(BUILD, os.path.basename(s)[:-3] + ".o") for s in srcs]
    if force or jobs or _newer(LIB, objs):
        cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-lcuda"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
