"""Build libkmer_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.environ.get("KMER_B200_LIB_OUT") or os.path.join(HERE, "libkmer_b200.so")   # KMER_B200_LIB_OUT: tuning builds
SOURCES = ["capi.cu", "build_kernels.cu", "onesweep.cu", "search_kernels.cu", "search_lean.cu", "search_approx.cu", "search_seeds.cu", "record_votes.cu", "spectrum.cu", "route_kernels.cu", "fastx_kernels.cu", "synth.cu", "host_pack.cpp"]
HEADERS = ["common.cuh", "radix.cuh", "launch.h", "host_pack.h", "query_pack.cuh", os.path.join("..", "..", "include", "kmer_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC,-O3,-Wall", "-Xptxas", "-v"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    objs = []
    build_dir = os.environ.get("KMER_B200_BUILD_DIR") or os.path.join(HERE, "build")
    os.makedirs(build_dir, exist_ok=True)
    log = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(build_dir, os.path.splitext(src)[0] + ".o")
        extra = os.environ.get("KMER_B200_NVCC_EXTRA", "").split()   # tuning experiments, e.g. -DKB_SEARCH_MIN_BLOCKS=6
        if src.endswith(".cpp"):   # plain host code (the query packer): x86-64-v3 for BMI2 PEXT
            extra = [*extra, "-Xcompiler", "-march=x86-64-v3"]
        cmd = [_nvcc(), *NVCC_FLAGS, *extra, "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = None
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"==== {src}\n{out}")
        if p.returncode != 0:
            failed = src
    if failed:
        sys.stderr.write("\n".join(log))
        raise RuntimeError(f"nvcc failed on {failed}")
    cmd = [_nvcc(), "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart", "-lpthread"]
    subprocess.run(cmd, check=True)
    with open(os.path.join(build_dir, "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
