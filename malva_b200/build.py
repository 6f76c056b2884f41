"""In-tree build of libmalva_gpu.so (hand-written sm_100a kernels + C ABI) and of the C++ host
program malva-geno (csrc/host/, the drop-in `malva-geno index|call` CLI over that C ABI).

    python -m malva_b200.build [--force] [-v]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the
GPU box with the repository snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmalva_gpu.so")
CLI = os.path.join(HERE, "malva-geno")
SOURCES = ["malva_gpu.cu"]
HEADERS = ["xxh3.cuh", "geno.cuh", "index.cuh", "kernels.cuh", "count.cuh", os.path.join("host", "signatures.hpp"),
           os.path.join("..", "..", "include", "malva_gpu.h")]
HOST_DIR = os.path.join(CSRC, "host")
HOST_SOURCES = ["malva_geno.cpp"]
HOST_HEADERS = ["signatures.hpp", "vcf_io.hpp", "kmc_db.hpp", "index_file.hpp"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "--fmad=false",  # the reference is built without FMA contraction (CMakeLists.txt has no -march)
    "-shared", "-Xcompiler", "-fPIC", "-cudart", "static",
]


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def _find(*cands):
    return next((p for p in cands if os.path.exists(p)), None)


def _cli_stale() -> bool:
    if not os.path.exists(CLI):
        return True
    t = os.path.getmtime(CLI)
    deps = [os.path.join(HOST_DIR, s) for s in HOST_SOURCES + HOST_HEADERS] + \
        [os.path.join(HERE, "..", "include", "malva_gpu.h"), LIB, os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build_cli(force: bool = False) -> str:
    """g++ build of malva-geno against libmalva_gpu.so (found at run time next to the binary, rpath $ORIGIN)."""
    if not force and not _cli_stale():
        return CLI
    stdcxx = _find("/usr/lib/x86_64-linux-gnu/libstdc++.so.6", "/lib/x86_64-linux-gnu/libstdc++.so.6")
    zstd = _find("/usr/lib/x86_64-linux-gnu/libzstd.so.1", "/lib/x86_64-linux-gnu/libzstd.so.1")
    if zstd is None:
        raise RuntimeError("libzstd.so.1 not found (needed for the index file)")
    cmd = [os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-Wall", "-Wextra", "-o", CLI] + \
        [os.path.join(HOST_DIR, s) for s in HOST_SOURCES] + [LIB, zstd, "-lz", "-lpthread", "-Wl,-rpath,$ORIGIN"]
    if stdcxx:
        cmd += ["-nostdlib++", stdcxx, "-lm"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("g++ failed building malva-geno")
    if r.stderr.strip():
        sys.stderr.write(r.stderr)
    return CLI


def build(force: bool = False, verbose: bool = False) -> str:
    lib = _build_lib(force, verbose)
    build_cli(force)
    return lib


def _build_lib(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.exists(nvcc):
        nvcc = "nvcc"
    # the image's g++ wrapper only resolves the static libstdc++; use the shared one so the
    # library can live in a process that already loaded libstdc++.so.6 (torch, numpy)
    stdcxx = next((p for p in ("/usr/lib/x86_64-linux-gnu/libstdc++.so.6", "/lib/x86_64-linux-gnu/libstdc++.so.6")
                   if os.path.exists(p)), None)
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else [])
    if stdcxx:
        cmd += ["-Xcompiler", "-nostdlib++", "-Xlinker", stdcxx]
    cmd += ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed building libmalva_gpu.so")
    if verbose:
        sys.stderr.write(r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
