"""In-tree builds of the native libraries.

    libfastore_host.so   host C++: FASTQ parser, chunk cutter, bin-file writer, synthetic generator
    libfastore_b200.so   the C ABI (include/fastore_b200.h) + the sm_100a CUDA kernels

Both are written next to this file (git-ignored, but they travel to the GPU box with the gpurun
snapshot).  nvcc cross-compiles sm_100a without a GPU.  `python -m fastore_b200.build` builds all.
"""
from __future__ import annotations

import os
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
HOST_LIB = PKG / "libfastore_host.so"
CUDA_LIB = PKG / "libfastore_b200.so"
CLI_BIN = PKG / "fastore_bin_b200"

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CXX = os.environ.get("CXX", "g++")

HOST_SOURCES = sorted((CSRC / "host").glob("*.cpp"))
CUDA_SOURCES = sorted(CSRC.glob("*.cu"))

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall",
    "--expt-relaxed-constexpr",
]


def _newer(target: Path, deps) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(Path(d).stat().st_mtime > t for d in deps)


def _run(cmd, verbose=False):
    if verbose:
        print(" ".join(str(c) for c in cmd), flush=True)
    r = subprocess.run([str(c) for c in cmd], capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError(f"build failed: {' '.join(str(c) for c in cmd)}")
    if verbose and (r.stdout or r.stderr):
        print(r.stdout + r.stderr)
    return r


def build_host(force=False, verbose=False) -> Path:
    deps = [s for s in HOST_SOURCES if s.name != "main.cpp"]
    hdrs = list((CSRC / "host").glob("*.h")) + [ROOT / "include" / "fastore_b200.h"]
    if force or _newer(HOST_LIB, deps + hdrs):
        _run([CXX, "-std=c++17", "-O2", "-fPIC", "-shared", "-pthread", "-Wall", "-Wextra",
              "-o", HOST_LIB, *deps], verbose)
    return HOST_LIB


def build_cuda(force=False, verbose=False, extra_flags=()) -> Path:
    hdrs = list(CSRC.glob("*.cuh")) + list(CSRC.glob("*.h")) + [ROOT / "include" / "fastore_b200.h"]
    if force or _newer(CUDA_LIB, CUDA_SOURCES + hdrs):
        _run([NVCC, *NVCC_FLAGS, *extra_flags, "-shared", "-o", CUDA_LIB, *CUDA_SOURCES, "-lcudart"], verbose)
    return CUDA_LIB


def build_cli(force=False, verbose=False) -> Path:
    main = CSRC / "host" / "main.cpp"
    if not main.exists():
        return CLI_BIN
    build_host(force, verbose)
    build_cuda(force, verbose)
    if force or _newer(CLI_BIN, [main, HOST_LIB, CUDA_LIB]):
        _run([CXX, "-std=c++17", "-O2", "-pthread", "-Wall", "-o", CLI_BIN, main,
              f"-L{PKG}", "-lfastore_host", "-lfastore_b200", f"-Wl,-rpath,$ORIGIN"], verbose)
    return CLI_BIN


def build_oracle(verbose=False) -> None:
    """Build the CPU checkers (test infrastructure): the C port always, the compiled reference only
    when FASTORE_REFERENCE names a checkout of the reference's sources (into oracle/_ref)."""
    _run(["make", "-C", ROOT / "oracle", "port"], verbose)
    ref = os.environ.get("FASTORE_REFERENCE")
    if ref and Path(ref).is_dir():
        _run(["make", "-C", ROOT / "oracle", "-j8", f"REF={ref}", "ref"], verbose)
        if CUDA_LIB.exists():                      # the reference's fastore_bin with the C ABI bound in (integration/)
            _run(["make", "-C", ROOT / "oracle", f"REF={ref}", "ref_gpu"], verbose)


def build_all(force=False, verbose=False) -> None:
    build_host(force, verbose)
    build_cuda(force, verbose)
    build_cli(force, verbose)
    build_oracle(verbose)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv, verbose=True)
