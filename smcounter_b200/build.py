"""Builds libsmc_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libsmc_b200.so")
SOURCES = ["smc_api.cu"]
HEADERS = ["smc_common.cuh", "smc_sort.cuh", "smc_pileup.cuh", "smc_stats.cuh", "smc_upload.cuh", os.path.join("..", "..", "include", "smc_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-fmad=false",                 # FP64 parity: no FMA contraction anywhere in the statistics
              "-shared", "-Xcompiler", "-fPIC"]


def needs_build() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


BAMIO_OUT = os.path.join(HERE, "libsmc_bamio.so")
BAMIO_SRC = os.path.join(CSRC, "smc_bamio.cpp")
ROWS_SRC = os.path.join(CSRC, "smc_rows.cpp")            # host-side output stage (include/smc_rows.h), same library
BAMIO_HDR = os.path.join(HERE, "..", "include", "smc_bamio.h")
ROWS_HDR = os.path.join(HERE, "..", "include", "smc_rows.h")
SOA_SRC = os.path.join(CSRC, "smc_soa.cpp")              # host-side batch packer (include/smc_soa.h), same library
SOA_HDR = os.path.join(HERE, "..", "include", "smc_soa.h")


def build_bamio(force: bool = False) -> str:
    """Host-side BAM decoder (C++17, zlib, threads) -> libsmc_bamio.so."""
    if not force and os.path.exists(BAMIO_OUT) and os.path.getmtime(BAMIO_OUT) >= max(os.path.getmtime(f) for f in (BAMIO_SRC, BAMIO_HDR, ROWS_SRC, ROWS_HDR, SOA_SRC, SOA_HDR, os.path.join(CSRC, "smc_inflate.h"))):
        return BAMIO_OUT
    cmd = [os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-o", BAMIO_OUT, BAMIO_SRC, ROWS_SRC, SOA_SRC, "-lz"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("g++ failed building libsmc_bamio.so")
    return BAMIO_OUT


def build(force: bool = False, verbose: bool = False) -> str:
    build_bamio(force)
    if not force and not needs_build():
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    extra = os.environ.get("SMC_NVCC_EXTRA", "").split()          # tuning builds only, e.g. SMC_NVCC_EXTRA=-DK3_GATHER=8
    out = os.environ.get("SMC_B200_OUT", OUT)
    cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", out] + SOURCES
    r = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed building libsmc_b200.so")
    if verbose:
        sys.stderr.write(r.stderr)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
