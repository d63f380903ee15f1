"""Build libradex_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libradex_b200.so")
SOURCES = ["radex_b200.cu", "moldata.cpp"]
HEADERS = [os.path.join(CSRC, "internal.h"), os.path.join(CSRC, "lvg_v2.cuh"), os.path.join(CSRC, "lvg_small.cuh"),
           os.path.join(CSRC, "stretch.cuh"), os.path.join(CSRC, "chain_stats.cuh"), os.path.join(CSRC, "chain_marginals.cuh"),
           os.path.join(CSRC, "predict_sled.cuh"),
           os.path.join(ROOT, "include", "radex_b200.h")]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + HEADERS
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    cmd = [nvcc_path(), "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
           "-Xcompiler", "-fPIC", "-shared", "-I", os.path.join(ROOT, "include"), "-I", CSRC,
           "-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building libradex_b200.so")
    if verbose:
        sys.stderr.write(res.stdout + res.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force=True, verbose="-v" in sys.argv))
