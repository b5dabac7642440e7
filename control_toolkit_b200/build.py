"""Build libctk_b200.so in-tree with nvcc for sm_100a (one nvcc job per translation unit, run in parallel).

    python -m control_toolkit_b200.build [--force] [--verbose]

The .so is git-ignored but travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import concurrent.futures as cf
import hashlib
import os
import shutil
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libctk_b200.so")
UNITS = ["ctk_engine.cu", "ctk_mppi.cu", "ctk_cem.cu", "ctk_rpgd.cu", "ctk_batch.cu", "ctk_gru.cu", "ctk_env.cu", "ctk_env_rpgd.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
              "-I", INCLUDE, "-I", CSRC] + os.environ.get("CTK_NVCC_EXTRA", "").split()  # e.g. -DCTK_K1_MAXT2=1024


def _nvcc() -> str:
    n = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(n):
        raise RuntimeError("nvcc not found; control_toolkit_b200 has no CPU fallback and cannot be built without CUDA")
    return n


def _sources_digest() -> str:
    h = hashlib.sha256()
    for root in (CSRC, INCLUDE):
        for f in sorted(os.listdir(root)):
            if f.endswith((".cu", ".cuh", ".h")):
                with open(os.path.join(root, f), "rb") as fh:
                    h.update(f.encode())
                    h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _compile(unit: str, verbose: bool) -> str:
    obj = os.path.join(OBJ, unit.replace(".cu", ".o"))
    cmd = [_nvcc(), *NVCC_FLAGS, "-c", os.path.join(CSRC, unit), "-o", obj]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    t0 = time.perf_counter()
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for {unit}:\n{r.stdout}\n{r.stderr}")
    if os.environ.get("CTK_BUILD_TIMES"):
        sys.stderr.write(f"{unit}: {time.perf_counter() - t0:.1f} s\n")
    if verbose:
        sys.stderr.write(r.stderr)
    return obj


def build(force: bool = False, verbose: bool = False) -> str:
    units = list(UNITS)
    missing = [u for u in units if not os.path.exists(os.path.join(CSRC, u))]
    if missing:
        raise RuntimeError(f"translation units listed in build.py but not in csrc/: {missing}")
    os.makedirs(OBJ, exist_ok=True)
    stamp = os.path.join(OBJ, "digest.txt")
    digest = _sources_digest()
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == digest:
        return LIB
    with cf.ThreadPoolExecutor(max_workers=min(len(units), os.cpu_count() or 1)) as ex:
        objs = list(ex.map(lambda u: _compile(u, verbose), units))
    cmd = [_nvcc(), "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp, "w") as f:
        f.write(digest)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
