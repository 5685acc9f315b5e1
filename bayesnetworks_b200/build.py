"""Build libbn_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m bayesnetworks_b200.build [--force]

The shared library lands next to this file so that it travels with the repo
snapshot to the GPU box; it is git-ignored (source-only history).  The three
translation units compile in parallel.  BN_B200_DEV_K8=1 is a developer switch
for kernel experiments: only the MaxPar <= 8 chain kernels are instantiated
(a third of the compile time); never used by __graft_entry__.build().
BN_B200_DIAG=1 compiles the per-phase cycle counters in (bn_chain_stats.phase_cycles).
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_obj")
LIB = os.path.join(HERE, "libbn_b200.so")
SOURCES = ["bn_api.cu", "gram.cu", "kernels.cu"]
HEADERS = ["bn_common.cuh", "chain_core.cuh", "rng_core.cuh", "score_core.cuh", "sweep_log.cuh", "gram.h", "kernels.h",
           os.path.join("..", "..", "include", "bn_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force: bool = False, verbose: bool = False, dev_k8: bool | None = None) -> str:
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "nvcc")
    if dev_k8 is None:
        dev_k8 = os.environ.get("BN_B200_DEV_K8") == "1"
    flags = NVCC_FLAGS + (["-DBN_DEV_BUILD_K8_ONLY"] if dev_k8 else [])
    if os.environ.get("BN_B200_DIAG") == "1":  # per-phase cycle counters in bn_chain_stats.phase_cycles
        flags = flags + ["-DBN_PHASE_CYCLES"]
    os.makedirs(OBJ, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        res = subprocess.run([nvcc] + flags + ["-c", "-o", obj, os.path.join(CSRC, src)], capture_output=True, text=True)
        return obj, res

    with ThreadPoolExecutor(len(SOURCES)) as ex:
        results = list(ex.map(compile_one, SOURCES))
    out = "".join(r.stdout + r.stderr for _, r in results)
    ok = all(r.returncode == 0 for _, r in results)
    if ok:
        link = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "--shared", "-o", LIB] +
                              [o for o, _ in results], capture_output=True, text=True)
        out += link.stdout + link.stderr
        ok = link.returncode == 0
    if verbose or not ok:
        sys.stderr.write(out)
    if not ok:
        raise RuntimeError("nvcc failed building libbn_b200.so")
    with open(os.path.join(CSRC, "_ptxas.log"), "w") as fh:
        fh.write(out)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
