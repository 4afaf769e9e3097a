"""Builds libgymcellular_b200.so in-tree with nvcc for sm_100a (no JIT cache, no torch extension).

    python -m gym_cellular_b200.build [--force]

The .so is git-ignored but travels with the repo snapshot to the GPU box.
"""
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB_DIR = os.environ.get("GC_B200_LIB_DIR") or os.path.join(PKG, "lib")     # override: A/B builds of tuning runs
LIB_PATH = os.path.join(LIB_DIR, "libgymcellular_b200.so")
SOURCES = ["gc_kernels.cu", "gc_cell_fast.cu", "gc_cell_pair8.cu", "gc_cell_packed.cu", "gc_grid.cu", "gc_rollout.cu", "gc_tables.cu", "gc_api.cu"]
HEADERS = [os.path.join(CSRC, "gc_internal.h"), os.path.join(CSRC, "gc_device.cuh"), os.path.join(REPO, "include", "gym_cellular_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-I" + os.path.join(REPO, "include"), "-I" + CSRC]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build libgymcellular_b200.so")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    mt = os.path.getmtime(target)
    return any(os.path.getmtime(d) > mt for d in deps)


def build(force=False, verbose=False):
    os.makedirs(LIB_DIR, exist_ok=True)
    nvcc = _nvcc()
    objs = []
    procs = []
    for src in SOURCES:
        path = os.path.join(CSRC, src)
        obj = os.path.join(LIB_DIR, src.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, [path] + HEADERS):
            extra = os.environ.get("GC_NVCC_EXTRA", "").split()       # e.g. -DGC_PACKED_MINB=3 (tuning runs)
            cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", path, "-o", obj]
            procs.append((cmd, subprocess.Popen(cmd)))
    for cmd, p in procs:
        if p.wait() != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    if force or procs or _stale(LIB_PATH, objs):
        cmd = [nvcc, "-shared", "-o", LIB_PATH] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
        subprocess.check_call(cmd)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
