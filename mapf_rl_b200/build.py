"""Builds libmapf_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

Every translation unit is compiled on its own (in parallel) and the objects are linked into the shared library, so a
change to one kernel file recompiles that file only.  `MAPF_ENABLE_DIAG=1 python -m mapf_rl_b200.build --diag` builds
`libmapf_b200_diag.so` with the diagnosis flags compiled in (profiles/ only; never loaded by the package by default)."""
from __future__ import annotations

import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
OBJ_DIR = os.path.join(_HERE, "build")
# MAPF_B200_LIB points the package at another build of the library (A/B runs of two builds on one GPU box); such a
# library is used as it is, never rebuilt
LIB_OVERRIDE = os.environ.get("MAPF_B200_LIB")
LIB_PATH = LIB_OVERRIDE or os.path.join(_HERE, "libmapf_b200.so")
DIAG_LIB_PATH = os.path.join(_HERE, "libmapf_b200_diag.so")
SOURCES = ["mapf_rollout_occ8.cu", "mapf_rollout_occ10.cu", "mapf_rollout_occ12.cu", "mapf_rollout_occ16.cu", "mapf_step_kernels.cu", "mapf_abi.cu",
           "mapf_env_kernels.cu", "mapf_rollout_kernels.cu", "mapf_reset_kernels.cu", "mapf_per_kernels.cu", "mapf_replay_kernels.cu",
           "mapf_cbs.cu", "mapf_plan_kernels.cu"]
HEADERS = ["mapf_common.cuh", "mapf_step_device.cuh", "mapf_bfs_device.cuh", "mapf_reset_device.cuh", "mapf_rollout_device.cuh",
           os.path.join("..", "..", "include", "mapf_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build libmapf_b200.so")


def _deps():
    return [os.path.join(CSRC, s) for s in SOURCES] + [os.path.normpath(os.path.join(CSRC, h)) for h in HEADERS]


def is_stale() -> bool:
    if LIB_OVERRIDE:
        return False
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(d) > t for d in _deps())


def build(force: bool = False, verbose: bool = False, diag: bool = False) -> str:
    lib = DIAG_LIB_PATH if diag else LIB_PATH
    if not diag and not force and not is_stale():
        return lib
    nvcc = _nvcc()
    os.makedirs(OBJ_DIR, exist_ok=True)
    header_time = max(os.path.getmtime(os.path.normpath(os.path.join(CSRC, h))) for h in HEADERS)
    extra = ["-DMAPF_ENABLE_DIAG"] if diag else []
    if verbose:
        extra += ["-Xptxas", "-v"]
    suffix = ".diag.o" if diag else ".o"

    def compile_one(src):
        obj = os.path.join(OBJ_DIR, os.path.splitext(src)[0] + suffix)
        path = os.path.join(CSRC, src)
        if not force and os.path.exists(obj) and os.path.getmtime(obj) > max(os.path.getmtime(path), header_time):
            return obj
        cmd = [nvcc, *NVCC_FLAGS, *extra, "-c", path, "-o", obj]
        if verbose:
            print(" ".join(cmd))
        r = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
        if verbose or r.returncode != 0:
            print(r.stdout + r.stderr)
        if r.returncode != 0:
            raise subprocess.CalledProcessError(r.returncode, cmd)
        return obj

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", lib, *objs], cwd=CSRC)
    return lib


if __name__ == "__main__":
    import sys
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, diag="--diag" in sys.argv))
