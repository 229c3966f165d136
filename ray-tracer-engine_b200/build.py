"""In-tree build of libore_b200.so (CUDA kernels + C ABI) for sm_100a.

`nvcc` cross-compiles without a GPU, so this runs in the build container; the resulting
.so is git-ignored but travels to the GPU box with the repo snapshot.  Every translation unit is
compiled to its own object (in parallel, only when stale) and the objects are linked into the library.
"""
from __future__ import annotations

import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
OBJ_DIR = os.path.join(PKG_DIR, "csrc", "_obj")
LIB_PATH = os.path.join(PKG_DIR, "libore_b200.so")
SOURCES = ["ore_capi.cu", "ore_scene_build.cu", "ore_mesh_refit.cu", "ore_mesh_build.cu"]
HEADERS = ["ore_kernels.cuh", "ore_primary.cuh", "ore_sweep.cuh", "ore_device.cuh", "ore_libm.cuh", "ore_clusters.h", "ore_scene_build.h", "ore_mesh_refit.h", "ore_mesh_build.h", "ore_stage_plan.h", os.path.join("..", "..", "include", "ore_render.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    # reference-exact sequences rely on unfused mul/add; filters use explicit fmaf
    "--fmad=false",
    "-Xcompiler", "-fPIC",
]


def find_nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise FileNotFoundError("nvcc not found; the render path has no non-CUDA fallback")


def _deps():
    return [os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]


def _newer(paths, t):
    return any(os.path.getmtime(d) > t for d in paths if os.path.isfile(d))


def is_stale() -> bool:
    if not os.path.isfile(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return _newer([os.path.join(CSRC, s) for s in SOURCES] + _deps(), t)


def _env():
    env = dict(os.environ)
    env.pop("CC", None)   # the image's CC/CXX point at a compiler without libgomp; nvcc uses the system g++
    env.pop("CXX", None)
    return env


def build_library(force: bool = False, verbose: bool = False, extra_flags=(), out: str | None = None) -> str:
    """out: path of a VARIANT library (tuning experiments built with extra -D flags, selected with ORE_LIB=...)"""
    target = out or LIB_PATH
    if not force and not extra_flags and not out and not is_stale():
        return LIB_PATH
    nvcc = find_nvcc()
    os.makedirs(OBJ_DIR, exist_ok=True)
    tag = ("_" + "_".join(f.strip("-").replace("=", "_") for f in extra_flags)) if extra_flags else ""
    jobs = []
    for s in SOURCES:
        obj = os.path.join(OBJ_DIR, s.replace(".cu", tag + ".o"))
        stale = force or not os.path.isfile(obj) or _newer([os.path.join(CSRC, s)] + _deps(), os.path.getmtime(obj))
        jobs.append((s, obj, stale))

    def compile_one(job):
        s, obj, stale = job
        if stale:
            cmd = [nvcc, *NVCC_FLAGS, *extra_flags, "-c", os.path.join(CSRC, s), "-o", obj]
            if verbose:
                print(" ".join(cmd), flush=True)
            subprocess.check_call(cmd, env=_env())
        return obj

    with ThreadPoolExecutor(max_workers=len(jobs)) as ex:
        objs = list(ex.map(compile_one, jobs))
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC", *objs, "-o", target]
    if verbose:
        print(" ".join(cmd), flush=True)
    subprocess.check_call(cmd, env=_env())
    return target


if __name__ == "__main__":
    print(build_library(force=True, verbose=True))
