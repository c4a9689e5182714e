"""In-tree build of libgslift.so (nvcc, sm_100a only).  `python -m` friendly:

    python 3d_gaussian_splatting_project_b200/build.py [--force] [-v]

Every .cu is compiled to an object under csrc/_obj (in parallel, only when it or a header is
newer) and linked into libgslift.so next to this file, so the library travels with the
repository snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_obj")
LIB = os.path.join(HERE, "libgslift.so")
SOURCES = ["api.cu", "lift.cu", "lift_order.cu", "lift_sort.cu", "kmeans.cu", "kmeans_tc.cu", "kmeans_ordered.cu",
           "ply_format.cu", "host_stage.cu", "viewer.cu", "region_growing.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-fmad=false",            # no implicit contraction: fused ops are spelled fma() in the source
    "-Xcompiler", "-fPIC", "-Xcompiler", "-pthread",
    "-I", os.path.join(ROOT, "include"),
]


def _headers():
    return [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))] + \
           [os.path.join(ROOT, "include", "gslift.h"), __file__]


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _newer(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def _env():
    env = dict(os.environ)
    env.pop("CC", None)       # the image exports a CC wrapper that nvcc must not pick up
    env.pop("CXX", None)
    return env


def stale() -> bool:
    """True when libgslift.so is missing or older than any source, header or this script."""
    return _newer(LIB, [os.path.join(CSRC, s) for s in _sources()] + _headers())


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(OBJ, exist_ok=True)
    hdrs = _headers()
    env = _env()

    def compile_one(src: str) -> str:
        obj = os.path.join(OBJ, src[:-3] + ".o")
        path = os.path.join(CSRC, src)
        if force or _newer(obj, [path] + hdrs):
            cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, path]
            subprocess.check_call(cmd, env=env)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as pool:
        objs = list(pool.map(compile_one, _sources()))
    subprocess.check_call([nvcc, "-shared", "-Xcompiler", "-pthread", "-o", LIB] + objs, env=env)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
