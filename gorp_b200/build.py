"""In-tree build of libgorpcuda.so for sm_100a (nvcc cross-compiles without a GPU).

    python -m gorp_b200.build [--force]

The shared library lands next to this file (gorp_b200/libgorpcuda.so): git-ignored, but it travels to the
GPU box with the repo snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libgorpcuda.so")

HOST_SOURCES = [os.path.join(CSRC, "host", f) for f in
                ("common.cpp", "definition.cpp", "automata.cpp", "capture.cpp", "model.cpp", "fused.cpp", "walktables.cpp", "tails.cpp")]
CUDA_SOURCES = [os.path.join(CSRC, "engine.cu"), os.path.join(CSRC, "kernels", "kernels.cu"),
                os.path.join(CSRC, "kernels", "fast.cu"),
                os.path.join(CSRC, "kernels", "dfawalk.cu"),
                os.path.join(CSRC, "kernels", "capwalk.cu"), os.path.join(CSRC, "kernels", "tailwalk.cu"), os.path.join(CSRC, "kernels", "utf8.cu"), os.path.join(CSRC, "kernels", "matchall.cu"), os.path.join(CSRC, "kernels", "pike.cu")]
OBJ_DIR = os.path.join(HERE, "_obj")
COMPILE_FLAGS = ["-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
                 "-Xcompiler", "-fPIC,-Wall", "-I", os.path.join(ROOT, "include")]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    deps = list(sources)
    for d in (os.path.join(CSRC, "host"), os.path.join(CSRC, "kernels"), os.path.join(ROOT, "include")):
        deps += [os.path.join(d, f) for f in os.listdir(d)]
    return any(os.path.getmtime(s) > t for s in deps)


def nvcc_path():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _compile_one(args):
    src, obj, verbose = args
    cmd = [nvcc_path()] + COMPILE_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
    subprocess.check_call(cmd)
    return obj


def build(force=False, verbose=False):
    """One object per source (compiled in parallel, only what changed), then one link."""
    from concurrent.futures import ThreadPoolExecutor
    import fcntl
    srcs = CUDA_SOURCES + HOST_SOURCES
    if not force and not _newer(LIB, srcs):
        return LIB
    os.makedirs(OBJ_DIR, exist_ok=True)
    lock = open(os.path.join(OBJ_DIR, ".lock"), "w")
    fcntl.flock(lock, fcntl.LOCK_EX)  # several ranks may get here at once (torchrun): one builds, the others wait
    if not force and not _newer(LIB, srcs):
        return LIB
    headers = []
    for d in (os.path.join(CSRC, "host"), os.path.join(CSRC, "kernels"), os.path.join(ROOT, "include")):
        headers += [os.path.join(d, f) for f in os.listdir(d) if f.endswith((".h", ".hpp", ".cuh"))]
    newest_header = max(os.path.getmtime(h) for h in headers)
    jobs, objs = [], []
    for s in srcs:
        obj = os.path.join(OBJ_DIR, os.path.basename(s) + ".o")
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(s), newest_header):
            jobs.append((s, obj, verbose))
    with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4) or 1) as ex:
        list(ex.map(_compile_one, jobs))
    subprocess.check_call([nvcc_path(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
