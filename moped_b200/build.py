"""Builds libmoped_cuda.so in-tree for sm_100a with nvcc (cross-compiles without a GPU).

    python -m moped_b200.build [--force]

The library lands in moped_b200/lib/libmoped_cuda.so; it is git-ignored but travels to the GPU box
with the gpurun snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libmoped_cuda.so")
SOURCES = ["api.cu", "match.cu", "adaptive.cu", "cluster.cu", "pose.cu", "pose_exact.cu", "pose_depth.cu", "filter.cu", "pipeline.cu", "depth_frames.cu", "sift.cu", "undistort.cu", "linkage.cu", "sm_partition.cu", "model_db.cpp"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall"] + os.environ.get("MOPED_NVCC_FLAGS", "").split()
LIB = os.environ.get("MOPED_LIB", LIB)
# pose.cu flushes denormals like the reference process does (SURVEY.md Appendix C)
# sift.cu keeps multiply and add separate so that its sums round like the reference's scalar code; filter.cu likewise (its
# reprojections and scores then equal the oracle's bit for bit: ownership and pruning decisions can never differ by a rounding)
PER_FILE = {"pose.cu": ["-ftz=true"], "pose_depth.cu": ["-ftz=true", "-fmad=false"], "pose_exact.cu": ["-ftz=true", "-fmad=false"], "sift.cu": ["-fmad=false"], "filter.cu": ["-fmad=false"], "linkage.cu": ["-fmad=false"],
            "adaptive.cu": ["-Xcompiler", "-ffp-contract=off"],   # its host arithmetic (ratio curves) rounds like a strict-IEEE build
            "undistort.cu": ["-Xcompiler", "-ffp-contract=off"]}  # likewise its host remap tables (OpenCV's scalar loop in double)


def nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    # this file is a dependency too: it holds the per-file compiler flags
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "moped_cuda.h"), os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(LIBDIR, os.path.splitext(src)[0] + ".o")
        cmd = [nvcc(), *ARCH, *COMMON, *PER_FILE.get(src, []), "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- {src}\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    subprocess.check_call([nvcc(), *ARCH, "-shared", "-o", LIB, *objs, "-lcudart"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))


def build_stage_driver() -> str:
    """tests/cpp/stages_main.cpp: the C++ stage classes driven through the plugin API (stand-alone build against
    moped_b200/stages/moped_api.hpp). Host-only g++ build; links libmoped_cuda.so."""
    root = os.path.dirname(HERE)
    out = os.path.join(LIBDIR, "stages_main")
    src = os.path.join(root, "tests", "cpp", "stages_main.cpp")
    deps = [src] + [os.path.join(HERE, "stages", f) for f in os.listdir(os.path.join(HERE, "stages"))]
    if os.path.exists(out) and all(os.path.getmtime(d) <= os.path.getmtime(out) for d in deps):
        return out
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-I" + os.path.join(root, "include"), "-I" + os.path.join(HERE, "stages"),
                           src, "-o", out, "-L" + LIBDIR, "-lmoped_cuda", "-Wl,-rpath,$ORIGIN"])
    return out
