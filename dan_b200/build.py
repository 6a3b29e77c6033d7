"""Build the C-ABI shared library dan_b200/libdan_b200.so for sm_100a with nvcc.

    python -m dan_b200.build            # build what is stale
    python -m dan_b200.build --force

Every .cu is compiled to its own object (in parallel, only when stale) and the objects are linked into the library.
The library is built IN-TREE so that it travels with the repository snapshot to the GPU box; it and the objects are
git-ignored (*.so, *.o)."""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libdan_b200.so")
SOURCES = ["api.cu", "anchors.cu", "encode.cu", "postprocess.cu", "mining.cu", "routing.cu", "vote.cu", "detect_face.cu", "handoff.cu", "gather.cu"]
HEADERS = ["common.cuh", "heap_order.cuh", "sort.cuh", os.path.join(ROOT, "include", "dan_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-fmad=false",            # no FMA contraction: every fp32 op separately rounded
    "-Xcompiler", "-fPIC",
    "-I" + os.path.join(ROOT, "include"),
    "-I" + CSRC,
]


def _header_time():
    return max(os.path.getmtime(h if os.path.isabs(h) else os.path.join(CSRC, h)) for h in HEADERS)


def _compile(nvcc, src, obj, extra, verbose):
    cmd = [nvcc] + NVCC_FLAGS + extra + ["-c", src, "-o", obj]
    if verbose:
        print(" ".join(cmd))
    subprocess.run(cmd, check=True)


def build(force=False, verbose=False, extra_flags=()):
    nvcc = os.environ.get("NVCC", "nvcc")
    os.makedirs(OBJ, exist_ok=True)
    ht = max(_header_time(), os.path.getmtime(os.path.abspath(__file__)))
    jobs, objs = [], []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJ, s[:-3] + ".o")
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), ht):
            jobs.append((src, obj))
    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            for f in [ex.submit(_compile, nvcc, src, obj, list(extra_flags), verbose) for src, obj in jobs]:
                f.result()
    if jobs or not os.path.exists(LIB) or any(os.path.getmtime(o) > os.path.getmtime(LIB) for o in objs):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a"] + objs + ["-o", LIB]
        if verbose:
            print(" ".join(cmd))
        subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
    print(LIB)
