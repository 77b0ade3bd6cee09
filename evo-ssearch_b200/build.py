"""Builds ``libevs.so`` in-tree with nvcc for sm_100a (the only target).

    python evo-ssearch_b200/build.py [--force]

The library is written next to this file so that it travels to the GPU box with the repo snapshot;
it is git-ignored.  ``__graft_entry__.build()`` calls :func:`build_libevs`.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libevs.so")
SOURCES = ["evs_scan_f32_512.cu", "evs_scan_f32_narrow.cu", "evs_scan_f32_wide.cu", "evs_scan_bf16_narrow.cu", "evs_scan_bf16_wide.cu", "evs_scan_i8.cu",
           "evs_scan_generic.cu", "evs_kernels.cu", "evs_api.cu", "evs_tc.cu", "evs_tc2.cu", "evs_large_k.cu"]
HEADERS = ["evs_common.cuh", "evs_scan.cuh", "evs_scan_launch.cuh", "evs_finalize.cuh", "evs_tc_common.cuh", "evs_internal.h", os.path.join("..", "..", "include", "evs.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-fvisibility=hidden,-O3",
    "-Xlinker", "--no-undefined",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(p) > t for p in deps if os.path.exists(p))


def build_libevs(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    objs = []
    procs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    hdr_t = max(os.path.getmtime(p) for p in [os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)] if os.path.exists(p))
    for s in SOURCES:
        o = os.path.join(HERE, "build", s.replace(".cu", ".o"))
        objs.append(o)
        # an object newer than its source, every header and this script is kept
        if not force and not verbose and os.path.exists(o) and os.path.getmtime(o) > max(hdr_t, os.path.getmtime(os.path.join(CSRC, s))):
            continue
        cmd = [_nvcc(), *NVCC_FLAGS[:-2], "-DEVS_BUILDING", "-c", os.path.join(CSRC, s), "-o", o]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    # symbols of include/evs.h are exported explicitly; everything else stays hidden
    link = [_nvcc(), "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a",
            "-Xcompiler", "-fPIC", "-Xlinker", "--no-undefined", "-lcudart"]
    subprocess.check_call(link)
    return LIB


if __name__ == "__main__":
    print(build_libevs(force="--force" in sys.argv, verbose="-v" in sys.argv))
