"""Builds the in-tree native libraries (nvcc, sm_100a only). Run: python -m inquistr_b200.build"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-shared", "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall",
]


def _stale(target: str, sources: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def build_libinqcall(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIBDIR, exist_ok=True)
    target = os.path.join(LIBDIR, "libinqcall.so")
    inc = os.path.join(os.path.dirname(HERE), "include")
    units = [os.path.join(CSRC, "inq_capi.cu"), os.path.join(CSRC, "inq_cohort_capi.cu"), os.path.join(CSRC, "inq_inflate_capi.cu")]
    sources = units + [os.path.join(CSRC, "inq_device.cuh"), os.path.join(CSRC, "inq_cohort.cuh"), os.path.join(CSRC, "inq_inflate.cuh"),
                       os.path.join(inc, "inqcall.h"), os.path.join(inc, "inqcohort.h"), os.path.join(inc, "inqbgzf.h")]
    if force or _stale(target, sources):
        cmd = ["nvcc", *NVCC_FLAGS, "-o", target, *units]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        subprocess.check_call(cmd)
    return target


def build_cli(force: bool = False) -> str:
    """C++ host `inquistr-b200` (CLI, BGZF/BAM reader, BED, TSV) linked against libinqcall.so."""
    bindir = os.path.join(HERE, "bin")
    os.makedirs(bindir, exist_ok=True)
    target = os.path.join(bindir, "inquistr-b200")
    host = os.path.join(CSRC, "host")
    sources = [os.path.join(host, "main.cpp"), os.path.join(host, "bam_reader.cpp"), os.path.join(host, "cohort_cli.cpp"),
               os.path.join(host, "shard_driver.cpp"), os.path.join(host, "call_common.cpp"), os.path.join(host, "cohort_call.cpp")]
    deps = sources + [os.path.join(host, f) for f in sorted(os.listdir(host)) if f.endswith(".hpp")] + [os.path.join(os.path.dirname(HERE), "include", "inqcall.h"),
                      os.path.join(os.path.dirname(HERE), "include", "inqcohort.h"),
                      os.path.join(LIBDIR, "libinqcall.so")]
    if force or _stale(target, deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-pthread", "-o", target, *sources,
                               "-L" + LIBDIR, "-linqcall", "-lz", "-Wl,-rpath,$ORIGIN/../lib"])
    return target


def build_all(force: bool = False, verbose: bool = False) -> list[str]:
    out = [build_libinqcall(force, verbose)]
    out.append(build_cli(force))
    return out


if __name__ == "__main__":
    for p in build_all(force="--force" in sys.argv, verbose="-v" in sys.argv):
        print(p)
