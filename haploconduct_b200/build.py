"""In-tree build of libhc_b200.so (sm_100a only).  `python -m haploconduct_b200.build`."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libhc_b200.so")
NVCC = os.environ.get("HC_NVCC", "/usr/local/cuda/bin/nvcc")
HOST_CXX = "/usr/bin/g++"

CU_SOURCES = ["hc_kernels.cu", "hc_api.cu", "hc_fno.cu", "hc_fno_text.cu", "hc_dedup.cu", "hc_ingest.cu", "hc_pack.cu", "hc_consensus.cu", "hc_stage.cu", "hc_adjacency.cu"]
CPP_SOURCES = ["hc_tables.cpp", "hc_cons_final.cpp"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _newer(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIBDIR, exist_ok=True)
    hostdir = os.path.join(HERE, "host")
    deps = ([os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(hostdir, f) for f in os.listdir(hostdir)]
            + [os.path.join(HERE, "..", "include", "hc_b200.h")])
    if not force and not _newer(LIB, deps):
        return LIB
    objs = []
    for src in CPP_SOURCES:
        obj = os.path.join(LIBDIR, src + ".o")
        # plain g++: no FMA contraction, so the double score table is bit-identical to the reference build (makefile:6)
        cmd = [HOST_CXX, "-O2", "-std=c++14", "-fPIC", "-ffp-contract=off", "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd)
        objs.append(obj)
    for src in CU_SOURCES:
        obj = os.path.join(LIBDIR, src + ".o")
        cmd = [NVCC, "-ccbin", HOST_CXX, "-O3", "-std=c++14", "-lineinfo", *ARCH, "-Xcompiler", "-fPIC,-fopenmp,-O2",
               "-Xptxas", "-v" if verbose else "-O3", "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd)
        objs.append(obj)
    cmd = [NVCC, "-ccbin", HOST_CXX, "-shared", *ARCH, "-Xcompiler", "-fPIC,-fopenmp", "-o", LIB, *objs, "-lgomp"]
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    build_host(verbose)
    return LIB


def build_host(verbose: bool = False) -> str:
    """hc_edgecalc: the C++ host mirror of the reference's EdgeCalculator stage, linked against the C ABI."""
    host = os.path.join(HERE, "host")
    exe = os.path.join(LIBDIR, "hc_edgecalc")
    cmd = [HOST_CXX, "-O2", "-std=c++14", "-Wall", "-fopenmp", "-o", exe, os.path.join(host, "hc_edgecalc_main.cpp"),
           os.path.join(host, "hcb_host.cpp"), "-L" + LIBDIR, "-lhc_b200", "-lpthread", "-Wl,-rpath,$ORIGIN"]
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    # hc_fno: the FindNextOverlaps step (hcb::SRBuilder, hcb_fno.h) on the C ABI
    fno = os.path.join(LIBDIR, "hc_fno")
    cmd = [HOST_CXX, "-O2", "-std=c++14", "-Wall", "-fopenmp", "-o", fno, os.path.join(host, "hc_fno_main.cpp"), os.path.join(host, "hcb_fno.cpp"),
           os.path.join(host, "hcb_host.cpp"), "-L" + LIBDIR, "-lhc_b200", "-lpthread", "-Wl,-rpath,$ORIGIN"]
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    # hc_sfo2overlaps: scripts/sfo2overlaps.py of the reference in C++ (host only)
    conv = os.path.join(LIBDIR, "hc_sfo2overlaps")
    cmd = [HOST_CXX, "-O2", "-std=c++14", "-Wall", "-fopenmp", "-o", conv, os.path.join(host, "hcb_sfo2overlaps.cpp")]
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    # hc_sam2overlaps: scripts/sam2overlaps.py of the reference in C++ (host only)
    conv = os.path.join(LIBDIR, "hc_sam2overlaps")
    cmd = [HOST_CXX, "-O2", "-std=c++14", "-Wall", "-fopenmp", "-o", conv, os.path.join(host, "hcb_sam2overlaps.cpp")]
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return exe


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
