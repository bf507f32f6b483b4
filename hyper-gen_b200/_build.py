"""In-tree build of libhypergen_b200.so (hand-written CUDA for sm_100a + the C ABI).

nvcc cross-compiles without a GPU.  The shared library is written next to this file so it
travels with the repository snapshot; nothing is installed into site-packages.
"""
from __future__ import annotations

import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(ROOT, "build", "obj")
LIB = os.path.join(HERE, "libhypergen_b200.so")

SOURCES = ["api.cu", "kmer_hash.cu", "encode.cu", "dist_simt.cu", "dist_tc.cu", "dist_narrow.cu", "probe.cu", "fasta.cu", "sort.cu", "peer.cu",
           "search.cu", "cluster.cu", "derep.cu", "matrix.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-fvisibility=hidden", "-diag-suppress", "177",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _deps_mtime() -> float:
    m = 0.0
    for d in (CSRC, os.path.join(ROOT, "include")):
        for f in os.listdir(d):
            if f.endswith((".cuh", ".h")):
                m = max(m, os.path.getmtime(os.path.join(d, f)))
    return m


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    lib_m = os.path.getmtime(LIB)
    if _deps_mtime() > lib_m:
        return True
    return any(os.path.getmtime(os.path.join(CSRC, s)) > lib_m for s in SOURCES)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu for sm_100a and link the shared library. Returns its path."""
    have_src = os.path.isdir(CSRC) and all(os.path.exists(os.path.join(CSRC, s)) for s in SOURCES)
    if not force and not needs_build():
        return LIB
    if not have_src:
        raise RuntimeError("CUDA sources missing under %s" % CSRC)
    nvcc = _nvcc()
    os.makedirs(OBJ, exist_ok=True)
    hdr_m = _deps_mtime()

    def compile_one(src: str) -> str:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src.replace(".cu", ".o"))
        if (not force and os.path.exists(o) and os.path.getmtime(o) > os.path.getmtime(s)
                and os.path.getmtime(o) > hdr_m):
            return o
        cmd = [nvcc, *NVCC_FLAGS, "-c", s, "-o", o]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        return o

    with cf.ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-o", LIB, *objs, "-cudart", "static"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    return LIB


HOST_SRC = os.path.join(HERE, "host", "hyper_gen.cpp")
HOST_BIN = os.path.join(HERE, "bin", "hyper-gen")


def build_host(force: bool = False) -> str:
    """The C++ host (hyper-gen sketch / dist CLI) on top of the C ABI."""
    build(force=False)
    if (not force and os.path.exists(HOST_BIN) and os.path.getmtime(HOST_BIN) > os.path.getmtime(HOST_SRC)
            and os.path.getmtime(HOST_BIN) > os.path.getmtime(LIB)):
        return HOST_BIN
    os.makedirs(os.path.dirname(HOST_BIN), exist_ok=True)
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    cmd = [cxx, "-O2", "-std=c++17", "-pthread", HOST_SRC, "-o", HOST_BIN, "-L" + HERE, "-lhypergen_b200",
           "-Wl,-rpath,$ORIGIN/.."]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("host build failed:\n%s\n%s" % (r.stdout, r.stderr))
    return HOST_BIN


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
    print(build_host(force="--force" in sys.argv))
