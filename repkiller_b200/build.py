"""Builds librk_b200.so (the C-ABI library with the sm_100a kernels) and the host binaries in-tree.

nvcc cross-compiles for sm_100a without a GPU; the built files are git-ignored but travel to the GPU box.
"""
from __future__ import annotations

import glob
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "librk_b200%s.so" % os.environ.get("RK_LIB_SUFFIX", ""))
CLI = os.path.join(HERE, "bin", "repkiller")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVCC_FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC,-O3,-Wall", "-Xptxas", "-v"] + os.environ.get("RK_EXTRA_NVCC", "").split()


def _newer(target: str, sources: list[str]) -> bool:
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)


def build_lib(force: bool = False, verbose: bool = False) -> str:
    cu = sorted(glob.glob(os.path.join(CSRC, "*.cu")))
    deps = cu + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(HERE, "..", "include", "*.h"))
    if not force and _newer(LIB, deps):
        return LIB
    objs = []
    BUILD = os.path.join(HERE, "build" + os.environ.get("RK_LIB_SUFFIX", ""))
    os.makedirs(BUILD, exist_ok=True)
    procs = []
    for src in cu:
        obj = os.path.join(BUILD, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        cmd = [NVCC, *ARCH, *NVCC_FLAGS, "-c", src, "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append(out)
        if p.returncode != 0:
            sys.stderr.write(out)
            raise RuntimeError(f"nvcc failed on {src}")
    with open(os.path.join(BUILD, "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    subprocess.check_call([NVCC, *ARCH, "-shared", "-o", LIB, *objs])
    return LIB


def build_host(force: bool = False) -> str | None:
    """Host C++ over the C ABI: the drop-in `repkiller` CLI and the rk_hostcheck test helper."""
    common = sorted(glob.glob(os.path.join(CSRC, "host", "*.cpp")))
    mains = sorted(glob.glob(os.path.join(CSRC, "host", "main", "*.cpp")))
    if not mains:
        return None
    deps = common + mains + glob.glob(os.path.join(CSRC, "host", "*.h")) + [os.path.join(CSRC, "rk_csv_row.cuh"), LIB]  # (the row rules)
    os.makedirs(os.path.dirname(CLI), exist_ok=True)
    for m in mains:
        exe = os.path.join(os.path.dirname(CLI), os.path.basename(m)[:-4])
        if not force and _newer(exe, deps):
            continue
        cmd = ["g++", "-std=c++17", "-O2", "-Wall", "-I", os.path.join(HERE, "..", "include"), *common, m, "-o", exe,
               "-L", HERE, "-lrk_b200", "-Wl,-rpath,$ORIGIN/..", "-lpthread"]
        subprocess.check_call(cmd)
    return CLI


if __name__ == "__main__":
    build_lib(force="--force" in sys.argv, verbose="-v" in sys.argv)
    build_host(force="--force" in sys.argv)
    print(LIB)
