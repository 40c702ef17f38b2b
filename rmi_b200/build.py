"""Builds librmi_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
# RMI_BUILD_TAG=<name> (with RMI_NVCC_DEFS="-DFOO ...") builds an experiment variant next to the
# default library: lib/librmi_b200_<name>.so, loaded by dev tools through RMI_B200_LIB.
_TAG = os.environ.get("RMI_BUILD_TAG", "")
LIB_PATH = os.path.join(LIB_DIR, f"librmi_b200{'_' + _TAG if _TAG else ''}.so")
OBJ_DIR = os.path.join(HERE, "build" + ("_" + _TAG if _TAG else ""))

SOURCES = ["kernels_top.cu", "kernels_leaf.cu", "kernels_shard.cu", "kernels_lookup.cu", "api.cu"]
HEADERS = ["rust_math.cuh", "models.cuh", "device_util.cuh", "spline.cuh", "kernels.h",
           os.path.join("..", "..", "include", "rmi_b200.h"), os.path.join("..", "..", "host", "cache_fix.hpp"), os.path.join("..", "..", "host", "codegen.hpp"),
           os.path.join("..", "..", "host", "optimizer.hpp")]

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
# -fmad=false: the reference fuses a multiply-add only where it writes mul_add; everything
# else must round twice (see csrc/rust_math.cuh).
EXTRA_DEFS = os.environ.get("RMI_NVCC_DEFS", "").split()
NVCC_FLAGS = EXTRA_DEFS + ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-fmad=false",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O2"]


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build_library(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIB_DIR, exist_ok=True)
    os.makedirs(OBJ_DIR, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]
    objs, jobs = [], []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            jobs.append([NVCC] + NVCC_FLAGS + ["-c", s, "-o", o])

    def run(cmd):
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed:\n{' '.join(cmd)}\n{r.stdout}\n{r.stderr}")
        return r

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        list(ex.map(run, jobs))
    if force or jobs or _stale(LIB_PATH, objs):
        run([NVCC, "-shared", "-o", LIB_PATH] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"])
    return LIB_PATH


CLI_PATH = os.path.join(HERE, "bin", "rmi")


def build_cli(force: bool = False) -> str:
    """The `rmi` command-line front end (host/rmi_main.cpp) linked against librmi_b200.so."""
    lib = build_library()
    root = os.path.dirname(HERE)
    srcs = [os.path.join(root, "host", f) for f in ("rmi_main.cpp", "codegen.hpp", "optimizer.hpp", "cache_fix.hpp", "param_grid.hpp")]
    os.makedirs(os.path.dirname(CLI_PATH), exist_ok=True)
    if force or _stale(CLI_PATH, srcs + [lib, os.path.join(root, "include", "rmi_b200.h")]):
        cmd = ["g++", "-std=c++17", "-O2", "-Wall", srcs[0], "-o", CLI_PATH, "-L", LIB_DIR, "-lrmi_b200",
               "-Wl,-rpath,$ORIGIN/../lib"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"g++ failed:\n{' '.join(cmd)}\n{r.stdout}\n{r.stderr}")
    return CLI_PATH


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose=True))
    print(build_cli(force="--force" in sys.argv))
