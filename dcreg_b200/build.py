"""Build the sm_100a shared library in-tree with nvcc (no JIT cache: the .so travels with the repo)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libdcreg_b200.so")
SOURCES = ["dcreg_b200.cu"]
HEADERS = ["corr.cuh", "k1_reduce.cuh", "k1_stream.cuh", "k2_solve.cuh", "k2_fast.cuh", "peer_reduce.cuh", "loop_plan.hpp", "p2p_bound.hpp", "small_la.cuh",
           "../../include/dcreg_b200.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--shared", "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
    "--fmad=true",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def is_stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    for f in SOURCES + HEADERS:
        if os.path.getmtime(os.path.join(CSRC, f)) > t:
            return True
    return False


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB_PATH
    cmd = [_nvcc()] + NVCC_FLAGS + [os.path.join(CSRC, s) for s in SOURCES] + ["-o", LIB_PATH, "-ldl"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    log = res.stdout + res.stderr
    with open(os.path.join(PKG_DIR, "build.log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + log)
    if res.returncode != 0:
        sys.stderr.write(log)
        raise RuntimeError("nvcc failed (see dcreg_b200/build.log)")
    if verbose:
        print(log)
    return LIB_PATH


HOST_DIR = os.path.join(PKG_DIR, "host")
RUNNER_PATH = os.path.join(PKG_DIR, "icp_test_runner")
RUNNER_SOURCES = ["icp_test_runner.cpp"]
RUNNER_HEADERS = ["yaml_lite.hpp", "pcd_io.hpp", "../../include/dcreg_b200.h"]


def build_runner(force: bool = False) -> str:
    """g++ build of the host CLI (the reference's `icp_test_runner` executable) against the C ABI library."""
    build(force=False)
    deps = [os.path.join(HOST_DIR, f) for f in RUNNER_SOURCES + RUNNER_HEADERS] + [LIB_PATH]
    if not force and os.path.exists(RUNNER_PATH) and all(os.path.getmtime(d) <= os.path.getmtime(RUNNER_PATH) for d in deps):
        return RUNNER_PATH
    cxx = os.environ.get("CXX") or shutil.which("g++") or "g++"
    cmd = [cxx, "-O2", "-std=c++17", "-Wall", "-Wextra"] + [os.path.join(HOST_DIR, s) for s in RUNNER_SOURCES] + [
        "-o", RUNNER_PATH, "-L" + PKG_DIR, "-ldcreg_b200", "-Wl,-rpath,$ORIGIN"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("g++ failed building icp_test_runner")
    return RUNNER_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
    print(build_runner(force="--force" in sys.argv))
