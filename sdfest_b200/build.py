"""Build libsdfrender.so (the sm_100a CUDA library behind the C ABI in include/sdfrender.h).

Plain nvcc, no torch headers: the library is torch-free by design, so a rebuild takes seconds
and the binary is usable from any host language over the C ABI.

    python -m sdfest_b200.build [--force] [--verbose]
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libsdfrender.so")
SOURCES = [os.path.join(CSRC, "sdfrender.cu")]
HEADERS = [
    os.path.join(CSRC, "sdfr_core.cuh"),
    os.path.join(CSRC, "sdfr_points.cuh"),
    os.path.join(CSRC, "sdfr_decoder.cuh"),
    os.path.join(CSRC, "sdfr_step.cuh"),
    os.path.join(os.path.dirname(PKG_DIR), "include", "sdfrender.h"),
]
NVCC_FLAGS = [
    "-O3",
    "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-Xcompiler", "-fPIC",
]
N_PARTS = 4  # sdfrender.cu compiles as four translation units (-DSDFR_PART=1..4) in parallel
OBJ_DIR = os.path.join(os.path.dirname(PKG_DIR), "build")


def find_nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def up_to_date() -> bool:
    if not os.path.isfile(LIB_PATH):
        return False
    t = os.path.getmtime(LIB_PATH)
    return all(os.path.getmtime(f) <= t for f in SOURCES + HEADERS)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and up_to_date():
        return LIB_PATH
    nvcc = find_nvcc()
    os.makedirs(OBJ_DIR, exist_ok=True)
    objs, procs = [], []
    for part in range(1, N_PARTS + 1):
        obj = os.path.join(OBJ_DIR, f"sdfrender_part{part}.o")
        cmd = [nvcc, *NVCC_FLAGS, f"-DSDFR_PART={part}", "-c", *SOURCES, "-o", obj]
        if verbose:
            cmd[1:1] = ["-Xptxas", "-v"]
            print(" ".join(cmd))
        log = open(obj + ".log", "w")
        procs.append((subprocess.Popen(cmd, stdout=log, stderr=subprocess.STDOUT), cmd, log))
        objs.append(obj)
    failed = None
    for proc, cmd, log in procs:
        rc = proc.wait()
        log.close()
        text = open(log.name).read()
        if verbose or rc != 0:
            sys.stdout.write(text)
        if rc != 0 and failed is None:
            failed = subprocess.CalledProcessError(rc, cmd)
    if failed is not None:
        raise failed
    subprocess.check_call([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", *objs, "-o", LIB_PATH])
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
