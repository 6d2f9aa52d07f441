"""In-tree build of libaprilsam_b200.so (host C + sm_100a CUDA) and the test/bench harness.

    python -m aprilsam_b200.build            # build what is out of date
    python -m aprilsam_b200.build --force

Outputs (git-ignored, but shipped to the GPU box by gpurun):
    aprilsam_b200/lib/libaprilsam_b200.so    the drop-in library (april_graph_* + asam_* C-ABI)
    harness/_build/harness_b200.so           harness/harness.c linked against it
    oracle/_ref/*                            the reference oracle (only where /root/reference exists)
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "aprilsam_b200")
LIB_DIR = os.path.join(PKG, "lib")
OBJ_DIR = os.path.join(PKG, "lib", "obj")
LIB = os.path.join(LIB_DIR, "libaprilsam_b200.so")
HARNESS = os.path.join(ROOT, "harness", "_build", "harness_b200.so")
REPLAY_CLI = os.path.join(ROOT, "examples", "_build", "asam_replay")

NVCC = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
CC = os.environ.get("CC", "gcc")

CUDA_SRCS = [os.path.join(PKG, "csrc", "asam_cuda.cu")]
HOST_SRCS = [os.path.join(PKG, "host", f) for f in ("graph.c", "ordering.c", "plan.c", "solver.c", "serial.c", "cliopt.c", "debug.c")]
INCLUDES = ["-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "include", "aprilsam"),
            "-I" + os.path.join(PKG, "host")]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC,-fvisibility=hidden", "-Xptxas", "-v"]
CC_FLAGS = ["-std=gnu11", "-O2", "-g", "-fPIC", "-fvisibility=hidden", "-fopenmp", "-Wall", "-Wextra",
            "-Wno-unused-parameter"]


def _run(cmd: list[str], log: list[str]) -> None:
    p = subprocess.run(cmd, capture_output=True, text=True)
    log.append("$ " + " ".join(cmd) + "\n" + p.stdout + p.stderr)
    if p.returncode != 0:
        sys.stderr.write(log[-1])
        raise RuntimeError(f"build step failed: {' '.join(cmd[:3])} ...")


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def _headers() -> list[str]:
    out = []
    for base in (os.path.join(ROOT, "include"), os.path.join(PKG, "host"), os.path.join(PKG, "csrc")):
        for dp, _, fs in os.walk(base):
            out += [os.path.join(dp, f) for f in fs if f.endswith((".h", ".cuh"))]
    return out


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile everything that is out of date; returns the path of the library."""
    os.makedirs(OBJ_DIR, exist_ok=True)
    os.makedirs(os.path.dirname(HARNESS), exist_ok=True)
    log: list[str] = []
    hdrs = _headers()
    objs = []
    for src in CUDA_SRCS:
        obj = os.path.join(OBJ_DIR, os.path.basename(src) + ".o")
        objs.append(obj)
        if force or _stale(obj, [src] + hdrs):
            _run([NVCC] + NVCC_FLAGS + INCLUDES + ["-c", src, "-o", obj], log)
    for src in HOST_SRCS:
        obj = os.path.join(OBJ_DIR, os.path.basename(src) + ".o")
        objs.append(obj)
        if force or _stale(obj, [src] + hdrs):
            _run([CC] + CC_FLAGS + INCLUDES + ["-c", src, "-o", obj], log)
    if force or _stale(LIB, objs):
        _run([NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs +
             ["-Xlinker", "-Bsymbolic", "-Xcompiler", "-fopenmp", "-lm"], log)
    hsrc = os.path.join(ROOT, "harness", "harness.c")
    if force or _stale(HARNESS, [hsrc, LIB] + hdrs):
        _run([CC, "-std=gnu99", "-O2", "-g", "-fPIC", "-shared", "-I" + os.path.join(ROOT, "include", "aprilsam"),
              "-o", HARNESS, hsrc, "-L" + LIB_DIR, "-laprilsam_b200", "-Wl,-rpath," + LIB_DIR,
              "-Wl,-rpath,$ORIGIN/../../aprilsam_b200/lib", "-lm"], log)
    csrc = os.path.join(ROOT, "examples", "asam_replay.c")
    os.makedirs(os.path.dirname(REPLAY_CLI), exist_ok=True)
    if force or _stale(REPLAY_CLI, [csrc, LIB] + hdrs):
        _run([CC, "-std=gnu99", "-O2", "-g", "-I" + os.path.join(ROOT, "include", "aprilsam"), "-o", REPLAY_CLI, csrc,
              "-L" + LIB_DIR, "-laprilsam_b200", "-Wl,-rpath," + LIB_DIR, "-Wl,-rpath,$ORIGIN/../../aprilsam_b200/lib",
              "-lm"], log)
    # the oracle: C restatement always; the real reference and its example programs (linked against this
    # library) only where the reference sources exist
    _run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "all"], log)
    with open(os.path.join(LIB_DIR, "build.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(LIB)
