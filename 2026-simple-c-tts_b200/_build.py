"""In-tree builds of the native libraries (no JIT cache: the .so files travel with the repo).

libctts_front.so  plain C host front end (gcc)
libctts_b200.so   texts -> PCM: planner threads feeding a device session, plain C over the two libraries (gcc)
libctts_gpu.so    C-ABI + hand-written sm_100a kernels (nvcc, -fmad=false: the
                  reference is built without FMA contraction and discrete
                  decisions flip on 1-ulp differences, SURVEY.md 7.3)
ctts_b200         the `ctts synth` command line in plain C over the two libraries (gcc)
"""
from __future__ import annotations

import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
INCLUDE = os.path.join(ROOT, "include")
CSRC = os.path.join(PKG_DIR, "csrc")

FRONT_SO = os.path.join(PKG_DIR, "libctts_front.so")
GPU_SO = os.path.join(PKG_DIR, "libctts_gpu.so")
PIPE_SO = os.path.join(PKG_DIR, "libctts_b200.so")
CLI_BIN = os.path.join(PKG_DIR, "ctts_b200")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC", "-shared",
]


def _newer(target: str, sources: list[str]) -> bool:
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)


def _headers() -> list[str]:
    return [os.path.join(INCLUDE, h) for h in os.listdir(INCLUDE) if h.endswith(".h")]


def build_front(force: bool = False) -> str:
    src = os.path.join(CSRC, "front", "ctts_front.c")
    deps = [src] + _headers()
    if not force and _newer(FRONT_SO, deps):
        return FRONT_SO
    cc = shutil.which("gcc") or "cc"
    cmd = [cc, "-O2", "-std=c99", "-ffp-contract=off", "-Wall", "-Wextra", "-fPIC", "-shared",
           "-I", INCLUDE, "-o", FRONT_SO, src, "-lm"]
    subprocess.run(cmd, check=True)
    return FRONT_SO


def gpu_sources() -> list[str]:
    d = os.path.join(CSRC, "gpu")
    return sorted(os.path.join(d, f) for f in os.listdir(d) if f.endswith((".cu", ".c")))


def build_gpu(force: bool = False, verbose: bool = False) -> str:
    d = os.path.join(CSRC, "gpu")
    srcs = gpu_sources()
    deps = srcs + _headers() + [os.path.join(d, f) for f in os.listdir(d) if f.endswith((".cuh", ".h"))]
    if not force and _newer(GPU_SO, deps):
        return GPU_SO
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    cus = [s for s in srcs if s.endswith(".cu")]
    cs = [s for s in srcs if s.endswith(".c")]
    objs = []
    # the host tables use libm cosf/sinf with C promotion rules: compile them as C
    cc = shutil.which("gcc") or "cc"
    for s in cs:
        o = s[:-2] + ".o"
        subprocess.run([cc, "-O2", "-std=c99", "-ffp-contract=off", "-fPIC", "-I", INCLUDE, "-c", s, "-o", o],
                       check=True)
        objs.append(o)
    # CTTS_NVCC_EXTRA: extra nvcc flags for development builds (e.g. -DCTTS_ASM_PROF=1 for CTTS_GPU_TASK_TIMES)
    cmd = [nvcc] + NVCC_FLAGS + os.environ.get("CTTS_NVCC_EXTRA", "").split() + (["-Xptxas", "-v"] if verbose else []) + \
        ["-I", INCLUDE, "-I", d, "-o", GPU_SO] + cus + objs + ["-lcudart"]
    subprocess.run(cmd, check=True)
    return GPU_SO


def build_pipeline(force: bool = False) -> str:
    """libctts_b200.so: ctts_b200_synth_texts (csrc/cli/ctts_pipeline.c) over the two libraries."""
    src = os.path.join(CSRC, "cli", "ctts_pipeline.c")
    deps = [src, FRONT_SO, GPU_SO] + _headers()
    if not force and _newer(PIPE_SO, deps):
        return PIPE_SO
    cc = shutil.which("gcc") or "cc"
    cmd = [cc, "-O2", "-std=gnu99", "-Wall", "-Wextra", "-fPIC", "-shared", "-I", INCLUDE, "-o", PIPE_SO, src,
           "-L", PKG_DIR, "-lctts_front", "-lctts_gpu", "-Wl,-rpath,$ORIGIN", "-Wl,-rpath-link," + PKG_DIR,
           "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64", "-lpthread", "-lm"]
    subprocess.run(cmd, check=True)
    return PIPE_SO


def build_cli(force: bool = False) -> str:
    """The plain-C drop-in command line (csrc/cli/ctts_b200.c) linked against the three libraries."""
    src = os.path.join(CSRC, "cli", "ctts_b200.c")
    build_pipeline(force)
    deps = [src, os.path.join(CSRC, "cli", "g711_wav.h"), FRONT_SO, GPU_SO, PIPE_SO] + _headers()
    if not force and _newer(CLI_BIN, deps):
        return CLI_BIN
    cc = shutil.which("gcc") or "cc"
    cmd = [cc, "-O2", "-std=gnu99", "-Wall", "-Wextra", "-I", INCLUDE, "-o", CLI_BIN, src,
           "-L", PKG_DIR, "-lctts_b200", "-lctts_front", "-lctts_gpu", "-Wl,-rpath,$ORIGIN", "-Wl,-rpath-link," + PKG_DIR,
           "-L/usr/local/cuda/lib64", "-Wl,-rpath,/usr/local/cuda/lib64", "-lm"]
    subprocess.run(cmd, check=True)
    return CLI_BIN
