"""Build recipe: nvcc (sm_100a) for the CUDA TU, gcc for the host C, one
shared library ``utree_b200/csrc/libutree_b200.so`` plus the CLI in ``bin/``.
Everything is built in-tree so it travels to the GPU box with the snapshot."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libutree_b200.so")
SYNTH_LIB = os.path.join(ROOT, "tools", "libutb_synth.so")   # bench/test input generator, not the product
BIN = os.path.join(ROOT, "bin")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
GCC = "gcc"   # PATH gcc: $CC in this image points at a gcc without libgomp specs

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]
C_FLAGS = ["-std=gnu11", "-O2", "-g", "-Wall", "-Wextra", "-Wno-unused-parameter", "-fPIC", "-pthread"]
C_SOURCES = ["ctr_loader.c", "pipeline.c", "compress.c"]


def _run(cmd, log=None):
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if log is not None:
        log.append(p.stdout)
    if p.returncode:
        sys.stderr.write(p.stdout)
        raise RuntimeError("build step failed: " + " ".join(cmd))
    return p.stdout


def _newer(target, sources):
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)


def build(force=False, verbose=False):
    srcs = [os.path.join(CSRC, f) for f in C_SOURCES + ["kernels.cu", "builder.cu", "utb_internal.h", "main.c", "main_shallow.c", "main_profile.c", "compress_main.c", "build_main.c"]]
    srcs.append(os.path.join(ROOT, "include", "utree_b200.h"))
    exe = os.path.join(BIN, "utree-search_gg")
    if not force and _newer(LIB, srcs) and _newer(exe, srcs):
        return LIB
    log = []
    objs = []
    o = os.path.join(CSRC, "kernels.o")
    extra = os.environ.get("UTB_NVCC_EXTRA", "").split()        # tuning builds, e.g. "-DFILT_ILP=4 -DFILT_MINB=3"
    _run([NVCC] + NVCC_FLAGS + extra + ["-c", os.path.join(CSRC, "kernels.cu"), "-o", o], log)
    objs.append(o)
    o = os.path.join(CSRC, "builder.o")                         # GPU utree-build_gg (CUB sort / scan / select)
    _run([NVCC] + NVCC_FLAGS + ["-c", os.path.join(CSRC, "builder.cu"), "-o", o], log)
    objs.append(o)
    for f in C_SOURCES:
        o = os.path.join(CSRC, f[:-2] + ".o")
        _run([GCC] + C_FLAGS + ["-c", os.path.join(CSRC, f), "-o", o], log)
        objs.append(o)
    _run([NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs +
         ["-Xcompiler", "-pthread", "-lpthread"], log)
    os.makedirs(BIN, exist_ok=True)
    _run([GCC] + C_FLAGS + [os.path.join(CSRC, "main.c"), "-o", exe, "-L" + CSRC, "-lutree_b200",
                            "-Wl,-rpath,$ORIGIN/../utree_b200/csrc"], log)
    shutil.copyfile(exe, os.path.join(BIN, "utree-searchGG"))
    os.chmod(os.path.join(BIN, "utree-searchGG"), 0o755)
    _run([GCC] + C_FLAGS + [os.path.join(CSRC, "main_shallow.c"), "-o", os.path.join(BIN, "utree-search"), "-L" + CSRC, "-lutree_b200",
                            "-Wl,-rpath,$ORIGIN/../utree_b200/csrc"], log)
    _run([GCC] + C_FLAGS + [os.path.join(CSRC, "main_profile.c"), "-o", os.path.join(BIN, "utree-profile"), "-L" + CSRC, "-lutree_b200",
                            "-Wl,-rpath,$ORIGIN/../utree_b200/csrc"], log)
    _run([GCC] + C_FLAGS + [os.path.join(CSRC, "build_main.c"), "-o", os.path.join(BIN, "utree-build_gg"), "-L" + CSRC, "-lutree_b200",
                            "-Wl,-rpath,$ORIGIN/../utree_b200/csrc"], log)
    _run([GCC] + C_FLAGS + [os.path.join(CSRC, "compress_main.c"), "-o", os.path.join(BIN, "utree-compress"), "-L" + CSRC,
                            "-lutree_b200", "-Wl,-rpath,$ORIGIN/../utree_b200/csrc"], log)
    with open(os.path.join(CSRC, "build.log"), "w") as f:
        f.write("".join(log))
    if verbose:
        print("".join(log))
    return LIB


def build_synth(force=False):
    """libutb_synth.so: synthetic CTR / reads generator (CUB sort).  Inputs only."""
    src = os.path.join(ROOT, "tools", "synth.cu")
    if not force and _newer(SYNTH_LIB, [src]):
        return SYNTH_LIB
    _run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
          "-Xcompiler", "-fPIC", "-shared", src, "-o", SYNTH_LIB])
    return SYNTH_LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
    build_synth(force="--force" in sys.argv)
