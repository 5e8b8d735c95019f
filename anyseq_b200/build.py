"""Build the sm_100a shared library (and the `align` CLI) in-tree with nvcc.

The built files live in anyseq_b200/_build/ (git-ignored, but shipped to the GPU
box by gpurun).  nvcc cross-compiles for sm_100a without a GPU.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
OUT = os.environ.get("ANYSEQ_BUILD_DIR") or os.path.join(_HERE, "_build")   # ANYSEQ_BUILD_DIR + ANYSEQ_NVCC_FLAGS: kernel-variant experiments (anyseq_b200/_build_*/ is git-ignored)
LIB = os.path.join(OUT, "libanyseq_b200.so")
CLI = os.path.join(OUT, "align")

LIB_SOURCES = ["engine.cu", "capi.cu", "microbench.cu", "inbox.cu", "traceback.cu", "traceback_full.cu", "batch.cu", "batch_x2.cu", "batch_stream.cu", "batch_packed2.cu", "batch_align.cu",
               "strip_inst_00.cu", "strip_inst_01.cu", "strip_inst_10.cu", "strip_inst_11.cu",
               "strip_inst_10t.cu", "strip_inst_11t.cu", "strip_inst_01p.cu"]
CLI_SOURCES = ["align_main.cpp", "sequence_io.cpp", "alignment_io.cpp"]
HEADERS = ["common.cuh", "engine.cuh", "strip_kernel.cuh", "strip_packed.cuh", "strip_inst.inl", "batch.cuh", "batch_kernel_body.inl", "traceback_full.cuh", "sequence_io.h", "alignment_io.h",
           os.path.join("..", "..", "include", "anyseq.h")]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"] + os.environ.get("ANYSEQ_NVCC_FLAGS", "").split()


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OUT, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS]
    lib_srcs = [os.path.join(CSRC, s) for s in LIB_SOURCES]
    if force or _stale(LIB, lib_srcs + hdrs):
        objs = []
        procs = []
        for src in lib_srcs:
            obj = os.path.join(OUT, os.path.basename(src) + ".o")
            objs.append(obj)
            if force or _stale(obj, [src] + hdrs):
                cmd = [_nvcc(), *NVCC_FLAGS, "-Xptxas", "-v", "-c", src, "-o", obj]
                procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        for cmd, p in procs:
            out, _ = p.communicate()
            if verbose or p.returncode != 0:
                sys.stderr.write(out)
            if p.returncode != 0:
                raise RuntimeError("nvcc failed: " + " ".join(cmd))
        cmd = [_nvcc(), "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a"]
        subprocess.run(cmd, check=True)
    cli_srcs = [os.path.join(CSRC, s) for s in CLI_SOURCES]
    if all(os.path.exists(s) for s in cli_srcs) and (force or _stale(CLI, cli_srcs + hdrs + [LIB])):
        cmd = ["/usr/bin/g++", "-O2", "-std=c++17", "-I", os.path.join(_HERE, "..", "include"),
               *cli_srcs, "-o", CLI, "-L", OUT, "-lanyseq_b200", "-Wl,-rpath,$ORIGIN"]
        subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
