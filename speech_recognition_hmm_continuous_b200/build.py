"""Builds the native code IN-TREE for sm_100a (nvcc cross-compiles without a GPU):

  libhmmcu.so                     CUDA kernels + C ABI (include/hmm_cuda.h) + the C host side
  bin/hmm_continuous_fs           drop-in trainer      (reference program name)
  bin/recognition_continuous_fs   drop-in recogniser   (reference program name)

python -m speech_recognition_hmm_continuous_b200.build [--force] [--verbose]
"""
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
INC = os.path.join(ROOT, "include")
LIB = os.path.join(PKG, "libhmmcu.so")
BIN = os.path.join(PKG, "bin")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-I", INC, "-I", CSRC]
HOST_C = ["hmm_host.c", "train_viterbi.c", "train_mmi.c", "ingest.c", "modelset.c", "train_main.c", "test_main.c"]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _run(cmd, verbose):
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)


def build(force=False, verbose=False):
    cu = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith(".cu")]
    hdr = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")] + [os.path.join(INC, "hmm_cuda.h")]
    csrc = [os.path.join(CSRC, "host", f) for f in HOST_C]
    objdir = os.path.join(PKG, "build")
    os.makedirs(objdir, exist_ok=True)
    os.makedirs(BIN, exist_ok=True)
    if force or _newer(LIB, cu + hdr + csrc):
        objs = []
        for c in csrc:
            o = os.path.join(objdir, os.path.basename(c)[:-2] + ".o")
            _run(["gcc", "-O2", "-fPIC", "-Wall", "-Wno-unused-result", "-I", INC, "-c", c, "-o", o], verbose)
            objs.append(o)
        _run(["nvcc"] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-shared", "-o", LIB] + cu + objs, verbose)
    for exe, src in (("hmm_continuous_fs", "cli_train.c"), ("recognition_continuous_fs", "cli_test.c")):
        out = os.path.join(BIN, exe)
        s = os.path.join(CSRC, "host", src)
        if force or _newer(out, [s, LIB]):
            _run(["gcc", "-O2", "-I", INC, s, "-o", out, "-L", PKG, "-lhmmcu", "-Wl,-rpath,$ORIGIN/..", "-lm"], verbose)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print("built", LIB)
