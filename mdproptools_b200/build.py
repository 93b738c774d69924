"""In-tree build of libmdprop_b200.so (sm_100a only).

``python -m mdproptools_b200.build`` or ``mdproptools_b200.build.build()``.  nvcc cross-compiles without a
GPU, so this also runs in the GPU-less build container; the resulting .so is git-ignored but travels to the
GPU box with the repo snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmdprop_b200.so")

CU_SOURCES = ["ctx.cu", "pair.cu", "reduce.cu", "corr.cu", "dump_device.cu", "survival.cu", "shell.cu", "fftcorr.cu", "msdfft.cu", "sk.cu", "isffft.cu", "orient.cu", "epilogue.cu"]
CPP_SOURCES = ["dump_parse.cpp"]
HEADERS = ["common.cuh", "pair_fast.cuh", "dump_line.h", "dump_rows.h", "survival_runs.h", "shell_grid.h", "fft_corr.h", "fft_pass.cuh", "msd_fft.h", "isf_fft.h", "orient.h", "sk_phase.h", "scratch_plan.h",
           os.path.join("..", "..", "include", "mdprop_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "--fmad=false",            # parity-critical arithmetic is unfused; FMAs are written explicitly where wanted
    "-Xcompiler", "-fPIC,-O2,-fno-fast-math,-pthread",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libmdprop_b200 cannot be built (there is no CPU fallback)")


def _host_cxx() -> str:
    # the /opt/gcc wrapper exported as $CXX in this image lacks some specs; prefer the system compiler
    for cand in ("/usr/bin/g++", shutil.which("g++")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("g++ not found")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    srcs = [os.path.join(CSRC, s) for s in CU_SOURCES + CPP_SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(s) > t for s in srcs)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    nvcc, cxx = _nvcc(), _host_cxx()
    extra = os.environ.get("MDP_NVCC_EXTRA", "").split()          # e.g. -DMDP_FAST_UNROLL=8 for A/B builds
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for s in CU_SOURCES:
        o = os.path.join(objdir, s + ".o")
        cmd = [nvcc, "-ccbin", cxx] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, s), "-o", o]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    for s in CPP_SOURCES:
        o = os.path.join(objdir, s + ".o")
        cmd = [cxx, "-O2", "-std=c++17", "-fPIC", "-fno-fast-math", "-pthread", "-c", os.path.join(CSRC, s), "-o", o]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            sys.stderr.write(f"--- {s} ---\n{out}\n")
        elif verbose and out.strip():
            print(f"--- {s} ---\n{out}")
    if failed:
        raise RuntimeError("compilation of libmdprop_b200 failed")
    tmp = LIB + ".tmp"
    cmd = [nvcc, "-ccbin", cxx, "-shared", "-o", tmp] + objs + ["-Xcompiler", "-pthread", "-lcudart_static", "-lpthread", "-ldl", "-lrt"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link of libmdprop_b200.so failed")
    os.replace(tmp, LIB)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
