"""Build libldagpu.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo).

    python -m ldagroupedgibbssampler_b200.build [--force] [--verbose]

There is one build: the kernel configuration (warps, occupancy, register tiles, unrolling) is fixed
in the sources at its measured values.

Flags that matter:
  -gencode arch=compute_100a,code=sm_100a   B200 only, no fallback architectures
  -fmad=false                               the contract arithmetic must not be contracted into
                                            FMAs behind our back (explicit fma calls are kept)
  -lineinfo                                 ncu source pages map back to the .cu files
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "_obj")
OUT = os.path.join(HERE, "libldagpu.so")

CU = ["kernels_z.cu", "kernels_z_big.cu", "kernels_sparse.cu", "kernels_phi.cu", "kernels_p2p.cu", "kernels_misc.cu", "kernels_heldout.cu",
      "engine.cu"]
CPP = []
SYNTH_SRC, SYNTH_OUT = os.path.join(CSRC, "synth.cpp"), os.path.join(HERE, "libldasynth.so")
HEADERS = ["common.cuh", "contract_math.cuh", "warp_draw.cuh", os.path.join("..", "..", "include", "ldagpu.h")]

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
NVFLAGS = ["-O3", "-std=c++17", "-lineinfo", "-fmad=false", "-Xcompiler", "-fPIC,-O2,-pthread",
           "-ccbin", "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"]


def _newer(src: str, dst: str) -> bool:
    return (not os.path.exists(dst)) or os.path.getmtime(src) > os.path.getmtime(dst)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    hdr_paths = [os.path.normpath(os.path.join(CSRC, h)) for h in HEADERS]
    objs = []
    procs = []
    for src in CU + CPP:
        sp = os.path.join(CSRC, src)
        op = os.path.join(OBJ, src + ".o")
        objs.append(op)
        stale = force or _newer(sp, op) or any(_newer(h, op) for h in hdr_paths)
        if not stale:
            continue
        cmd = [NVCC] + ARCH + NVFLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", sp, "-o", op]
        if verbose:
            print(" ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        text, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- {src}\n{text}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    if force or procs or not os.path.exists(OUT):
        cmd = [NVCC] + ARCH + ["-shared", "-o", OUT] + objs + ["-Xcompiler", "-pthread", "-ldl"]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)
    build_synth(force)
    return OUT


def build_synth(force: bool = False) -> str:
    """libldasynth.so: the synthetic-corpus generator, host C++ only (no CUDA), its own library."""
    hdr = os.path.normpath(os.path.join(CSRC, "..", "..", "include", "ldasynth.h"))
    if force or _newer(SYNTH_SRC, SYNTH_OUT) or _newer(hdr, SYNTH_OUT):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-pthread", SYNTH_SRC, "-o", SYNTH_OUT])
    return SYNTH_OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
