"""In-tree builds: the CUDA C-ABI library (nvcc, sm_100a), the CPU oracle and the host-emulation
harness used by the CPU-only logic tests.  Artefacts stay next to the sources so that they travel
with a gpurun snapshot."""
from __future__ import annotations

import os
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
CSRC = os.path.join(_HERE, "csrc")
LIB = os.path.join(_HERE, "libimmesh_b200.so")
EMU = os.path.join(_ROOT, "tests", "emu", "libimmesh_emu.so")
ORACLE = os.path.join(_ROOT, "oracle", "liborc.so")
GXX = "/usr/bin/g++"

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false",            # numerics contract: no FMA contraction (bit parity with the reference's SSE2 build)
    "-Xcompiler", "-fPIC", "-shared",
]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _sources(dirpath, exts):
    return sorted(os.path.join(dirpath, f) for f in os.listdir(dirpath) if f.endswith(exts))


def build_cuda(force=False, verbose=False):
    cu = _sources(CSRC, (".cu",))
    deps = cu + _sources(CSRC, (".cuh", ".hpp")) + [os.path.join(_ROOT, "include", "immesh_b200.h")]
    if force or _newer(LIB, deps):
        cmd = ["nvcc", *NVCC_FLAGS, "-ccbin", GXX, "-o", LIB, *cu]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        subprocess.check_call(cmd, cwd=_ROOT)
    return LIB


def build_oracle(force=False):
    src = _sources(os.path.join(_ROOT, "oracle"), (".cpp", ".hpp"))
    if force or _newer(ORACLE, src):
        subprocess.check_call(["make", "-C", os.path.join(_ROOT, "oracle"), "-B"])
    return ORACLE


def build_emu(force=False):
    emu_dir = os.path.join(_ROOT, "tests", "emu")
    src = _sources(emu_dir, (".cpp",))
    deps = src + _sources(CSRC, (".cuh", ".hpp"))
    if force or _newer(EMU, deps):
        cmd = [GXX, "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-Wno-unknown-pragmas", "-I/usr/local/cuda/include", "-shared", "-o", EMU]
        for s in src:
            cmd += ["-x", "c++", s]
        subprocess.check_call(cmd)
    return EMU


def build_all(force=False):
    build_cuda(force)
    build_oracle(force)
    build_emu(force)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv)
    print("built:", LIB, ORACLE, EMU)
