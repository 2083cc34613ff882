"""In-tree build of libddrl_b200.so (hand-written sm_100a CUDA behind the C ABI in include/ddrl_b200.h).

nvcc cross-compiles without a GPU; the built .so is git-ignored but travels to the GPU box with the
gpurun snapshot.  ``python -m ddrl_b200.build`` or ``__graft_entry__.build()``."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libddrl_b200.so")
SOURCES = ["stream.cu", "filter_stream.cu", "fcnet.cu", "graphnet.cu", "graphnet_tc.cu", "graphvar.cu", "tc.cu", "tc2.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--use_fast_math=false"]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found: libddrl_b200.so cannot be built (there is no CPU fallback)")


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(PKG, "..", "include", "ddrl_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    nvcc = _nvcc()
    objs = []
    build_dir = os.path.join(PKG, "csrc", "_build")
    os.makedirs(build_dir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(build_dir, src.replace(".cu", ".o"))
        objs.append(obj)
        flags = [f for f in NVCC_FLAGS if not f.startswith("--use_fast_math")]
        cmd = [nvcc, *flags, "-Xptxas", "-v", "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}")
        with open(os.path.join(build_dir, src + ".ptxas.log"), "w") as f:
            f.write(out)
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs]
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose=True))
