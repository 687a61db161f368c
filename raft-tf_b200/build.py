"""Build libraft_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = ["capi.cu", "corr.cu", "conv_simt.cu", "conv_tc.cu", "conv_api.cu", "gemm_tc.cu", "update.cu", "upsample.cu",
           "encoder.cu", "frames.cu", "consistency.cu"]
LIB = os.path.join(HERE, "lib", "libraft_b200.so")


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(HERE, "csrc", f) for f in os.listdir(os.path.join(HERE, "csrc"))]
    deps.append(os.path.join(HERE, "..", "include", "raft_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objdir = os.path.join(HERE, "lib", "obj")
    os.makedirs(objdir, exist_ok=True)
    flags = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC"]
    if verbose:
        flags += ["-Xptxas", "-v"]
    # one nvcc per translation unit, in parallel (the tcgen05 kernels dominate the build time); objects are rebuilt
    # when the source or any header is newer
    hdrs = [os.path.join(HERE, "csrc", f) for f in os.listdir(os.path.join(HERE, "csrc")) if f.endswith(".cuh")]
    hdrs.append(os.path.join(HERE, "..", "include", "raft_b200.h"))
    hdr_t = max(os.path.getmtime(h) for h in hdrs)
    procs, objs = [], []
    for s in SOURCES:
        src = os.path.join(HERE, "csrc", s)
        obj = os.path.join(objdir, s[:-3] + ".o")
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_t):
            procs.append((s, subprocess.Popen([nvcc] + flags + ["-c", src, "-o", obj])))
    failed = [s for s, p in procs if p.wait() != 0]
    if failed:
        raise RuntimeError(f"nvcc failed for {failed}")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-cudart", "static", "-o", LIB] + objs, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
