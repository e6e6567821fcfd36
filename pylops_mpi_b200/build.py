"""Build libb200lops.so in-tree with nvcc for sm_100a (no torch involvement).

    python -m pylops_mpi_b200.build [--force]

The shared library is written next to this file so that it travels with the
repo snapshot to the GPU box (it is git-ignored, not gpurun-ignored).
"""
from __future__ import annotations

import os
import subprocess
import sys
import sysconfig

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libb200lops.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

SOURCES = ["ctx.cu", "elementwise.cu", "reduce.cu", "sparsity.cu", "stencil.cu", "convolve.cu", "gemv.cu", "gemm_simt.cu",
           "gemm_tc.cu", "gemm_tc2.cu", "fredholm_tc.cu", "host_pipe.cu", "comm.cu", "peer.cu"]


def _nccl_paths():
    site = sysconfig.get_paths()["purelib"]
    inc = os.path.join(site, "nvidia", "nccl", "include")
    lib = os.path.join(site, "nvidia", "nccl", "lib")
    if os.path.exists(os.path.join(inc, "nccl.h")) and os.path.exists(os.path.join(lib, "libnccl.so.2")):
        return inc, lib
    return "/usr/include", "/usr/lib/x86_64-linux-gnu"


def needs_build() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "b200lops.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return OUT
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    inc, lib = _nccl_paths()
    objs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        objs.append(obj)
        srcp = os.path.join(CSRC, src)
        if (not force and os.path.exists(obj) and os.path.getmtime(obj) > os.path.getmtime(srcp)
                and os.path.getmtime(obj) > os.path.getmtime(os.path.join(CSRC, "common.cuh"))
                and os.path.getmtime(obj) > os.path.getmtime(os.path.join(CSRC, "tc_ptx.cuh"))
                and os.path.getmtime(obj) > os.path.getmtime(os.path.join(INCLUDE, "b200lops.h"))):
            continue
        cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
               "-Xcompiler", "-fPIC", "-I", INCLUDE, "-I", inc, "-c", srcp, "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd))
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            print(f"[b200lops build] {src} FAILED:\n{out}", file=sys.stderr)
        elif verbose or out.strip():
            print(f"[b200lops build] {src}:\n{out}")
    if failed:
        raise RuntimeError("nvcc failed building libb200lops.so")
    link = [nvcc, "-shared", "-o", OUT] + objs + ["-L", lib, "-l:libnccl.so.2", "-lcuda",
            "-Xlinker", f"-rpath={lib}", "-Xlinker", "-rpath=/usr/lib/x86_64-linux-gnu"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        print(r.stdout, file=sys.stderr)
        raise RuntimeError("link of libb200lops.so failed")
    return OUT


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(path)
