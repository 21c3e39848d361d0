"""Build libzsgpu.so (the sm_100a CUDA engine + C ABI) in-tree with nvcc.

The shared library is written next to this file so that it travels to the GPU box with the repo
snapshot (it is git-ignored).  nvcc cross-compiles for sm_100a without a GPU.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libzsgpu.so")
SOURCES = ["zs_api.cu", "zs_checksum.cu", "zs_inflate.cu", "zs_inflate_par.cu", "zs_inflate_tps.cu", "zs_lz77.cu", "zs_huff.cu", "zs_stream.cu", "zs_gunzip.cu", "zs_inflate_index.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--use_fast_math",
    "-diag-suppress", "550",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libzsgpu cannot be built (there is no CPU fallback)")


def needs_build() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "zsgpu.h")]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return OUT
    nvcc = _nvcc()
    extra = os.environ.get("ZS_NVCC_EXTRA", "").split()   # e.g. -DZS_LZ_PROF for the role-cycle dump
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc, *NVCC_FLAGS, *extra, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            failed = True
            sys.stderr.write(f"nvcc failed for {src}:\n{out}\n")
        elif verbose and out:
            sys.stderr.write(out)
    if failed:
        raise RuntimeError("libzsgpu build failed")
    link = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", OUT, *objs, "-lcudart"]
    subprocess.run(link, check=True)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
