"""Builds libcia.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels
with the repo snapshot to the GPU box)."""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libcia.so")
SOURCES = ["api.cu", "scan.cu", "crop.cu", "cae_fp32.cu", "cae_tc.cu", "score.cu", "score_tc.cu", "segment.cu", "fit.cu", "transport.cu", "tiff_dev.cu", "host_rle.cpp", "host_tiff.cpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC"]


def _nvcc():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + \
           [os.path.join(HERE, "..", "include", "cia.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, os.path.splitext(src)[0] + ".o")
        objs.append(obj)
        if src.endswith(".cpp"):      # host-only sources: the host compiler directly
            cmd = [shutil.which("g++") or "g++", "-O3", "-std=c++17", "-fPIC", "-c", os.path.join(CSRC, src), "-o", obj]
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
            continue
        cmd = [_nvcc(), *NVCC_FLAGS, *os.environ.get("CIA_NVCC_EXTRA", "").split(), "-c",
               os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if verbose and out:
            print(out)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
    cmd = [_nvcc(), "-shared", "-o", LIB, *objs, "-lcudart"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    return LIB


if __name__ == "__main__":
    import sys
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
