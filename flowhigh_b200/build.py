"""Builds libflowhigh_b200.so (all CUDA kernels + the C ABI) in-tree for sm_100a.

    python -m flowhigh_b200.build            # nvcc cross-compiles without a GPU

The shared object lands in flowhigh_b200/lib/ so that it travels with the source tree
(no JIT cache).  There is exactly one target architecture: sm_100a.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIBNAME = "libflowhigh_b200.so"
SOURCES = ["dsp.cu", "backbone.cu", "vocoder_f32.cu", "vocoder_tc.cu", "tc_conv.cu", "attention_tc5.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]


def lib_path() -> str:
    # FLOWHIGH_B200_LIB: an explicitly built variant (A/B of compile-time options, tools/build_variant.sh); never rebuilt
    return os.environ.get("FLOWHIGH_B200_LIB") or os.path.join(LIBDIR, LIBNAME)


def _needs_build() -> bool:
    out = lib_path()
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "flowhigh_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if os.environ.get("FLOWHIGH_B200_LIB"):
        return lib_path()
    if not force and not _needs_build():
        return lib_path()
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(LIBDIR, exist_ok=True)
    objdir = os.path.join(LIBDIR, "obj")
    os.makedirs(objdir, exist_ok=True)

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-o", lib_path(), *objs, "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    return lib_path()


if __name__ == "__main__":
    p = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(p)
