"""Builds lightzero_b200/_lib/liblzb200.so (the C-ABI library, include/lzb200.h) with nvcc for sm_100a.

In-tree build: the .so is git-ignored but travels to the GPU box with the gpurun snapshot.
tree.cu and gumbel.cu are compiled with -fmad=false (the reference tree is built for baseline x86-64 and never
contracts a*b+c; bit-exact visit counts depend on it); the network kernels want FMA.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "_lib")
LIB = os.path.join(LIBDIR, "liblzb200.so")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fno-fast-math"]
# Experiment builds: `python -m lightzero_b200._build --tag NAME -DFOO ...` writes _lib/NAME/liblzb200.so with the extra
# defines; LZ_LIB_TAG=NAME makes cabi.load() pick it (one GPU session can then compare several kernel variants).
UNITS = [("tree.cu", ["-fmad=false"]), ("gumbel.cu", ["-fmad=false"]), ("model.cu", []), ("net_tc.cu", []), ("conv_tc.cu", []), ("mlp.cu", []), ("ez.cu", []), ("search.cu", []), ("collector.cu", [])]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, tag: str = None, defines=()) -> str:
    libdir = os.path.join(LIBDIR, tag) if tag else LIBDIR
    lib = os.path.join(libdir, "liblzb200.so")
    os.makedirs(libdir, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "lzb200.h"))
    objs = []
    for src, extra in UNITS:
        s = os.path.join(CSRC, src)
        o = os.path.join(libdir, src.replace(".cu", ".o"))
        if force or _stale(o, [s] + headers):
            cmd = ["nvcc"] + ARCH + COMMON + list(defines) + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            subprocess.check_call(cmd)
        objs.append(o)
    if force or _stale(lib, objs):
        subprocess.check_call(["nvcc"] + ARCH + ["-shared", "-o", lib] + objs)
    return lib


if __name__ == "__main__":
    _tag = sys.argv[sys.argv.index("--tag") + 1] if "--tag" in sys.argv else None
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, tag=_tag, defines=[a for a in sys.argv[1:] if a.startswith("-D")]))
