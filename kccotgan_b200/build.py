"""Build libkccot.so (all CUDA sources under csrc/) for sm_100a, in-tree.

    python -m kccotgan_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU box with the
repo snapshot.  Objects are rebuilt only when their source (or any header) is newer.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(HERE, "csrc", "build")
LIB = os.path.join(HERE, "libkccot.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
         "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-Xptxas", "-v"]


def _sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def _headers_mtime():
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hs.append(os.path.join(os.path.dirname(HERE), "include", "kccot.h"))
    return max(os.path.getmtime(h) for h in hs)


def _compile(src, verbose):
    obj = os.path.join(BUILD, src[:-3] + ".o")
    cmd = [NVCC, *FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    log = r.stdout + r.stderr
    with open(obj + ".log", "w") as f:
        f.write(log)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed on {src}:\n{log}")
    if verbose:
        print(log)
    return obj


def build(force=False, verbose=False):
    os.makedirs(BUILD, exist_ok=True)
    hm = _headers_mtime()
    todo, objs = [], []
    for src in _sources():
        obj = os.path.join(BUILD, src[:-3] + ".o")
        objs.append(obj)
        newest = max(os.path.getmtime(os.path.join(CSRC, src)), hm)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < newest:
            todo.append(src)
    if todo:
        with ThreadPoolExecutor(max_workers=min(8, len(todo))) as ex:
            list(ex.map(lambda s: _compile(s, verbose), todo))
    if todo or not os.path.exists(LIB):
        cmd = [NVCC, "-shared", "-o", LIB, *objs, "-lcudart"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
