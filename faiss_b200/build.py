"""Build libfaiss_b200.so in-tree with nvcc for sm_100a (no JIT cache, no torch extension).

Usage: python faiss_b200/build.py [-j N] [--force]   (a script: importing the package needs the library it builds)
Objects go to faiss_b200/csrc/_obj/, the library to faiss_b200/libfaiss_b200.so.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(SRC, "_obj")
LIB = os.path.join(HERE, "libfaiss_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "--expt-relaxed-constexpr", "-I" + os.path.join(HERE, "..", "include"), "-I" + SRC,
]


def _sources():
    out = []
    for f in sorted(os.listdir(SRC)):
        if f.endswith(".cu") or f.endswith(".cpp"):
            out.append(os.path.join(SRC, f))
    return out


def _headers_mtime():
    m = 0.0
    for root in (SRC, os.path.join(HERE, "..", "include")):
        for f in os.listdir(root):
            if f.endswith((".h", ".cuh")):
                m = max(m, os.path.getmtime(os.path.join(root, f)))
    return m


def build(jobs=None, force=False, verbose=True):
    os.makedirs(OBJ, exist_ok=True)
    srcs = _sources()
    hm = _headers_mtime()
    todo = []
    objs = []
    for s in srcs:
        o = os.path.join(OBJ, os.path.basename(s) + ".o")
        objs.append(o)
        if force or not os.path.exists(o) or os.path.getmtime(o) < max(os.path.getmtime(s), hm):
            todo.append((s, o))

    def cc(so):
        s, o = so
        cmd = [NVCC] + FLAGS + ["-x", "cu", "-c", s, "-o", o]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (s, r.stdout, r.stderr))
        if verbose and r.stderr.strip():
            sys.stderr.write(r.stderr)
        return o

    if todo:
        if verbose:
            print("[faiss_b200.build] compiling %d file(s) for sm_100a" % len(todo), flush=True)
        with ThreadPoolExecutor(max_workers=jobs or min(8, os.cpu_count() or 4)) as ex:
            list(ex.map(cc, todo))
    if todo or not os.path.exists(LIB):
        cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-lcudart", "-ldl", "-Xlinker", "-z", "-Xlinker", "defs"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
        if verbose:
            print("[faiss_b200.build] linked", LIB, flush=True)
    return LIB


if __name__ == "__main__":
    j = None
    if "-j" in sys.argv:
        j = int(sys.argv[sys.argv.index("-j") + 1])
    build(jobs=j, force="--force" in sys.argv)
