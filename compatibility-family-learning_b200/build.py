"""Builds libcfl_b200.so (the C-ABI library) in-tree with nvcc for sm_100a.

    python compatibility-family-learning_b200/build.py [--force] [--verbose]

Objects go to compatibility-family-learning_b200/build/ (git-ignored), the library to
compatibility-family-learning_b200/cfl/_lib/libcfl_b200.so (git-ignored, travels with gpurun).
"""
from __future__ import annotations

import concurrent.futures as cf
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIBDIR = os.path.join(HERE, "cfl", "_lib")
LIB = os.path.join(LIBDIR, "libcfl_b200.so")
SOURCES = ["api.cu", "pair.cu", "project.cu", "project_umma.cu", "project_bwd_umma.cu", "score.cu", "score_umma.cu", "score_lb.cu", "score_monomer.cu", "score_monomer_tc.cu", "rank_counts.cu", "rank_counts_tc.cu", "within.cu", "auc.cu"]
EXTRA = os.environ.get("CFL_NVCC_EXTRA", "").split()
NVCC_FLAGS = EXTRA + ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v", "-I", os.path.join(ROOT, "include"), "-I", CSRC]


def _nvcc() -> str:
    for c in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found: the CFL B200 library cannot be built (no fallback)")


def _digest() -> str:
    h = hashlib.sha256()
    files = sorted(os.listdir(CSRC)) + [os.path.join(ROOT, "include", "cfl_b200.h")]
    for f in files:
        p = f if os.path.isabs(f) else os.path.join(CSRC, f)
        with open(p, "rb") as fh:
            h.update(fh.read())
    # flags with the checkout's location factored out: the library built here must count as fresh in a copy of the tree
    # under another path (the GPU box runs a snapshot from a scratch directory)
    h.update(" ".join(f.replace(ROOT, "<root>") for f in NVCC_FLAGS).encode())
    return h.hexdigest()


def _compile(src: str, verbose: bool) -> str:
    obj = os.path.join(OBJ, src.replace(".cu", ".o"))
    cmd = [_nvcc(), *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    with open(obj.replace(".o", ".log"), "w") as fh:
        fh.write(r.stdout + r.stderr)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed on {src}:\n{r.stdout}\n{r.stderr}")
    if verbose:
        print(r.stderr)
    return obj


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(LIBDIR, exist_ok=True)
    stamp = os.path.join(LIBDIR, "libcfl_b200.sha256")
    dig = _digest()
    def fresh() -> bool:
        return os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == dig

    if not force and fresh():
        return LIB
    # one builder at a time (several ranks of one torchrun job may get here together): the others wait on the lock
    # and find the library fresh when they get it
    import fcntl
    with open(os.path.join(OBJ, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and fresh():
                return LIB
            with cf.ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
                objs = list(ex.map(lambda s: _compile(s, verbose), SOURCES))
            tmp = LIB + ".tmp%d" % os.getpid()
            cmd = [_nvcc(), "-shared", "-o", tmp, *objs, "-lcudart"]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
            os.replace(tmp, LIB)                                   # a process that has the old library mapped keeps it
            with open(stamp, "w") as fh:
                fh.write(dig)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
