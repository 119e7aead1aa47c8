"""Builds the CUDA engine in-tree: geneticscre_b200/libgcre_b200.so (sm_100a only, -lineinfo).

A build happens only when a source is newer than the library.  Concurrent starters (the N ranks of a torchrun launch, pytest
workers) serialise on a lock file: one of them compiles into a temporary name and renames it over the library, the others
find it fresh when they get the lock - nobody ever dlopens a half-written file.  Run as a script
(``python geneticscre_b200/build.py [--force]``), a build also writes the ptxas resource table of the build (registers, spills and shared memory of every kernel) to the tracked
profiles/ptxas_sm100a.log; an ordinary build leaves the tracked files alone.
"""
from __future__ import annotations

import fcntl
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
LIB = os.path.join(PKG, "libgcre_b200.so")
CSRC = os.path.join(PKG, "csrc")
SOURCES = [os.path.join(CSRC, "gcre_capi.cu"), os.path.join(CSRC, "host_pack.cpp")]
SOURCE_SUFFIXES = (".cu", ".cuh", ".cpp", ".h", ".hpp")
PTXAS_LOG = os.path.join(ROOT, "profiles", "ptxas_sm100a.log")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC,-O3,-Wall,-pthread", "-shared", "-Xptxas", "-v", "-I", os.path.join(ROOT, "include")]


def dependencies() -> list:
    deps = [os.path.join(ROOT, "include", "gcre_b200.h")]
    deps += [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith(SOURCE_SUFFIXES) and not f.startswith(".")]
    return deps


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(d) > t for d in dependencies())


def build(force: bool = False, verbose: bool = False, ptxas_log: bool = False) -> str:
    if not force and not _stale():
        return LIB
    with open(os.path.join(PKG, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not _stale():  # another process built it while this one waited for the lock
                return LIB
            nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
            tmp = f"{LIB}.{os.getpid()}.tmp"
            cmd = [nvcc] + NVCC_FLAGS + ["-o", tmp] + SOURCES
            res = subprocess.run(cmd, capture_output=True, text=True)
            if verbose or res.returncode != 0:
                sys.stderr.write(res.stdout + res.stderr)
            if res.returncode != 0:
                if os.path.exists(tmp):
                    os.unlink(tmp)
                raise RuntimeError("nvcc failed building libgcre_b200.so")
            os.replace(tmp, LIB)  # atomic: a process that already mapped the old file keeps its inode
            if ptxas_log:
                with open(PTXAS_LOG, "w") as f:
                    f.write(res.stderr)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True, ptxas_log=True))
