"""Builds libtwixt_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m twixt_for_open_spiel_b200.build [--force]
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
INCLUDE = os.path.join(os.path.dirname(PKG), "include")
LIB = os.path.join(PKG, "libtwixt_b200.so")
OBJ_DIR = os.path.join(PKG, "build")
# (source, extra flags, object): the playout kernel is compiled once per size group (see its last section)
SOURCES = [("twixt_kernels_api.cu", [], "twixt_kernels_api.o"), ("twixt_batch.cu", [], "twixt_batch.o"),
           ("twixt_mcts.cu", [], "twixt_mcts.o")] + [
    ("twixt_kernel_playout.cu", ["-DTW_PLAYOUT_GROUP=%d" % g], "twixt_kernel_playout_g%d.o" % g) for g in range(5)]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2", "--expt-relaxed-constexpr",
] + os.environ.get("TWIXT_NVCC_EXTRA", "").split()  # experiments only (e.g. -DTW_X=1)


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libtwixt_b200.so cannot be built")


def nvcc_path() -> str:
    return _nvcc()


def _fingerprint() -> str:
    h = hashlib.sha256()
    names = sorted(os.listdir(CSRC)) + ["../../include/twixt_b200.h"]
    for name in names:
        path = os.path.normpath(os.path.join(CSRC, name))
        if os.path.isfile(path):
            with open(path, "rb") as f:
                h.update(name.encode())
                h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def needs_build() -> bool:
    stamp = os.path.join(OBJ_DIR, "fingerprint")
    if not os.path.exists(LIB) or not os.path.exists(stamp):
        return True
    with open(stamp) as f:
        return f.read().strip() != _fingerprint()


def build(force: bool = False, verbose: bool = False, out: str = None, extra_flags=()) -> str:
    """Build the library.  `out` / `extra_flags` build a VARIANT elsewhere (tests use it for the playout
    kernel's bounds-checking build, tools/ab_playout.py for timing experiments); the default build is the
    product."""
    variant = out is not None
    lib = out if variant else LIB
    obj_dir = (os.path.splitext(out)[0] + "_obj") if variant else OBJ_DIR
    if not variant and not force and not needs_build():
        return LIB
    nvcc = _nvcc()
    os.makedirs(obj_dir, exist_ok=True)
    # ranks started together (torchrun) must not compile into the same object directory at once
    import fcntl
    lock = open(os.path.join(obj_dir, ".lock"), "w")
    fcntl.flock(lock, fcntl.LOCK_EX)
    try:
        if not variant and not force and not needs_build():
            return LIB  # another process built it while we waited
        return _build_locked(nvcc, lib, obj_dir, variant, verbose, extra_flags)
    finally:
        fcntl.flock(lock, fcntl.LOCK_UN)
        lock.close()


def _build_locked(nvcc, lib, obj_dir, variant, verbose, extra_flags) -> str:

    def compile_one(job) -> str:
        src, flags, obj_name = job
        obj = os.path.join(obj_dir, obj_name)
        cmd = [nvcc, *NVCC_FLAGS, *flags, *extra_flags, "-I", INCLUDE, "-I", CSRC, "-c", os.path.join(CSRC, src),
               "-o", obj]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, res.stdout, res.stderr))
        if verbose and (res.stdout or res.stderr):
            print(res.stdout, res.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 4)) as pool:
        objs = list(pool.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-o", lib, *objs, "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (res.stdout, res.stderr))
    if not variant:
        with open(os.path.join(OBJ_DIR, "fingerprint"), "w") as f:
            f.write(_fingerprint())
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
