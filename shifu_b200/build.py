"""In-tree build of ``libshifu_b200.so`` (nvcc, sm_100a only).

    python -m shifu_b200.build            # (re)build when the sources differ from the ones the .so was built from

nvcc cross-compiles without a GPU, so this also runs in the CPU-only build container.  The built
library stays inside the package directory (git-ignored) so that it travels with the repo snapshot
to the GPU box and is visible to the driver's "which .so got loaded" check.
"""
from __future__ import annotations

import fcntl
import hashlib
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
INCLUDE = os.path.join(os.path.dirname(PKG_DIR), "include")
LIB_PATH = os.path.join(PKG_DIR, "libshifu_b200.so")

SOURCES = ["capi.cu"]
DEPS = ["capi.cu", "a1_kernels.cuh", "a1_fused.cuh", "a1_fused_tma.cuh", "a1_fused_kernel.inc", "a1_fused_tma_kernel.inc", "tma_pipe.cuh", "f32x2.cuh","abb_kernels.cuh", "arm_ik.cuh", "camera_gather.cuh", "common_kernels.cuh", "exact_math.cuh", "philox.cuh", "terrain_gen.cuh", "scan_pairs.cuh"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--fmad=false",                    # no implicit FMA contraction: see csrc/exact_math.cuh
    "-Xcompiler", "-fPIC", "-shared",
    "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libshifu_b200.so cannot be built (there is no CPU fallback)")


STAMP_PATH = LIB_PATH + ".srchash"      # hash of the sources the library was built from
LOCK_PATH = LIB_PATH + ".lock"


def _dep_paths():
    return [os.path.join(CSRC, d) for d in DEPS] + [os.path.join(INCLUDE, "shifu_b200.h")]


def source_hash() -> str:
    """Content hash of every source the library depends on (+ the flags).  Content, not mtimes:
    a repo snapshot copied to another machine, or a ``git checkout`` of an unchanged file, must not
    trigger a rebuild — with one process per GPU that would mean N concurrent nvcc runs."""
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for path in _dep_paths():
        with open(path, "rb") as f:
            h.update(os.path.basename(path).encode() + b"\0" + f.read())     # not the absolute path: the tree moves
    return h.hexdigest()


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH) or os.path.getsize(LIB_PATH) == 0:
        return True
    try:
        with open(STAMP_PATH) as f:
            return f.read().strip() != source_hash()
    except OSError:
        # no stamp (library built by hand): fall back to modification times
        t = os.path.getmtime(LIB_PATH)
        return any(os.path.getmtime(d) > t for d in _dep_paths())


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB_PATH
    # one builder at a time (ranks of a torchrun job share the tree); the others wait, then find
    # the library up to date.  The library is written under a temporary name and renamed into
    # place, so a concurrent reader never maps a half-written file.
    with open(LOCK_PATH, "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():
                return LIB_PATH
            return _build_locked(verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(verbose: bool) -> str:
    tmp = f"{LIB_PATH}.tmp{os.getpid()}"
    cmd = [_nvcc(), *NVCC_FLAGS, "-I", INCLUDE, "-o", tmp] + [os.path.join(CSRC, s) for s in SOURCES]
    digest = source_hash()
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        if os.path.exists(tmp):
            os.remove(tmp)
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    os.replace(tmp, LIB_PATH)
    with open(STAMP_PATH + ".tmp", "w") as f:
        f.write(digest + "\n")
    os.replace(STAMP_PATH + ".tmp", STAMP_PATH)
    log = res.stdout + res.stderr
    with open(os.path.join(PKG_DIR, "csrc", "ptxas.log"), "w") as f:
        f.write(log)
    if verbose:
        print(log)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
