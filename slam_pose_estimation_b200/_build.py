"""Builds the CUDA engine (csrc/ukf_batch.cu -> lib/libukfb.so) for sm_100a with nvcc.

nvcc cross-compiles without a GPU, so this runs in the GPU-less build container; the
resulting .so stays in-tree (git-ignored) and travels to the GPU box with the snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_PKG, "csrc")
# UKFB_LIB: load another build of the same library (kernel tuning experiments)
LIB = os.environ.get("UKFB_LIB") or os.path.join(_PKG, "lib", "libukfb.so")
SOURCES = ["ukf_batch.cu"]
DEPS = ["ukf_batch.cu", "ukf_device.cuh", "ukf_thread.cuh", "ukf_pose_fast.cuh", "ukf_ori_fast.cuh", "ukf_index.cuh", "so3.cuh", "simt.cuh", "../../include/ukf_batch.h", "../../include/ukfb_constants.h"]
# the step kernels' sources: what source_hash() covers (ukf_index.cuh holds per-filter access kernels, no step code)
STEP_KERNEL_SOURCES = ["simt.cuh", "so3.cuh", "ukf_device.cuh", "ukf_ori_fast.cuh", "ukf_pose_fast.cuh", "ukf_thread.cuh"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-shared", "-Xcompiler", "-fPIC",
]


def nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the engine is CUDA-only and cannot be built without the CUDA toolkit")


def source_hash() -> str:
    """sha256 (first 16 hex digits) of the STEP KERNEL sources (STEP_KERNEL_SOURCES; the host side of the ABI in
    ukf_batch.cu and the per-filter access kernels do not change what a step executes) the library is built from:
    profiles/traffic.json is stamped with it, so that ncu figures of an older kernel are not reported for a newer one.
    Comments and white space do not count."""
    import hashlib
    import re

    h = hashlib.sha256()
    for d in sorted(STEP_KERNEL_SOURCES):
        with open(os.path.join(CSRC, d), "r") as f:
            code = re.sub(r"/\*.*?\*/|//[^\n]*", " ", f.read(), flags=re.S)
        h.update(d.encode() + b"\0" + " ".join(code.split()).encode())
    return h.hexdigest()[:16]


def _content_hash() -> str:
    """sha256 of everything the library is compiled from, and of the flags"""
    import hashlib

    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for d in DEPS:
        with open(os.path.join(CSRC, d), "rb") as f:
            h.update(d.encode() + b"\0" + f.read())
    return h.hexdigest()


def stale() -> bool:
    """Is the library missing or built from other sources?  By content (the hash written next to the library when it was
    built), not by time stamps: a snapshot copied to another machine keeps contents, not necessarily times.  A library
    given through UKFB_LIB is taken as it is."""
    if not os.path.exists(LIB):
        return True
    if os.environ.get("UKFB_LIB"):
        return False
    try:
        with open(LIB + ".srchash") as f:
            return f.read().strip() != _content_hash()
    except OSError:
        t = os.path.getmtime(LIB)  # a library from before the hash file existed
        return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def build(force: bool = False, verbose: bool = False, extra: list[str] | None = None) -> str:
    """Compile lib/libukfb.so if missing or older than its sources; returns its path."""
    if not force and not stale():
        return LIB
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    cmd = [nvcc(), *NVCC_FLAGS, *(extra or []), "-o", LIB + ".tmp", *[os.path.join(CSRC, s) for s in SOURCES]]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd))
    subprocess.run(cmd, check=True, cwd=CSRC)
    os.replace(LIB + ".tmp", LIB)
    if not extra:
        with open(LIB + ".srchash", "w") as f:
            f.write(_content_hash() + "\n")
    return LIB


if __name__ == "__main__":
    import sys

    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
