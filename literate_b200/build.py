"""Builds literate_b200/_lib/libliterate_b200.so with nvcc for sm_100a, in-tree.

The shared library is the product; there is no CPU fallback and no other architecture.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
OUT_DIR = os.path.join(PKG, "_lib")
LIB = os.path.join(OUT_DIR, "libliterate_b200.so")
SOURCES = ["lr_api.cu", "k1_binstats.cu", "k3_chains.cu", "k4_direct.cu", "k5_summary.cu", "k6_trend.cu", "k7_ddrate.cu", "k8_hpd.cu", "k9_diag.cu", "k10_rank.cu", "k11_predictive.cu", "k12_loo.cu"]
HEADERS = ["lr_common.cuh", "chain_device.cuh", "k3_team.cuh", os.path.join(REPO, "include", "literate_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"] + os.environ.get("LR_EXTRA_NVCC_FLAGS", "").split()


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: literate_b200 needs the CUDA toolkit to build (no CPU fallback exists)")


def _digest():
    h = hashlib.sha256()
    h.update(" ".join(NVCC_FLAGS).encode())
    for f in SOURCES + HEADERS:
        p = f if os.path.isabs(f) else os.path.join(CSRC, f)
        with open(p, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def _up_to_date(dig):
    stamp = os.path.join(OUT_DIR, "build.sha256")
    return os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read().strip() == dig


def build(force=False, verbose=False):
    """Compile if sources changed; returns the path of the shared library.  Safe under torchrun: ranks serialise on a file
    lock, the first one compiles into rank-private object files and renames the finished library into place, the others
    find it up to date."""
    import fcntl
    os.makedirs(OUT_DIR, exist_ok=True)
    dig = _digest()
    if not force and _up_to_date(dig):
        return LIB
    with open(os.path.join(OUT_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and _up_to_date(dig):
                return LIB
            return _build_locked(dig, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(dig, verbose):
    stamp = os.path.join(OUT_DIR, "build.sha256")
    nvcc = _nvcc()
    objs = []
    log = []
    tmp_lib = LIB + ".tmp%d" % os.getpid()
    for src in SOURCES:
        obj = os.path.join(OUT_DIR, os.path.splitext(src)[0] + ".o")
        cmd = [nvcc] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        p = subprocess.run(cmd, capture_output=True, text=True)
        log.append("$ " + " ".join(cmd) + "\n" + p.stdout + p.stderr)
        if p.returncode != 0:
            sys.stderr.write(log[-1])
            raise RuntimeError("nvcc failed on " + src)
        objs.append(obj)
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", tmp_lib] + objs
    p = subprocess.run(cmd, capture_output=True, text=True)
    log.append("$ " + " ".join(cmd) + "\n" + p.stdout + p.stderr)
    if p.returncode != 0:
        sys.stderr.write(log[-1])
        raise RuntimeError("link failed")
    os.replace(tmp_lib, LIB)
    with open(os.path.join(OUT_DIR, "build.log"), "w") as fh:
        fh.write("\n".join(log))
    with open(stamp, "w") as fh:
        fh.write(dig)
    if verbose:
        print("\n".join(log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
