"""Builds liblstep_b200.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

`python -m lstep_b200.build` or `lstep_b200.build.build()`; `__graft_entry__.build()` calls it.
nvcc cross-compiles without a GPU, so this runs in the build container; the .so travels to the
GPU box with the snapshot (it is git-ignored, not gpurun-ignored).
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "liblstep_b200.so")
STAMP = os.path.join(PKG, ".liblstep_b200.stamp")
SOURCES = ["api.cu", "sampler.cu", "dft_filter.cu", "mlp.cu", "mlp_cluster.cu", "mlp_umma.cu", "aggregate.cu", "update.cu", "update_push.cu", "csr_build.cu", "csr_grow.cu", "step.cu", "host_step.cu", "changelog.cu", "peer.cu"]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xcompiler", "-fPIC",
              "--shared", "-Xptxas", "-v", "-Wno-deprecated-gpu-targets"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; the lstep_b200 CUDA library cannot be built")


def cuobjdump() -> str:
    """The cuobjdump of the toolkit whose nvcc builds the library (CUDA's bin directory need not be on PATH), else the one
    on PATH."""
    nvcc = _nvcc()
    for cand in (os.path.join(os.path.dirname(d), "cuobjdump") for d in (nvcc, os.path.realpath(nvcc))):
        if os.path.exists(cand):
            return cand
    found = shutil.which("cuobjdump")
    if found is None:
        raise RuntimeError(f"cuobjdump not found next to {nvcc} or on PATH")
    return found


def _digest() -> str:
    """Content hash of the sources and flags. File NAMES enter relative to the repo (the snapshot on the GPU box lives
    under another path; an absolute path here would force a rebuild there, by every rank at once)."""
    h = hashlib.sha256()
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))] + [os.path.join(ROOT, "include", "lstep_b200.h")]
    for f in files:
        with open(f, "rb") as fh:
            h.update(os.path.basename(f).encode())
            h.update(fh.read())
    h.update((" ".join(NVCC_FLAGS) + os.environ.get("LSTEP_NVCC_EXTRA", "")).encode())
    return h.hexdigest()


def _up_to_date(dig: str) -> bool:
    return os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read().strip() == dig


def build(force: bool = False, verbose: bool = False) -> str:
    dig = _digest()
    if not force and _up_to_date(dig):
        return LIB
    import fcntl
    with open(os.path.join(PKG, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)  # one builder at a time (torchrun starts one process per GPU)
        try:
            if not force and _up_to_date(dig):  # another process built it while this one waited
                return LIB
            extra = os.environ.get("LSTEP_NVCC_EXTRA", "").split()  # e.g. -DLSTEP_MLP_TIMING for instrumented builds
            tmp = LIB + f".tmp{os.getpid()}"
            cmd = [_nvcc()] + NVCC_FLAGS + extra + ["-I", os.path.join(ROOT, "include"), "-I", CSRC, "-o", tmp] + \
                  [os.path.join(CSRC, s) for s in SOURCES]
            res = subprocess.run(cmd, capture_output=True, text=True)
            log = res.stdout + res.stderr
            with open(os.path.join(PKG, ".build.log"), "w") as fh:
                fh.write(" ".join(cmd) + "\n" + log)
            if res.returncode != 0:
                if os.path.exists(tmp):
                    os.remove(tmp)
                raise RuntimeError("nvcc failed:\n" + log[-6000:])
            if verbose:
                print(log)
            os.replace(tmp, LIB)  # atomic: a concurrent loader sees the old or the new library, never a partial file
            with open(STAMP, "w") as fh:
                fh.write(dig)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
