"""In-tree build of the CUDA C-ABI library (sm_100a only) with plain nvcc.

    python -m pioneer_b200.build [--force] [--verbose]

Output: pioneer_b200/_lib/libpioneer_b200.so (git-ignored; travels to the GPU box with gpurun).
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "_lib")
LIB_PATH = os.path.join(LIB_DIR, "libpioneer_b200.so")
SOURCES = ["pnr_kernels.cu", "pnr_dynamic.cu", "pnr_dynamic_bullet.cu", "pnr_filter.cu", "pnr_api.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "--threads", "4",
              "-Xcompiler", "-fPIC,-O2", "-shared"]


def _sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


HASH_MARKER = b"PNR_SRC_HASH:"


def _source_hash() -> str:
    """Content hash of everything the library is built from (file times do not survive a snapshot copy to another box)."""
    import hashlib
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    deps = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC)) + [os.path.join(HERE, "..", "include", "pioneer_b200.h")]
    for d in deps:
        h.update(os.path.basename(d).encode())
        with open(d, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _built_hash(path: str) -> str:
    """The hash the library carries inside itself (pnr_source_hash() in pnr_api.cu), read from the file without loading it."""
    try:
        with open(path, "rb") as f:
            blob = f.read()
    except OSError:
        return ""
    i = blob.find(HASH_MARKER)
    return blob[i + len(HASH_MARKER):i + len(HASH_MARKER) + 64].decode("ascii", "replace") if i >= 0 else ""


def _stale() -> bool:
    return _built_hash(LIB_PATH) != _source_hash()


def build(force: bool = False, verbose: bool = False) -> str:
    """Safe when several processes (the ranks of a torchrun job) import the package at once: one of them builds under a
    file lock into a temporary file that is renamed into place, the others wait and find the library fresh."""
    import fcntl
    out = LIB_PATH
    if not force and not _stale():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    extra = os.environ.get("PNR_EXTRA_NVCC_FLAGS", "").split()     # developer experiments (e.g. -DPNR_STEP_MIN_CTAS=6)
    if extra:
        out = os.environ.get("PNR_LIB_OUT", out)
    product = (out == LIB_PATH)
    with open(os.path.join(LIB_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if product and not force and not _stale():             # another process built it while we waited
                return LIB_PATH
            nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
            tmp = f"{out}.tmp.{os.getpid()}"
            cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) \
                + [f'-DPNR_SRC_HASH="{_source_hash()}"'] + _sources() + ["-o", tmp]
            proc = subprocess.run(cmd, capture_output=True, text=True)
            if proc.returncode != 0:
                if os.path.exists(tmp):
                    os.remove(tmp)
                raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + proc.stdout + proc.stderr)
            os.replace(tmp, out)                                   # atomic: readers see the old or the new file, never a part
            if verbose:
                print(proc.stdout + proc.stderr)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
