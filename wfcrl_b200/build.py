"""Builds libwfcrl_b200.so (hand-written sm_100a CUDA kernels + C-ABI) IN-TREE with nvcc.

Usage: python -m wfcrl_b200.build [--force]
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libwfcrl_b200.so")
SOURCES = ["wf_api.cu", "wf_kernels.cu", "wf_fast.cu", "wf_fast64.cu"]
HEADERS = ["wf_device.cuh", "wf_host_const.h", "gen_baked.cu", os.path.join("..", "..", "include", "wfcrl_b200.h")]
BAKED = os.path.join(CSRC, "wf_fast_baked.inc")
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-shared", "-Xcompiler", "-fPIC", "-Xptxas", "-v", "--resource-usage",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the wfcrl_b200 CUDA library cannot be built (there is no CPU fallback)")


def source_hash() -> str:
    """SHA-256 (first 16 hex digits) over every source the library is built from: csrc/*.cu, *.cuh, *.h (the generated
    wf_fast_baked.inc excluded: it is a function of gen_baked.cu + wf_host_const.h) and include/*.h, in name order."""
    h = hashlib.sha256()
    files = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h")))
    inc = os.path.join(HERE, "..", "include")
    paths = [os.path.join(CSRC, f) for f in files] + [os.path.join(inc, f) for f in sorted(os.listdir(inc)) if f.endswith(".h")]
    for path in paths:
        h.update(os.path.basename(path).encode() + b"\0")
        with open(path, "rb") as fp:
            h.update(fp.read())
        h.update(b"\0")
    return h.hexdigest()[:16]


def library_hash(path: str = LIB):
    """The source hash baked into a built library (read from the file, without loading it); None if absent."""
    try:
        with open(path, "rb") as fp:
            blob = fp.read()
    except OSError:
        return None
    tag = b"wfcrl_b200-src-sha256:"
    k = blob.find(tag)
    return blob[k + len(tag):k + len(tag) + 16].decode() if k >= 0 else None


def needs_build() -> bool:
    """True when the library is missing or was built from other sources than the ones in the tree (hash, not mtime)."""
    return library_hash() != source_hash()


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    # step 1: bake the default model's kernel constants into a header (host program built and run at build time)
    gen_exe = os.path.join(HERE, "_gen_baked")
    subprocess.run([_nvcc(), "-O1", "-std=c++17", "-o", gen_exe, os.path.join(CSRC, "gen_baked.cu")], check=True,
                   capture_output=True, text=True)
    with open(BAKED, "w") as fp:
        fp.write(subprocess.run([gen_exe], check=True, capture_output=True, text=True).stdout)
    os.remove(gen_exe)
    # step 2: the library
    # a function of the tree alone, so that the source hash wf_version() reports stands for the binary
    cmd = ([_nvcc()] + NVCC_FLAGS + [f'-DWF_SOURCE_HASH="{source_hash()}"', "-o", LIB] +
           [os.path.join(CSRC, s) for s in SOURCES])
    proc = subprocess.run(cmd, capture_output=True, text=True)
    log = proc.stdout + proc.stderr
    with open(os.path.join(HERE, "build.log"), "w") as fp:
        fp.write(" ".join(cmd) + "\n" + log)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + log)
    if verbose:
        print(log)
    return LIB


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose=True))
