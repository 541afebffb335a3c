"""In-tree build of the CUDA library (sm_100a only).  `python -m evacuation_b200.build`.

Staleness is decided by CONTENT, not by mtime: the SHA-256 of every file under csrc/ (`*.cu`, `*.cuh`) and
include/ (`*.h`) -- names and bytes -- is compiled into the library (`-DEVAC_BUILD_ID=...`, exported as
`evac_build_id()` and as the byte string ``EVAC_BUILD_ID=<hash>`` inside the binary).  `is_stale()` compares the
tree's hash with the one found in the binary; `_native.load()` does the same and rebuilds (or raises) on a mismatch,
so a test or benchmark can never run a library that was built from other sources than the ones in the tree.
"""
from __future__ import annotations

import glob
import hashlib
import os
import re
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
INCLUDE = os.path.join(os.path.dirname(PKG_DIR), "include")
LIB_PATH = os.environ.get("EVAC_B200_LIB") or os.path.join(PKG_DIR, "libevac_b200.so")  # override: a library built elsewhere (A/B runs)
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC"]
_ID_MARKER = b"EVAC_BUILD_ID="


def sources() -> list:
    """Translation units: every csrc/*.cu."""
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def headers() -> list:
    """Everything a translation unit can include from this tree: csrc/*.cuh and include/*.h."""
    return sorted(glob.glob(os.path.join(CSRC, "*.cuh"))) + sorted(glob.glob(os.path.join(INCLUDE, "*.h")))


def source_hash() -> str:
    """SHA-256 (first 16 hex digits) over the names and contents of sources() + headers()."""
    h = hashlib.sha256()
    for p in sources() + headers():
        h.update(os.path.basename(p).encode() + b"\0")
        with open(p, "rb") as f:
            h.update(f.read())
        h.update(b"\0")
    return h.hexdigest()[:16]


def library_build_id(path: str = None):
    """The build id embedded in the binary at `path` (read from the file's bytes; nothing is loaded), or None."""
    path = path or LIB_PATH
    if not os.path.exists(path):
        return None
    with open(path, "rb") as f:
        data = f.read()
    m = re.search(_ID_MARKER + rb"([0-9a-f]{16})", data)
    return m.group(1).decode() if m else None


def find_nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; evacuation_b200 has no CPU fallback and needs the CUDA toolkit to build")


def is_stale() -> bool:
    """True when the library is missing or was built from other sources than the tree holds now."""
    return library_build_id() != source_hash()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile libevac_b200.so next to this file (cross-compiles without a GPU)."""
    if not force and not is_stale():
        return LIB_PATH
    nvcc = find_nvcc()
    build_id = source_hash()
    objs, procs = [], []
    for src in sources():  # one nvcc per translation unit, in parallel
        obj = os.path.join(CSRC, os.path.splitext(os.path.basename(src))[0] + ".o")
        cmd = [nvcc, *NVCC_FLAGS, f'-DEVAC_BUILD_ID="{build_id}"', *(["-Xptxas=-v"] if verbose else []), "-c", "-o", obj, src]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        objs.append(obj)
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)))
    for cmd, pr in procs:
        out, err = pr.communicate()
        if pr.returncode != 0:
            raise RuntimeError(f"nvcc failed: {' '.join(cmd)}\n{out}\n{err}")
        if verbose:
            print(err, file=sys.stderr)
    tmp = LIB_PATH + ".tmp"
    res = subprocess.run([nvcc, "-shared", "-o", tmp, *objs], capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"link failed:\n{res.stdout}\n{res.stderr}")
    os.replace(tmp, LIB_PATH)
    if library_build_id() != build_id:
        raise RuntimeError(f"{LIB_PATH} does not carry build id {build_id} after the build (sources edited during the build?)")
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv), library_build_id())
