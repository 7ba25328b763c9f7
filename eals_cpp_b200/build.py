"""In-tree build of libeals_b200.so (nvcc, sm_100a only).  Cross-compiles without a GPU.

Staleness is decided by CONTENT, not by modification times: a digest of every source file and of the
compiler flags is stored next to the artefact (`<artefact>.stamp`).  After a checkout, a copy to another
box or a `touch`, the artefact is rebuilt exactly when it was built from different sources."""
from __future__ import annotations

import hashlib
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIB_DIR, "libeals_b200.so")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def _sources():
    deps = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh"))]
    deps.append(os.path.join(ROOT, "include", "eals_b200.h"))
    return deps


def _digest(paths, extra) -> str:
    h = hashlib.sha256(repr(extra).encode())
    for p in paths:
        h.update(os.path.basename(p).encode())
        with open(p, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _fresh(artefact: str, digest: str) -> bool:
    try:
        with open(artefact + ".stamp") as f:
            return os.path.exists(artefact) and f.read().strip() == digest
    except OSError:
        return False


def _stamp(artefact: str, digest: str) -> None:
    with open(artefact + ".stamp", "w") as f:
        f.write(digest + "\n")


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/eals_b200.cu -> lib/libeals_b200.so unless it was built from exactly these sources."""
    os.makedirs(LIB_DIR, exist_ok=True)
    digest = _digest(_sources(), NVCC_FLAGS)
    if not force and _fresh(LIB, digest):
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc, *NVCC_FLAGS, "-o", LIB, os.path.join(CSRC, "eals_b200.cu")]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    subprocess.run(cmd, check=True)
    _stamp(LIB, digest)
    return LIB


def build_host_example(force: bool = False) -> str:
    """Compile the C++ drop-in driver (host/eals_main.cpp over include/MF_fastALS.h) against the
    library — the 'same three call sites' check of SURVEY.md §8b."""
    src = os.path.join(HERE, "host", "eals_main.cpp")
    out = os.path.join(LIB_DIR, "eals_main")
    if not os.path.exists(src):
        return ""
    deps = [src, os.path.join(ROOT, "include", "MF_fastALS.h"), os.path.join(ROOT, "include", "eals_b200.h"),
            os.path.join(ROOT, "include", "eals_host_types.h")]
    cmd = ["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "include"), src, "-o", out,
           "-L", LIB_DIR, "-leals_b200", "-Wl,-rpath,$ORIGIN"]
    # paths relative to the tree: a built tree that is moved or copied stays fresh
    digest = _digest(deps, [os.path.relpath(c, ROOT) if os.path.isabs(c) else c for c in cmd])
    if not force and _fresh(out, digest):
        return out
    subprocess.run(cmd, check=True)
    _stamp(out, digest)
    return out


if __name__ == "__main__":
    print(build_library(force=True, verbose=True))
    print(build_host_example(force=True))
