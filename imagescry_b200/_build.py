"""Compile csrc/*.cu into lib/libimagescry_b200.so with nvcc for sm_100a (in-tree, no JIT cache).

The shared object travels to the GPU box with the repo snapshot; `python -m imagescry_b200._build`
rebuilds it.  No torch headers are involved: the library exposes the plain C ABI declared in
include/imagescry_b200.h.
"""

from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB_DIR = os.path.join(PKG, "lib")
OBJ_DIR = os.path.join(LIB_DIR, "obj")
LIB = os.path.join(LIB_DIR, "libimagescry_b200.so")
STAMP = os.path.join(LIB_DIR, "build.stamp")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
    "-I", os.path.join(REPO, "include"),
    "-I", CSRC,
    "-DISX_BUILD",
]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found (set NVCC or add /usr/local/cuda/bin to PATH)")


def sources() -> list[str]:
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _extra_flags() -> list[str]:
    # diagnostic builds only, e.g. ISX_NVCC_EXTRA="-DISX_KNN_PROFILE" python -m imagescry_b200._build --force
    return os.environ.get("ISX_NVCC_EXTRA", "").split()


def _digest() -> str:
    # the flags are part of the digest: a library built with them is never taken for a plain build
    h = hashlib.sha256(repr(_extra_flags()).encode())
    files = sources() + sorted(
        os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))
    ) + [os.path.join(REPO, "include", "imagescry_b200.h"), os.path.abspath(__file__)]
    for f in files:
        h.update(f.encode())
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def is_current() -> bool:
    if not (os.path.exists(LIB) and os.path.exists(STAMP)):
        return False
    with open(STAMP) as fh:
        return fh.read().strip() == _digest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Build the library if any source changed.  Returns the path of the shared object."""
    if not force and is_current():
        return LIB
    os.makedirs(OBJ_DIR, exist_ok=True)
    nvcc = _nvcc()
    extra = ["-Xptxas", "-v"] if verbose else []
    extra += _extra_flags()

    def compile_one(src: str) -> str:
        obj = os.path.join(OBJ_DIR, os.path.basename(src)[:-3] + ".o")
        cmd = [nvcc, *NVCC_FLAGS, *extra, "-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        objs = list(ex.map(compile_one, sources()))
    cmd = [nvcc, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(STAMP, "w") as fh:
        fh.write(_digest())
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
