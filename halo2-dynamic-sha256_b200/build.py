"""Builds libh2sha_b200.so (CUDA kernels + C-ABI) in-tree with nvcc for sm_100a.

The library has no torch / Python dependency: it links only the CUDA runtime.  The SHA-256 of every source, header and
build flag is compiled into the library (`h2sha_build_id()`); `needs_build()` compares that stamp with the sources as
they are now, so a stale binary (the .so is git-ignored but travels to the GPU box) is never benchmarked.
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libh2sha_b200.so")
SOURCES = ["engine.cu", "planner.cc", "permutation.cc"]
HEADERS = ["h2sha_defs.h", "planner.h", "fr_host.h", "fr_dev.cuh", "lookup_geom.h", "lookup_prework.cuh", "batch_check.cuh", "grand_product.cuh", "lookup_product.cuh", "permutation.h", "permutation_product.cuh", "export.cuh", os.path.join("..", "..", "include", "h2sha_b200.h")]
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-cudart", "shared", "-ldl"]
MARKER = b"H2SHA_BUILD_ID="


def source_hash() -> str:
    h = hashlib.sha256()
    for f in SOURCES + HEADERS:
        p = os.path.join(CSRC, f)
        h.update(f.encode() + b"\0")
        if os.path.exists(p):
            with open(p, "rb") as fh:
                h.update(fh.read())
    h.update(" ".join(FLAGS).encode())
    return h.hexdigest()[:32]


def built_hash():
    """The stamp compiled into the in-tree library (read from the file, no dlopen), or None."""
    try:
        with open(LIB, "rb") as fh:
            blob = fh.read()
    except OSError:
        return None
    i = blob.find(MARKER)
    if i < 0:
        return None
    return blob[i + len(MARKER): i + len(MARKER) + 32].decode("ascii", "replace")


def needs_build() -> bool:
    return built_hash() != source_hash()


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + FLAGS + [f'-DH2SHA_BUILD_ID_STR="{source_hash()}"', "-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    subprocess.check_call(cmd)
    if built_hash() != source_hash():
        raise RuntimeError("the freshly built library does not carry the source stamp")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
