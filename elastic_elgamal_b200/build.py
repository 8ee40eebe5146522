"""Builds the in-tree CUDA library (libeg_b200.so) for sm_100a with nvcc.

`python -m elastic_elgamal_b200.build` or `__graft_entry__.build()`.  The .so is git-ignored but travels to the
GPU box with the repo snapshot.  nvcc cross-compiles without a GPU.
"""
import pathlib
import shutil
import subprocess
import sys

PKG = pathlib.Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "libeg_b200.so"
SOURCES = [CSRC / "eg_b200.cu"]
HEADERS = sorted(CSRC.glob("*.cuh")) + sorted(CSRC.glob("*.inc")) + [PKG.parent / "include" / "eg_b200.h"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared", "-cudart", "static",
]


def needs_build(lib=LIB):
    if not lib.exists():
        return True
    t = lib.stat().st_mtime
    return any(p.stat().st_mtime > t for p in SOURCES + HEADERS)


def build(force=False, verbose=False, lib=LIB):
    """Compiles the library to `lib` unless it is newer than every source; the engine loads LIB unless EG_B200_LIB names
    another file."""
    if not force and not needs_build(lib):
        return lib
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    # EG_B200_WIDE_BITS=16|20 at build time: the small-footprint variant (48 MiB / 0.61 GiB per fixed-base table instead of
    # the default 8.25 GiB of 24-bit windows; csrc/ge.cuh), e.g. for several processes sharing one GPU
    import os
    bits = os.environ.get("EG_B200_WIDE_BITS")
    extra = ["-DEG_WIDE_BITS=%d" % int(bits)] if bits else []
    cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-o", str(lib)] + [str(s) for s in SOURCES]
    proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + proc.stdout)
    if verbose:
        print(proc.stdout)
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
