"""Builds spacefortress_b200/libsf_b200.so (C-ABI, include/sf_b200.h) in-tree with nvcc for sm_100a.

The .so is git-ignored but travels to the GPU box with the repository snapshot. There is no other
implementation of the hot path: if this library is missing the package refuses to work.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libsf_b200.so")
SOURCES = ["sf_kernels.cu", "sf_tables.cpp"]
HEADERS = ["sf_geom.h", "sf_tables.h", "sf_state.cuh", "sf_probe.cuh", "sf_step.cuh", "sf_render.cuh", os.path.join("..", "..", "include", "sf_b200.h")]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force=False, verbose=False, out=None, defs=None):
    """out / defs: a variant build beside the product library, e.g. a probe of csrc/sf_probe.cuh (defs="-DSF_TIMELINE")."""
    if out is None and not force and not needs_build():
        return LIB
    if out is not None:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    cmd = [
        _nvcc(), "-shared", "-o", out or LIB,
        "-gencode", "arch=compute_100a,code=sm_100a",
        "-O3", "-lineinfo", "-std=c++17",
        # host side (static tables) and device side must not contract a*b+c: the model is defined
        # with individually rounded operations (sf_geom.h)
        "-Xcompiler", "-fPIC,-O2,-ffp-contract=off",
        "--fmad=false",
        "-Xptxas", "-v" if verbose else "-O3",
        "-I", os.path.join(HERE, "..", "include"),
    ] + (defs or "").split() + [os.path.join(CSRC, s) for s in SOURCES]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n%s\n%s" % (r.stdout, r.stderr))
    if verbose:
        print(r.stderr)
    return out or LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
