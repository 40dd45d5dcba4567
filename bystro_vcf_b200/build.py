"""Builds libbvcf.so (and the synthetic-workload helper library) in-tree with nvcc for sm_100a.

nvcc cross-compiles without a GPU, so this runs on the CPU-only build box; the .so travels to the
GPU box with the repo snapshot.  Usage: python -m bystro_vcf_b200.build [--force]
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
ROOT = os.path.dirname(HERE)

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared", "-diag-suppress", "128",
]

TARGETS = {
    "libbvcf.so": (["bvcf_api.cu", "bvcf_index.cpp", "bvcf_bgzf.cpp"], ["-lz"]),
    # host and device must produce the same bytes: no FMA contraction in the generator
    "libbvcfsynth.so": (["bvcf_synth.cu"], ["-fmad=false"]),
}


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def _stale(out: str, srcs) -> bool:
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(ROOT, "include", "bvcf.h")]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> None:
    os.makedirs(LIBDIR, exist_ok=True)
    for lib, (srcs, extra) in TARGETS.items():
        srcs = [os.path.join(CSRC, s) for s in srcs]
        if not all(os.path.exists(s) for s in srcs):
            continue
        out = os.path.join(LIBDIR, lib)
        if not force and not _stale(out, srcs):
            continue
        cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + extra + ["-o", out] + srcs
        print("[build]", " ".join(cmd), file=sys.stderr)
        subprocess.check_call(cmd)


def _arrow_paths():
    """include dir, library dir and library file of the Arrow C++ that ships inside the pyarrow wheel, or None"""
    try:
        import pyarrow
    except Exception:
        return None
    inc = pyarrow.get_include()
    for d in pyarrow.get_library_dirs():
        for f in sorted(os.listdir(d)):
            if f.startswith("libarrow.so."):
                return inc, d, f
    return None


def build_host(force: bool = False) -> str:
    """g++ build of the C++ host binary (the reference's main()/readVcf over the C ABI).  The Arrow IPC writer of
    --dosageOutput links the libarrow of the pyarrow wheel; without pyarrow the binary is built with -DBVCF_NO_ARROW."""
    bindir = os.path.join(HERE, "bin")
    os.makedirs(bindir, exist_ok=True)
    out = os.path.join(bindir, "bystro-vcf-b200")
    src = os.path.join(CSRC, "bvcf_host.cpp")
    asrc = os.path.join(CSRC, "bvcf_arrow.cpp")
    lib = os.path.join(LIBDIR, "libbvcf.so")
    deps = [src, asrc, lib, os.path.join(CSRC, "bvcf_arrow.h"), os.path.join(ROOT, "include", "bvcf.h")]
    if force or not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(d) for d in deps):
        arrow = _arrow_paths()
        objs, extra = [], []
        if arrow:
            inc, libdir, libfile = arrow
            aobj = os.path.join(bindir, "bvcf_arrow.o")
            cmd = ["g++", "-O2", "-std=c++20", "-Wall", "-c", "-I", inc, "-o", aobj, asrc]
            print("[build]", " ".join(cmd), file=sys.stderr)
            subprocess.check_call(cmd)
            objs.append(aobj)
            extra = ["-L", libdir, "-l:" + libfile, "-Wl,-rpath," + libdir]
        else:
            extra = ["-DBVCF_NO_ARROW"]
        cmd = (["g++", "-O2", "-std=c++17", "-Wall", "-pthread", "-o", out, src] + objs +
               ["-L", LIBDIR, "-lbvcf", "-lz", "-Wl,-rpath,$ORIGIN/../lib"] + extra)
        print("[build]", " ".join(cmd), file=sys.stderr)
        subprocess.check_call(cmd)
    return out


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    build_host(force="--force" in sys.argv)
