"""Builds the in-tree native library spz_b200/_lib/libspz_b200.so with nvcc for sm_100a.

    python -m spz_b200.build [--force]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with the
gpurun snapshot.  Flags that matter for parity: -fmad=false (no FMA contraction in device code),
-Xcompiler -ffp-contract=off (none in the host-side table construction), IEEE div/sqrt and no
flush-to-zero (nvcc defaults, stated explicitly).
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_lib")
LIB = os.path.join(OUT_DIR, "libspz_b200.so")

CUDA_SOURCES = ["codec_kernels.cu", "ply_kernels.cu", "pergaussian_kernels.cu", "gather_kernels.cu", "deflate_kernels.cu", "inflate_kernels.cu", "quantize_kernels.cu", "move_kernels.cu", "cabi.cu"]
CXX_SOURCES = ["spz_api.cc", "spz_ply.cc", "spz_gzip.cc"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math,-Wall,-Wno-unused-function",
    "-diag-suppress", "177,179",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _sources():
    srcs = [os.path.join(CSRC, s) for s in CUDA_SOURCES]
    srcs += [os.path.join(CSRC, s) for s in CXX_SOURCES if os.path.exists(os.path.join(CSRC, s))]
    return srcs


def _deps():
    deps = []
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for dirpath, _, files in os.walk(root):
            deps += [os.path.join(dirpath, f) for f in files]
    deps.append(os.path.abspath(__file__))
    return deps


def up_to_date() -> bool:
    if not os.path.exists(LIB):
        return False
    t = os.path.getmtime(LIB)
    return all(os.path.getmtime(d) <= t for d in _deps())


def build(force: bool = False, verbose: bool = False, extra_flags=(), out: str | None = None) -> str:
    """Default: the shipped library.  `extra_flags` + `out` build a tuning variant next to it
    (loaded with SPZB200_LIB=<path>); used only by scripts/ experiments."""
    if out is None and not force and up_to_date():
        return LIB
    os.makedirs(OUT_DIR, exist_ok=True)
    lib_path = out or LIB
    tag = "" if out is None else "." + os.path.basename(out)
    objs = []
    procs = []
    for src in _sources():
        obj = os.path.join(OUT_DIR, os.path.basename(src) + tag + ".o")
        cmd = [_nvcc()] + NVCC_FLAGS + list(extra_flags) + ["-I", os.path.join(HERE, "..", "include"), "-c", src, "-o", obj]
        if src.endswith(".cc"):
            cmd.insert(1, "-x")
            cmd.insert(2, "cu")
        if verbose:
            print(" ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        if verbose and out.strip():
            print(out)
    link = [_nvcc(), "-shared", "-o", lib_path] + objs + ["-lz", "-cudart", "static"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout)
    return lib_path


PY_DIR = os.path.join(HERE, "pyspz")


def python_module_path() -> str:
    import sysconfig
    return os.path.join(PY_DIR, "spz" + sysconfig.get_config_var("EXT_SUFFIX"))


def build_python_module(force: bool = False) -> str:
    """The Python module `spz` (csrc/py_spz.cc, pybind11) next to spz_b200/pyspz/__init__.py,
    linked against the in-tree libspz_b200.so."""
    import sysconfig

    import pybind11
    out = python_module_path()
    src = os.path.join(CSRC, "py_spz.cc")
    hdr = os.path.join(HERE, "..", "include", "spz_b200", "spz.hpp")
    lib = build()
    if not force and os.path.exists(out) and os.path.getmtime(out) >= max(os.path.getmtime(p) for p in (src, hdr, lib)):
        return out
    cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden", "-ffp-contract=off",
           "-I", pybind11.get_include(), "-I", sysconfig.get_paths()["include"], src, "-o", out,
           "-L", OUT_DIR, "-lspz_b200", "-Wl,-rpath,$ORIGIN/../_lib"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("python module build failed:\n" + r.stdout)
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
    print(build_python_module(force="--force" in sys.argv))
