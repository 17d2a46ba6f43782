"""Builds libfic_b200.so (and the dev probe) in-tree with nvcc for sm_100a.

    python fractal-image-compression_b200/build.py [--force] [--probe]

The shared library has no torch or Python dependency: it is the C ABI of
include/fic_b200.h, linked against the static CUDA runtime.
"""
from __future__ import annotations

import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libfic_b200.so")
PROBE = os.path.join(LIBDIR, "umma_probe")
CLI = os.path.join(LIBDIR, "fic_cli")

SOURCES = ["fic_kernels.cu", "fic_decode.cu", "fic_search_umma.cu", "fic_quadtree.cu", "fic_encode.cu", "fic_api.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--fmad=false",            # Java never fuses a*b+c; parity-critical code also uses *_rn intrinsics
    "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(out: str, deps: list[str]) -> bool:
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    return any(os.path.getmtime(d) > t for d in deps)


def _headers() -> list[str]:
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    hs.append(os.path.join(ROOT, "include", "fic_b200.h"))
    return hs


def _compile(src: str, force: bool) -> str:
    obj = os.path.join(OBJ, os.path.basename(src).replace(".cu", ".o"))
    if force or _stale(obj, [src] + _headers()):
        cmd = [_nvcc()] + NVCC_FLAGS + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        with open(obj + ".log", "w") as f:
            f.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError(f"nvcc failed on {src}")
    return obj


def build(force: bool = False, probe: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(LIBDIR, exist_ok=True)
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    with cf.ThreadPoolExecutor(max_workers=4) as ex:
        objs = list(ex.map(lambda s: _compile(s, force), srcs))
    arch = ["-gencode", "arch=compute_100a,code=sm_100a"]
    if force or _stale(LIB, objs):
        subprocess.check_call([_nvcc(), "-shared", "-o", LIB] + objs + arch)
    cli_src = os.path.join(HERE, "host", "fic_cli.cpp")
    cli_deps = [cli_src, os.path.join(HERE, "host", "fractal_compression.hpp"), LIB]
    if force or _stale(CLI, cli_deps):  # C++ host mirror + headless CLI over the C ABI
        gxx = shutil.which("g++") or "g++"
        subprocess.check_call([gxx, "-std=c++17", "-O2", "-o", CLI, cli_src, "-L" + LIBDIR, "-lfic_b200",
                               "-Wl,-rpath,$ORIGIN"])
    if probe:
        psrc = os.path.join(ROOT, "tools", "umma_probe.cu")
        if os.path.exists(psrc) and (force or _stale(PROBE, [psrc] + objs)):
            pobj = _compile(psrc, force)
            subprocess.check_call([_nvcc(), "-o", PROBE, pobj] + objs + arch)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, probe="--probe" in sys.argv))
