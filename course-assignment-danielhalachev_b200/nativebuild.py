"""In-tree build of the native libraries (no JIT cache: the built .so files travel to the GPU box with the snapshot).

  csrc/libcrtb200.so   CUDA core + C ABI        nvcc -gencode arch=compute_100a,code=sm_100a --fmad=false -lineinfo
  csrc/libcrtfront.so  C++ host front end       g++ -ffp-contract=off (no -march=native: FMA is a parity variable)
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)

CORE_SO = os.path.join(CSRC, "libcrtb200.so")
FRONT_SO = os.path.join(CSRC, "libcrtfront.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "--fmad=false", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared", "-cudart", "static",
]
GXX_FLAGS = ["-std=c++17", "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-shared", "-pthread", "-Wall"]


def _newer(target: str, sources: list[str]) -> bool:
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)


def _run(cmd: list[str], verbose: bool) -> None:
    if verbose:
        print("+", " ".join(cmd), flush=True)
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("build failed: " + " ".join(cmd))
    if verbose and (r.stdout or r.stderr):
        print(r.stdout + r.stderr)


def nvcc_path() -> str:
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def build_core(force: bool = False, verbose: bool = False, extra: list[str] | None = None, out: str | None = None) -> str:
    """extra: additional nvcc flags (e.g. -DCRT_LOOP_MODE=1 for a tuning variant written to `out`)."""
    if out:
        src = os.path.join(CSRC, "crtb200_core.cu")
        _run([nvcc_path(), *NVCC_FLAGS, *(extra or []), "-o", out, src], verbose)
        return out
    srcs = [os.path.join(CSRC, f) for f in ("crtb200_core.cu", "crt_kernels.cuh", "crt_device.cuh", "crt_powf5.h", "crt_sampling.h", "crt_build.cuh")]
    srcs.append(os.path.join(ROOT, "include", "crtb200.h"))
    if force or not _newer(CORE_SO, srcs):
        _run([nvcc_path(), *NVCC_FLAGS, *(extra or []), "-o", CORE_SO, srcs[0]], verbose)
    return CORE_SO


def build_front(force: bool = False, verbose: bool = False) -> str:
    fdir = os.path.join(CSRC, "frontend")
    cpps = [os.path.join(fdir, f) for f in ("crt_scene.cpp", "crt_kdtree.cpp", "crt_raytracer.cpp", "crt_front_c.cpp")]
    deps = cpps + [os.path.join(fdir, f) for f in os.listdir(fdir) if f.endswith(".hpp")]
    deps += [os.path.join(ROOT, "include", "crtb200.h"), os.path.join(ROOT, "include", "crtfront.h"), CORE_SO]
    if force or not _newer(FRONT_SO, deps):
        _run(["g++", *GXX_FLAGS, "-o", FRONT_SO, *cpps, "-L" + CSRC, "-lcrtb200", "-Wl,-rpath,$ORIGIN", "-lz"], verbose)
    return FRONT_SO


def build_all(force: bool = False, verbose: bool = False) -> None:
    build_core(force, verbose)
    build_front(force, verbose)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv, verbose=True)
