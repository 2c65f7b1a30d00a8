"""TEST INFRASTRUCTURE ONLY.  ctypes binding of tests/progressive_oracle.c: the CPU restatement of a progressive
session's accumulator (DESIGN.md 3.10.1) on top of tests/gi_oracle.c.  The library is compiled on first use into a
temporary directory."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from gi_oracle import CSRC, HERE

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="progressive_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libprogressive_oracle.so")
        subprocess.run(["gcc", "-std=gnu11", "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-shared",
                        "-I", CSRC, "-o", so, os.path.join(HERE, "progressive_oracle.c"), "-lm"], check=True)
        l = C.CDLL(so)
        l.crt_oracle_render_sums.argtypes = [C.c_void_p] * 6 + [C.c_int]
        _lib = l
    return _lib


def render_sums(scene_ptr, camera, options, sampling, threads: int = 0):
    """crt_oracle_render_sums: a progressive session's S and Q after sampling.rays_per_pixel samples (HxWx3 f32 each,
    0 outside the rects)."""
    s = scene_ptr.contents
    sums = np.zeros((s.height, s.width, 3), np.float32)
    sumsq = np.zeros((s.height, s.width, 3), np.float32)
    if threads <= 0:
        threads = os.cpu_count() or 1
    rc = lib().crt_oracle_render_sums(C.cast(scene_ptr, C.c_void_p), C.addressof(camera), C.addressof(options),
                                      C.addressof(sampling), sums.ctypes.data, sumsq.ctypes.data, threads)
    if rc != 0:
        raise RuntimeError("crt_oracle_render_sums failed")
    return sums, sumsq
