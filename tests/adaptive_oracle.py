"""TEST INFRASTRUCTURE ONLY.  ctypes binding of tests/adaptive_oracle.c: the CPU restatement of an adaptive progressive
session (DESIGN.md 3.10.2) on top of tests/gi_oracle.c.  The library is compiled on first use into a temporary
directory."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from gi_oracle import CSRC, HERE, OracleStats

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="adaptive_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libadaptive_oracle.so")
        subprocess.run(["gcc", "-std=gnu11", "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-shared",
                        "-I", CSRC, "-o", so, os.path.join(HERE, "adaptive_oracle.c"), "-lm"], check=True)
        l = C.CDLL(so)
        l.crt_oracle_render_adaptive.argtypes = [C.c_void_p] * 5 + [C.c_uint32] + [C.c_void_p] * 5 + [C.c_int]
        l.crt_oracle_adapt_stop.argtypes = [C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = l
    return _lib


def render_adaptive(scene_ptr, camera, options, sampling, adaptive, passes: int, threads: int = 0):
    """crt_oracle_render_adaptive: (S, Q HxWx3 f32, counts HxW u32, stats dict with rays_diffuse) after `passes`
    passes; 0 outside the rects."""
    s = scene_ptr.contents
    sums = np.zeros((s.height, s.width, 3), np.float32)
    sumsq = np.zeros((s.height, s.width, 3), np.float32)
    counts = np.zeros((s.height, s.width), np.uint32)
    st = OracleStats()
    diffuse = C.c_uint64(0)
    if threads <= 0:
        threads = os.cpu_count() or 1
    rc = lib().crt_oracle_render_adaptive(C.cast(scene_ptr, C.c_void_p), C.addressof(camera), C.addressof(options),
                                          C.addressof(sampling), C.addressof(adaptive), passes, sums.ctypes.data,
                                          sumsq.ctypes.data, counts.ctypes.data, C.byref(st), C.byref(diffuse), threads)
    if rc != 0:
        raise RuntimeError("crt_oracle_render_adaptive failed")
    d = {n: getattr(st, n) for n, _ in st._fields_ if n != "max_query_tests"}
    d["rays_diffuse"] = diffuse.value
    return sums, sumsq, counts, d


def adapt_stop(n: int, S, Q, adaptive) -> bool:
    """crt_s_adapt_stop, as compiled for the CPU."""
    s = np.ascontiguousarray(S, np.float32)
    q = np.ascontiguousarray(Q, np.float32)
    return bool(lib().crt_oracle_adapt_stop(n, s.ctypes.data, q.ctypes.data, C.addressof(adaptive)))
