"""TEST INFRASTRUCTURE ONLY.  ctypes binding of tests/gi_oracle.c: the CPU restatement of the sampling contract
(DESIGN.md 3.10) on top of the restated reference of oracle/crt_oracle.c, plus the shared header's Philox / tangent
frame / direction sampler as test hooks.  The library is compiled on first use into a temporary directory."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "course-assignment-danielhalachev_b200", "csrc")
HIT_DTYPE = np.dtype([("mesh", np.int32), ("triangle", np.int32), ("t", np.float32)])


class OracleStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("rays_primary", "rays_shadow", "rays_reflection", "rays_refraction",
                                          "node_tests_closest", "triangle_tests_closest", "node_tests_shadow",
                                          "triangle_tests_shadow", "max_query_tests")]


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="gi_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libgi_oracle.so")
        subprocess.run(["gcc", "-std=gnu11", "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-shared",
                        "-I", CSRC, "-o", so, os.path.join(HERE, "gi_oracle.c"), "-lm"], check=True)
        l = C.CDLL(so)
        l.crt_oracle_render_sampled.argtypes = [C.c_void_p] * 6 + [C.POINTER(OracleStats), C.POINTER(C.c_uint64), C.c_int]
        l.crt_oracle_philox.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        l.crt_oracle_unit.argtypes = [C.c_uint32]
        l.crt_oracle_unit.restype = C.c_float
        l.crt_oracle_tangent_frame.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        l.crt_oracle_diffuse_dirs.argtypes = [C.c_uint32] * 6 + [C.c_void_p, C.c_uint32, C.c_void_p]
        _lib = l
    return _lib


def render_sampled(scene_ptr, camera, options, sampling, threads: int = 0, want_hits: bool = True):
    """crt_oracle_render_sampled: returns (rgb HxWx3 f32, hits | None, stats dict with rays_diffuse)."""
    s = scene_ptr.contents
    rgb = np.zeros((s.height, s.width, 3), np.float32)
    hits = np.zeros((s.height, s.width), HIT_DTYPE) if want_hits else None
    st = OracleStats()
    diffuse = C.c_uint64(0)
    if threads <= 0:
        threads = os.cpu_count() or 1
    rc = lib().crt_oracle_render_sampled(C.cast(scene_ptr, C.c_void_p), C.addressof(camera), C.addressof(options),
                                         C.addressof(sampling), rgb.ctypes.data,
                                         hits.ctypes.data if hits is not None else None, C.byref(st), C.byref(diffuse), threads)
    if rc != 0:
        raise RuntimeError("crt_oracle_render_sampled failed")
    d = {n: getattr(st, n) for n, _ in st._fields_ if n != "max_query_tests"}
    d["rays_diffuse"] = diffuse.value
    return rgb, hits, d


def philox(ctr, key) -> list[int]:
    c = (C.c_uint32 * 4)(*ctr)
    k = (C.c_uint32 * 2)(*key)
    out = (C.c_uint32 * 4)()
    lib().crt_oracle_philox(c, k, out)
    return list(out)


def unit(u: int) -> float:
    return lib().crt_oracle_unit(u)


def tangent_frame(n):
    n = np.ascontiguousarray(n, np.float32)
    t = np.zeros(3, np.float32)
    b = np.zeros(3, np.float32)
    lib().crt_oracle_tangent_frame(n.ctypes.data, t.ctypes.data, b.ctypes.data)
    return t, b


def diffuse_dirs(n, count: int, seed=0, frame=0, p=0, s=0, key0=0, k=0) -> np.ndarray:
    n = np.ascontiguousarray(n, np.float32)
    out = np.zeros((count, 3), np.float32)
    lib().crt_oracle_diffuse_dirs(seed, frame, p, s, key0, k, n.ctypes.data, count, out.ctypes.data)
    return out
